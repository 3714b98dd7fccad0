"""GPU: a slab holds one kind of fused face exchange at a time.  Mapped peer buffers and mailboxes address the
neighbour's memory differently, and the launch of a one-plane slab covers both of its faces with a single flag that
says which addressing to use; so attaching one kind while either side of the slab holds the other is refused
(LBM_ERR_STATE, detach first).  Virtual slabs of the dense in-place storage on one device: every case checks the
refusal before any step is launched, then wires the slabs one way and must still equal the single domain bit for bit."""
import numpy as np
import pytest

import helpers as H

pytestmark = pytest.mark.gpu

N, STEPS = 12, 5
STATE = -2  # LBM_ERR_STATE


def _peer_args(cs, r, side):
    """lbm_p2p_attach arguments for side `side` of slab r: its neighbour's two buffers"""
    e = cs[r - 1 if side == 0 else r + 1].p2p_export()
    return e["ptrs"][0], e["ptrs"][1], e["qs"], e["halo_c0"][1 - side], e["face_c0"][1 - side]


def _mail_ptr(cs, r, side):
    """the neighbour's mailbox facing side `side` of slab r, once slab r has its own mailbox of that side"""
    cs[r].mail_export(side)
    return cs[r - 1 if side == 0 else r + 1].mail_export(1 - side)["ptr"]


def _refused(call, *args):
    import lattice_boltzmann_method_gpu_b200 as L

    with pytest.raises(L.LbmError) as e:
        call(*args)
    assert e.value.status == STATE and "detach" in str(e.value)


def _equals_single_domain(cs):
    import lattice_boltzmann_method_gpu_b200 as L

    one = H.gpu_case("ldc", N, L.F64, L.MATH_FAST, storage=L.STORE_DENSE_AA)
    H.gpu_setup(one, "ldc")
    one.step(STEPS)
    H.step_virtual_slabs(cs, STEPS)
    ref = one.get_fields()
    for k in range(4):
        assert np.array_equal(np.concatenate([c.get_fields()[k] for c in cs]), ref[k]), k


def test_peer_buffers_refused_on_a_mailbox_side():
    cs = H.virtual_slabs("ldc", N, 3)
    H.attach_virtual_slabs(cs, mail=True)
    _refused(cs[1].p2p_attach, 1, *_peer_args(cs, 1, 1))
    _equals_single_domain(cs)


def test_mailboxes_refused_on_a_peer_buffer_side():
    cs = H.virtual_slabs("ldc", N, 3)
    H.attach_virtual_slabs(cs, mail=False)
    _refused(cs[1].mail_attach, 1, _mail_ptr(cs, 1, 1))
    _refused(cs[1].mail_stage, 1)
    _equals_single_domain(cs)


@pytest.mark.parametrize("first", ["mailbox", "peer_buffers"])
def test_one_plane_slab_holds_one_kind_on_both_faces(first):
    """slab 5 of 12 owns one plane: its face launch covers both sides.  One kind on side 0, the other refused on
    side 1 (which holds nothing yet), then every face wired with the first kind"""
    cs = H.virtual_slabs("ldc", N, N)
    r = 5
    if first == "mailbox":
        cs[r].mail_attach(0, _mail_ptr(cs, r, 0))
        _refused(cs[r].p2p_attach, 1, *_peer_args(cs, r, 1))
    else:
        cs[r].p2p_attach(0, *_peer_args(cs, r, 0))
        _refused(cs[r].mail_attach, 1, _mail_ptr(cs, r, 1))
        _refused(cs[r].mail_stage, 1)
    H.attach_virtual_slabs(cs, mail=first == "mailbox")
    _equals_single_domain(cs)
