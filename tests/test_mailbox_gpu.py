"""GPU: mailboxes of the dense in-place storage (lbm_mail_export / lbm_mail_attach): the 5 populations that enter
through a slab face live in a small per-side allocation instead of in the halo / face planes of the population
buffer, so that a neighbouring process maps ~80 MB instead of the whole buffer.  Virtual slabs on one device: must
equal the single domain bit for bit at odd and even step counts, with one- and two-plane slabs, through
checkpoints and lbm_debug_get_populations, and after switching back to the buffers."""
import numpy as np
import pytest

import helpers as H

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name,n,P", [("ldc", 24, 3), ("bif", None, 4), ("cor", None, 5), ("pos", 24, 2), ("ldc", 12, 12),
                                      ("ldc", 12, 6), ("corstep", None, 7)])
def test_mailbox_slabs_equal_single_domain_bitwise(name, n, P):
    import lattice_boltzmann_method_gpu_b200 as L

    one = H.gpu_case(name, n, L.F64, L.MATH_FAST, storage=L.STORE_DENSE_AA)
    H.gpu_setup(one, name)
    cs = H.virtual_slabs(name, n, P)
    H.attach_virtual_slabs(cs, mail=True)
    for steps in (1, 1, 1, 18):  # totals 1, 2, 3, 21
        one.step(steps)
        H.step_virtual_slabs(cs, steps)
        ref = one.get_fields()
        for k in range(4):
            assert np.array_equal(np.concatenate([c.get_fields()[k] for c in cs]), ref[k]), (name, k, one.step_count)


def test_mailbox_checkpoint_populations_and_switching_back(tmp_path):
    import lattice_boltzmann_method_gpu_b200 as L

    name, n, P = "bif", None, 3
    one = H.gpu_case(name, n, L.F64, L.MATH_FAST, storage=L.STORE_DENSE_AA)
    H.gpu_setup(one, name)
    one.step(30)
    ref = one.get_fields()
    cs = H.virtual_slabs(name, n, P)
    H.attach_virtual_slabs(cs, mail=True)
    H.step_virtual_slabs(cs, 7)
    pops = [c.get_populations() for c in cs]      # drains and refills the mailboxes around the gather
    for r, c in enumerate(cs):
        c.checkpoint_save(tmp_path / f"ck{r}.bin")
    H.step_virtual_slabs(cs, 4)
    # (a) continue after a restore: same as never having stopped
    for r, c in enumerate(cs):
        c.checkpoint_load(tmp_path / f"ck{r}.bin")
        assert np.array_equal(c.get_populations(), pops[r])
    H.step_virtual_slabs(cs, 10)
    # (b) switch every face back to storing into the neighbours' buffers, and on
    for c in cs:
        for side in (0, 1):
            try:
                c.mail_attach(side, None)
            except L.LbmError:
                pass  # no neighbour on that side
    H.attach_virtual_slabs(cs, mail=False)
    H.step_virtual_slabs(cs, 13)
    for k in range(4):
        assert np.array_equal(np.concatenate([c.get_fields()[k] for c in cs]), ref[k]), k
    # a checkpoint written with mailboxes loads into a fresh set of slabs without
    ds = H.virtual_slabs(name, n, P)
    H.attach_virtual_slabs(ds, mail=False)
    for r, c in enumerate(ds):
        c.checkpoint_load(tmp_path / f"ck{r}.bin")
    H.step_virtual_slabs(ds, 23)
    for k in range(4):
        assert np.array_equal(np.concatenate([c.get_fields()[k] for c in ds]), ref[k]), k


def test_mailboxes_are_for_the_dense_in_place_storage():
    import lattice_boltzmann_method_gpu_b200 as L

    c = H.gpu_case("ldc", 16, L.F32, L.MATH_FAST, z_range=(0, 8), storage=L.STORE_DENSE_AB)
    c.geo_pre()
    c.set_compact_offset(0, 16 ** 3)
    c.index_transform()
    c.initialize()
    with pytest.raises(L.LbmError):
        c.mail_export(1)
