"""z-slab domain decomposition over the GPUs of one box (SURVEY.md 8e).

The reference is single-GPU; this is new work whose oracle is "N slabs == one domain, bit for bit".
One process per GPU (torchrun); rank r owns global planes [z_begin, z_end) plus one halo plane per
interior face.  Per time step each rank sends, per face, the 5 populations that cross it
(c_z = +1: q in {5,11,13,15,16} upward, c_z = -1: q in {6,12,14,17,18} downward) of its outermost
owned plane -- one contiguous staging buffer per face, packed by the library right after the face
planes were computed so the transfer overlaps the interior update -- with
torch.distributed P2P ops (NCCL over NVLink on GPUs; gloo on CPU for the host-logic tests).

With the fused peer-store exchange (the default) the time loop itself is `lbm_slab_step` inside the
library: neighbours are ordered by progress flags in peer memory, so neither Python nor NCCL runs per
step; torch.distributed only bootstraps (counts, IPC handles) and all-reduces the residual when the
caller asks for one.

Nothing here computes: the kernels live in liblbm_b200.so.  `exchange_halos` and `slab_ranges` /
`compact_offsets` are backend-agnostic so the same code runs under gloo in the CPU tests.
"""
from __future__ import annotations


import numpy as np

from . import api


def slab_ranges(nz: int, world: int):
    """contiguous, near-equal z ranges; every slab gets at least one plane"""
    if world > nz:
        raise ValueError("more slabs than planes")
    base, rem = divmod(nz, world)
    out, z = [], 0
    for r in range(world):
        n = base + (1 if r < rem else 0)
        out.append((z, z + n))
        z += n
    return out


def compact_offsets(local_counts):
    """exclusive running sum of the per-slab stored-node counts: the single-domain z,y,x numbering
    of index_transform (bifurcation.cu:241-252) continues across slabs"""
    offs, run = [], 0
    for c in local_counts:
        offs.append(run)
        run += int(c)
    return offs, run


def exchange_halos(send_lo, recv_lo, send_hi, recv_hi, rank: int, world: int, group=None):
    """Post the (up to four) point-to-point transfers of one step and return the work handles.

    send_lo -> rank-1's recv_hi,  send_hi -> rank+1's recv_lo.  Any of the tensors may be None at
    the outer faces of the domain.  Works for CUDA tensors (NCCL) and CPU tensors (gloo)."""
    import torch.distributed as dist

    ops = []
    if rank > 0 and send_lo is not None:
        ops.append(dist.P2POp(dist.isend, send_lo, rank - 1, group))
        ops.append(dist.P2POp(dist.irecv, recv_lo, rank - 1, group))
    if rank < world - 1 and send_hi is not None:
        ops.append(dist.P2POp(dist.isend, send_hi, rank + 1, group))
        ops.append(dist.P2POp(dist.irecv, recv_hi, rank + 1, group))
    if not ops:
        return []
    return dist.batch_isend_irecv(ops)


class _DevBuf:
    """zero-copy view of a library-owned device buffer for torch (CUDA array interface v2)"""

    def __init__(self, ptr: int, nbytes: int, dtype: np.dtype):
        self.__cuda_array_interface__ = {
            "shape": (nbytes // dtype.itemsize,), "typestr": dtype.str, "data": (ptr, False), "version": 2,
            "strides": None,
        }


class SlabCase(api.Case):
    """A `Case` that owns one z-slab of a larger domain and steps in lock-step with its neighbours."""

    def __init__(self, desc: api.CaseDesc, group=None):
        import torch.distributed as dist

        super().__init__(desc)
        self.group = group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        self._bufs = None
        self._p2p = False
        self._sync_ptrs = []
        self.timing = {}         # seconds spent in the phases of setup / enable_p2p (bench.py reports them)
        self._mapped = []        # IPC handles this rank holds a mapping of
        self.p2p_error = None    # why enable_p2p fell back, if it did

    def setup(self, flag=None, bc_planes=None, flag_slab=None):
        """geo_pre -> (all-gather of stored counts) -> index_transform -> read_vel -> initialize"""
        import torch
        import torch.distributed as dist

        import time

        t0 = time.perf_counter()
        if flag is not None:
            self.set_flag(flag)
        if flag_slab is not None:  # only the planes this rank needs: (uint8 array, z_first)
            self.set_flag_slab(*flag_slab)
        self.geo_pre()
        t1 = time.perf_counter()
        mine = torch.tensor([self.local_stored_count()], dtype=torch.int64, device="cuda")
        allc = torch.empty(self.world, dtype=torch.int64, device="cuda")
        dist.all_gather_into_tensor(allc, mine, group=self.group)
        offs, total = compact_offsets(allc.cpu().tolist())
        t2 = time.perf_counter()
        self.set_compact_offset(offs[self.rank], total)
        self.index_transform()
        if bc_planes is not None:
            self.set_bc_planes(*bc_planes)
        self.initialize()
        self._wrap_buffers()
        self.timing.update(geo_pre=t1 - t0, count_exchange=t2 - t1, index_init=time.perf_counter() - t2)

    def enable_p2p(self):
        """Fused halo exchange: every rank maps what its neighbours export for it and their sync blocks (CUDA IPC
        over NVLink); the step kernel stores the crossing populations there itself and the slabs order their steps
        through progress flags in that memory (lbm_slab_step) -- no collective is left in the time loop.

        The dense in-place storage exports small per-face mailboxes (lbm_mail_export / attach), the other storages
        their whole population buffers (lbm_p2p_export / attach): cudaIpcOpenMemHandle costs 50-65 ms per GB mapped,
        0.74 s for a 512^3 fp64 slab, against a few ms for the ~80 MB mailbox of a 1024^2 face.  Returns False on
        every rank, with nothing attached, when any rank cannot map its neighbours."""
        import time

        import torch
        import torch.distributed as dist

        t0 = time.perf_counter()
        mail = self.desc.storage == api.STORE_DENSE_AA
        sides = [s for s, nb in ((0, self.rank - 1), (1, self.rank + 1)) if 0 <= nb < self.world]
        # fixed-size record, one all_gather of bytes (no pickling): 3 IPC handles (mailbox low / high or population
        # buffer a / b, sync block), then 8 int64: their byte offsets, q stride, halo_c0[2], face_c0[2]
        rec = np.zeros(3 * 64 + 8 * 8, dtype=np.uint8)
        ints = rec[192:].view(np.int64)
        if mail:
            for s in sides:
                m = self.mail_export(s)
                rec[64 * s:64 * s + 64] = np.frombuffer(m["handle"], dtype=np.uint8)
                ints[s] = m["boff"]
        else:
            e = self.p2p_export()
            for k in (0, 1):
                rec[64 * k:64 * k + 64] = np.frombuffer(e["handles"][k], dtype=np.uint8)
            ints[:2], ints[3:] = e["boff"], [e["qs"], *e["halo_c0"], *e["face_c0"]]
        sy = self.sync_export()
        rec[128:192] = np.frombuffer(sy["handle"], dtype=np.uint8)
        ints[2] = sy["boff"]
        t = torch.from_numpy(rec).cuda()
        allt = torch.empty(self.world * rec.size, dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(allt, t, group=self.group)
        allr = allt.cpu().numpy().reshape(self.world, rec.size)
        t1 = time.perf_counter()
        ok, links = 1, []
        try:
            for s in sides:
                r = allr[self.rank - 1 if s == 0 else self.rank + 1]
                o = [int(v) for v in r[192:].view(np.int64)]
                # the neighbour's mailbox of the side FACING this slab, or both its buffers; then its sync block
                ptrs = []
                for k in ((1 - s,) if mail else (0, 1)) + (2,):
                    h = r[64 * k:64 * k + 64].tobytes()
                    ptrs.append(api.p2p_open(h) + o[k])
                    self._mapped.append(h)
                links.append((s, ptrs, o))
        except api.LbmError as e:
            ok, self.p2p_error = 0, str(e)
        # all ranks or none: a rank that cannot map its neighbour (no peer access / IPC) sends everyone
        # back to the pack / staged path
        flag = torch.tensor([ok], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        if int(flag.item()) == 0:
            self._release_mappings()
            return False
        t2 = time.perf_counter()
        dist.barrier(group=self.group)  # both slabs of a face switch over between the same two steps
        for s, ptrs, o in links:
            if mail:
                self.mail_attach(s, ptrs[0])
            else:  # my low face feeds the neighbour's HIGH halo plane and vice versa
                self.p2p_attach(s, ptrs[0], ptrs[1], o[3], o[5 - s], o[7 - s])
        self._sync_ptrs = [(s, ptrs[-1]) for s, ptrs, _ in links]
        self._attach_sync()
        self._p2p = True
        self.timing.update(handle_exchange=t1 - t0, ipc_open=t2 - t1, sync_attach=time.perf_counter() - t2)
        return True

    def _attach_sync(self):
        """collective: every rank zeroes its progress counters, then nobody steps before all have"""
        import torch.distributed as dist

        dist.barrier(group=self.group)   # nobody is still stepping
        for side, ptr in self._sync_ptrs:
            self.sync_attach(side, ptr)
        dist.barrier(group=self.group)   # every counter is zero before the first new signal

    def checkpoint_load(self, path):
        super().checkpoint_load(path)
        if self._p2p:
            self._attach_sync()

    def _release_mappings(self):
        for h in self._mapped:
            api.p2p_release(h)
        self._mapped = []

    def close(self):
        """collective when peer mappings exist: every rank unmaps its neighbours' buffers before anyone
        frees them"""
        if self._mapped:
            import torch.distributed as dist

            self.sync()
            self._release_mappings()
            if dist.is_initialized():
                dist.barrier(group=self.group)
        self._p2p = False
        super().close()

    def __del__(self):  # never collective: a garbage-collected case only drops its own mappings
        try:
            self._release_mappings()
            api.Case.close(self)
        except Exception:
            pass

    def _wrap_buffers(self):
        import torch

        self._ext = torch.cuda.ExternalStream(self.stream)
        bufs = []
        for side in (0, 1):
            s, r, ns, nr = self.halo_buffers(side)
            if not s:
                bufs.append((None, None))
            else:  # an empty plane (sparse storage) still takes part in the exchange with 0-size-safe tensors
                bufs.append((torch.as_tensor(_DevBuf(s, max(ns, self.dtype.itemsize), self.dtype), device="cuda")[: ns // self.dtype.itemsize],
                             torch.as_tensor(_DevBuf(r, max(nr, self.dtype.itemsize), self.dtype), device="cuda")[: nr // self.dtype.itemsize]))
        self._bufs = bufs

    def enable_staged(self):
        """In-place dense storage WITHOUT peer mapping (no peer access between the GPUs, or --halo nccl): the mailbox
        exchange through local staging buffers that torch.distributed (NCCL send/recv) moves between the ranks
        (lbm_mail_stage).  Steps are then driven like the two-buffer storage's: begin / exchange / interior / end."""
        if self.desc.storage != api.STORE_DENSE_AA:
            raise api.LbmError(-2, "staged mailboxes exist for the dense in-place storage only")
        for side, present in ((0, self.rank > 0), (1, self.rank < self.world - 1)):
            if present:
                self.mail_stage(side)
        self._staged, self._p2p = True, False
        self._bufs_by_parity = {}

    def _one_step(self, flags=0):
        import torch

        self.step_begin(flags)  # face planes + pack, queued on the library's stream
        if getattr(self, "_staged", False):  # the staging parts alternate with the step's parity (A / B)
            par = self.step_count & 1
            if par not in self._bufs_by_parity:
                self._wrap_buffers()
                self._bufs_by_parity[par] = self._bufs
            self._bufs = self._bufs_by_parity[par]
        (s_lo, r_lo), (s_hi, r_hi) = self._bufs
        # torch.distributed orders NCCL's stream after what `self._ext` holds so far (faces + pack)
        with torch.cuda.stream(self._ext):
            works = exchange_halos(s_lo, r_lo, s_hi, r_hi, self.rank, self.world, self.group)
        self.step_interior()  # interior planes run while the faces travel over NVLink
        with torch.cuda.stream(self._ext):
            for w in works:
                w.wait()  # stream-ordered wait, no host sync
        self.step_end()  # unpack + buffer swap

    def step(self, n: int = 1):
        if self._p2p:
            self.slab_step(n)
            return
        for i in range(int(n)):
            self._one_step(api.STEP_MOMENTS if i == n - 1 else 0)
        self.sync()

    def run_converge(self, max_it=10000, tol=1e-6, stag_max=50, time_save=500, write_files=False):
        """ldc.cu:653-685 on a sharded domain: S_k is all-reduced over the slabs once per batch of steps;
        the stopping rule is the reference's, applied identically on every rank.  Returns (iterations,
        residual).  File output of a multi-process run: lbm_set_output_format(BINARY) pieces per slab."""
        import torch
        import torch.distributed as dist

        if not self._p2p:
            raise api.LbmError(-2, "run_converge on slabs needs the fused exchange (enable_p2p)")
        tol = np.float32(tol)
        residual, s_cur, k, hits = np.float32(0), np.float32(0), 0, 0
        while k <= max_it and hits <= stag_max:
            nb = min(48, max(1, stag_max + 1 - hits), max_it - k + 1)
            for j in range(nb):
                if (k + j) % time_save == 0:
                    nb = j + 1
                    break
            _, S = self.slab_step(nb, True, velsum=True)
            t = torch.from_numpy(S).cuda()
            dist.all_reduce(t, group=self.group)
            for s_next in t.cpu().numpy().astype(np.float32):
                residual = np.abs(s_next - s_cur) / s_next
                if k % time_save == 0 and write_files:
                    self.outputSave(k)
                k += 1
                s_cur = s_next
                if residual <= tol:
                    hits += 1
                if not (k <= max_it and hits <= stag_max):
                    break
        return k, float(residual)

    def step_timed(self, n: int) -> float:
        import torch

        if self._p2p:
            return self.slab_step(n)[0]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(self._ext):
            e0.record()
        for i in range(int(n)):
            self._one_step(api.STEP_MOMENTS if i == n - 1 else 0)
        with torch.cuda.stream(self._ext):
            e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)
