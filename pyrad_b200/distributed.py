"""Multi-GPU plumbing: one process per GPU, wavenumber-chunk sharding, ONE all-gather of the
finished spectra (torch.distributed; NCCL over NVLink on the GPU box, gloo in the CPU tests).

The compute is injected (`compute_chunk`) so that the host-side logic -- partition, per-rank line
subsetting, padded all-gather, assembly -- is exercised on CPU with gloo, and runs unchanged on
B200s with the CUDA engine behind it.
"""
import numpy as np

from . import partition as pt


class ShardPlan:
    """Everything a rank needs to know about its chunk."""

    def __init__(self, nu0, range_min, res, n_total, windows, rank, world, balance=True, chunks=None, cost=None,
                 farfield=False):
        idx = pt.line_index(nu0, range_min, res)
        self.cost = cost
        if chunks is not None:
            self.chunks = [tuple(c) for c in chunks]
        elif balance and world > 1:
            self.cost = pt.block_time_cost(idx, n_total, windows, farfield=farfield)
            self.chunks = pt.balanced_chunks(self.cost, n_total, world)
        else:
            self.chunks = pt.equal_chunks(n_total, world)
        self._args = (nu0, range_min, res, n_total, windows)
        self.rank, self.world = rank, world
        self.i_begin, self.i_end = self.chunks[rank]
        self.wmax = max(max(int(w) - 2, 0) for w in np.atleast_1d(windows))
        # lines whose window reaches the chunk (+1 line of slack each side, harmless)
        l0 = int(np.searchsorted(idx, self.i_begin - self.wmax, side="left"))
        l1 = int(np.searchsorted(idx, self.i_end - 1 + self.wmax, side="right"))
        # the subset starts on a multiple of four lines: K2 aligns its staging chunks to four records in the coordinates
        # of the UPLOADED list, so this keeps every tile's chunk boundaries -- hence the triple grouping and the FP32
        # flush points -- those of the unsharded run (bitwise shard invariance, tests/test_partition.py)
        l0 &= ~3
        self.l0, self.l1 = l0, max(l1, l0)
        self.max_chunk = max(b - a for a, b in self.chunks)
        self.n_total = n_total

    def rebalanced(self, measured_ms):
        """A new plan after one measured run: measured_ms[r] = device time rank r spent on its chunk (all ranks pass
        the same list).  Returns self when the model had no cost array (equal chunks) or nothing moves."""
        if self.cost is None or self.world == 1:
            return self
        chunks, corrected = pt.rebalanced_chunks(self.cost, self.chunks, measured_ms, self.n_total)
        if chunks == self.chunks:
            return self
        return ShardPlan(*self._args, self.rank, self.world, chunks=chunks, cost=corrected)

    def subset(self, lines):
        return {k: np.ascontiguousarray(np.asarray(v)[self.l0:self.l1]) for k, v in lines.items()}


def all_gather_spectra(local, plan, dist=None, device=None):
    """local: torch tensor of the rank's finished chunk (any float dtype, on `device`).
    Pads to the widest chunk, runs ONE all_gather_into_tensor, returns the (world, max_chunk) tensor."""
    import torch
    n = plan.i_end - plan.i_begin
    pad = torch.zeros(plan.max_chunk, dtype=local.dtype, device=local.device)
    pad[:n] = local[:n]
    out = torch.empty(plan.world * plan.max_chunk, dtype=local.dtype, device=local.device)
    if dist is None or plan.world == 1:
        out[:plan.max_chunk] = pad
    else:
        dist.all_gather_into_tensor(out, pad)
    return out.view(plan.world, plan.max_chunk)


def assemble(gathered, plan):
    import torch
    parts = [gathered[r, : b - a] for r, (a, b) in enumerate(plan.chunks)]
    return torch.cat(parts) if parts else gathered.new_zeros(0)


def sum_over_ranks(values, dist=None):
    """Sum of a small float64 array of any shape over the ranks -- e.g. the level fluxes of Engine.atmosphere_fluxes or
    the (n_bands, L+1) band fluxes of Engine.atmosphere_band_fluxes, of which every rank holds its wavenumber chunk's
    share.  ONE all_gather, then the ranks' arrays added in rank order on every rank, so the result is deterministic and
    the same everywhere (an all_reduce leaves the order to the backend)."""
    import torch
    v = torch.as_tensor(np.ascontiguousarray(values, dtype=np.float64))
    if dist is None or dist.get_world_size() == 1:
        return v.numpy().copy()
    if dist.get_backend() == "nccl":
        v = v.cuda()
    parts = [torch.empty_like(v) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, v)
    total = parts[0].clone()
    for p in parts[1:]:
        total += p
    return total.cpu().numpy()


def connect_peers(engine, rank, world, max_chunk_points, dist):
    """Set up the engine's peer-memory gather: allocate this rank's buffer, exchange the CUDA IPC handles
    with ONE all_gather of 64 bytes per rank (torch.distributed: plumbing), map every peer.  After this,
    engine.atmosphere() leaves the gathered spectra of all ranks in engine.peer_gathered_dev() -- the
    all-gather is fused into the compute step (stores over NVLink from inside the kernel)."""
    import torch
    handle = engine.peer_alloc(rank, world, max_chunk_points)
    if world == 1:
        engine.peer_connect([handle])
        return
    mine = torch.frombuffer(bytearray(handle), dtype=torch.uint8).cuda()
    allh = torch.empty(world * len(handle), dtype=torch.uint8, device="cuda")
    dist.all_gather_into_tensor(allh, mine)
    blob = bytes(allh.cpu().numpy().tobytes())
    engine.peer_connect(blob)
    dist.barrier()


def gathered_spectra(engine, plan_or_chunks=None):
    """(radiance, transmittance) as torch views [world, ld] of the engine's gather buffer (no copy)."""
    rp, tp, ld = engine.peer_gathered_dev()
    world = engine._peer_world
    return (device_tensor(rp, world * ld).view(world, ld), device_tensor(tp, world * ld).view(world, ld))


class CudaArrayView:
    """Zero-copy view of engine-owned device memory for torch (``torch.as_tensor(view, device='cuda')``)."""

    def __init__(self, ptr, n, typestr="<f4"):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 3, "strides": None}


def device_tensor(ptr, n, typestr="<f4", device="cuda"):
    import torch
    return torch.as_tensor(CudaArrayView(ptr, n, typestr), device=device)
