"""Multi-GPU MSM: one process per GPU, points sharded contiguously, one small all-gather.

Replaces the reference's only parallel mechanism, the SPMD thread pool of src/threads/*.ts: there
every worker runs the same msm() on a `range(N)` slice of the inputs (threads.ts:354-359) and the
main thread adds the per-thread partial sums (msm-batched-affine.ts:311-320).  Here rank r owns the
pairs [lo, hi) of `shard_range`, computes the partial sum of its shard on its own B200, and the G
un-normalised partial accumulators (192 bytes each for BLS12-377) are exchanged with ONE all-gather
over NCCL / NVLink; every rank then adds them and normalises.  MSM has no other exchange step.
The collective lives in the C library (`mgb_comm_init`, `mgb_msm_sharded`, include/montgomery_b200.h):
ncclAllGather on the engine's stream straight after the Horner kernel, one combine + normalise
kernel, one device-to-host copy, one synchronisation.
"""
import torch
import torch.distributed as dist

from .api import MsmEngine


def shard_range(n: int, rank: int, world: int):
    """Contiguous split, the rule of the reference's `range()` (src/threads/threads.ts:354-359)."""
    per = -(-n // world)
    lo = min(n, per * rank)
    return lo, min(n, lo + per)


def all_gather_partials(partial: torch.Tensor) -> torch.Tensor:
    """partial: 1-D tensor (any device / backend) -> (world, len) tensor in rank order."""
    world = dist.get_world_size()
    out = torch.empty(world * partial.numel(), dtype=partial.dtype, device=partial.device)
    dist.all_gather_into_tensor(out, partial.contiguous())
    return out.view(world, partial.numel())


def exchange_comm_id(rank: int, device=None) -> bytes:
    """Rank 0 draws the NCCL unique id (mgb_comm_unique_id) and broadcasts its 128 bytes over the already
    initialised torch.distributed group -- the host-side channel of this Python host; any other (MPI, a TCP
    store, a worker message) does as well.  Works on the nccl backend (device = this rank's GPU) and on gloo."""
    from . import _native
    from .api import comm_unique_id
    dev = torch.device("cuda", device) if dist.get_backend() == "nccl" else torch.device("cpu")
    if rank == 0:
        t = torch.tensor(list(comm_unique_id()), dtype=torch.uint8, device=dev)
    else:
        t = torch.zeros(_native.COMM_ID_BYTES, dtype=torch.uint8, device=dev)
    dist.broadcast(t, src=0)
    return bytes(t.cpu().tolist())


class ShardedMsm:
    """The sharded engine.  Every rank calls the same methods with its own shard.  The data path is entirely
    inside the C library: the context owns its NCCL communicator, and `mgb_msm_sharded` runs the partial MSM,
    the all-gather of the partial sums and the combine on the engine's stream with one synchronisation.
    torch.distributed is used once, to hand the communicator id to the other ranks."""

    def __init__(self, curve, local_device: int, max_points_per_rank: int):
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.engine = MsmEngine(curve, local_device, max_points_per_rank)
        if self.world > 1:
            self.engine.comm_init(exchange_comm_id(self.rank, local_device), self.rank, self.world)

    def set_points(self, xy_bytes_shard, is_zero=None, check=False):
        """check=True: this rank's shard is checked on its device (MsmEngine.set_points); indices are shard-local."""
        return self.engine.set_points(xy_bytes_shard, is_zero, check=check)

    def random_points(self, n_local: int, seed: int):
        """Known-dlog points; rank r uses seed + r so the global set is the union of the shards."""
        self.engine.random_points(n_local, seed + self.rank)

    def msm(self, scalars, n_local: int, on_device: bool = False, c=None):
        """scalars: pinned/any host tensor or numpy array (on_device=False) or a CUDA uint8 tensor (complete
        before the call: the engine reads it on its own stream).  Every rank returns the full result."""
        if n_local == 0:
            return self.engine.msm_sharded(0, on_device, 0, c=c)
        ptr = scalars.data_ptr() if isinstance(scalars, torch.Tensor) else scalars.ctypes.data
        nbytes = scalars.numel() * scalars.element_size() if isinstance(scalars, torch.Tensor) else scalars.nbytes
        if n_local * 32 > nbytes:
            raise ValueError("msm: n_local = %d exceeds the %d scalars in the buffer" % (n_local, nbytes // 32))
        return self.engine.msm_sharded(ptr, on_device, n_local, c=c)

    def prefetch(self, scalars, n_local: int):
        """Starts the upload of this rank's NEXT host scalar set (pinned tensor or numpy array) while the current MSM
        runs; the msm(...) call that passes the same buffer and n_local then finds it on the device."""
        ptr = scalars.data_ptr() if isinstance(scalars, torch.Tensor) else scalars.ctypes.data
        nbytes = scalars.numel() * scalars.element_size() if isinstance(scalars, torch.Tensor) else scalars.nbytes
        if n_local * 32 > nbytes:
            raise ValueError("prefetch: n_local = %d exceeds the %d scalars in the buffer" % (n_local, nbytes // 32))
        self.engine.prefetch(ptr, n_local)

    def close(self):
        self.engine.close()
