"""Sharding of chains across ranks and the algebra of the pooled-statistics all-reduce (SURVEY.md §8e).

Chains are independent (the reference is a single chain; an ensemble is N replicas with different RNG
sub-streams), so stepping needs no communication.  The only collective of the path is a sum all-reduce of the
shifted raw moments ``[sum(x-s), sum (x-s)(x-s)^T, sum obs]`` (plus counts) at measure / reporting boundaries.
Everything here is plain tensor code so that it can be exercised with the ``gloo`` backend on CPU.
"""
import numpy as np
import torch


def shard_range(n_total, rank, world_size, granule=1):
    """Contiguous global chain-id range [lo, hi) owned by ``rank``.  The Philox counter of a chain carries its
    GLOBAL id, so results do not depend on ``world_size``.  ``granule``: the range is made of whole groups of that
    many chains (the ladders of a tempering engine); ``n_total`` must be a multiple of it."""
    if n_total % granule:
        raise ValueError("n_total (%d) is not a multiple of the granule (%d)" % (n_total, granule))
    units = n_total // granule
    if units < world_size:
        raise ValueError("fewer chains (%d) than ranks (%d)" % (n_total, world_size) if granule == 1 else
                         "fewer ladders (%d) than ranks (%d)" % (units, world_size))
    base, rem = divmod(units, world_size)
    lo = rank * base + min(rank, rem)
    hi = lo + base + (1 if rank < rem else 0)
    return lo * granule, hi * granule


def world(group=None):
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def allreduce_sum_(t, group=None):
    """In-place sum all-reduce when a process group is up (NCCL for CUDA tensors, gloo for CPU); identity
    otherwise."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


def pool_words(n_real, n_complex):
    d = n_real + 2 * n_complex
    return d + d * (d + 1) // 2 + 2 * n_real + n_complex


def pooled_moments_reference(samples, shift, n_real, n_complex):
    """Moment vector in the kernel's layout, computed with numpy from explicit samples [N, D] (tests)."""
    x = np.asarray(samples, dtype=np.float64)
    d = n_real + 2 * n_complex
    dx = x - np.asarray(shift)[None, :]
    out = [dx.sum(0)]
    il = np.tril_indices(d)
    out.append((dx[:, il[0]] * dx[:, il[1]]).sum(0))
    obs = [np.abs(x[:, :n_real]), np.hypot(x[:, n_real:n_real + n_complex], x[:, n_real + n_complex:]),
           x[:, :n_real] ** 2]
    out.append(np.concatenate(obs, axis=1).sum(0))
    return np.concatenate(out)


def finalize_pooled(sums, count, shift, n_real, n_complex):
    """Pooled ensemble statistics from the all-reduced moment vector.

    Returns dict(mean_real, mean_complex, cov_real, cov_complex, observables_mean, count); covariances are the
    unbiased sample covariances over every (chain, measure) sample — the *clean* ensemble estimate, unlike the
    reference's per-chain recursion which carries the sigma^2/n regulariser (SURVEY App. B-7).
    """
    sums = np.asarray(sums, dtype=np.float64)
    shift = np.asarray(shift, dtype=np.float64)
    d = n_real + 2 * n_complex
    n = float(count)
    s1 = sums[:d]
    il = np.tril_indices(d)
    s2 = np.zeros((d, d))
    s2[il] = sums[d:d + d * (d + 1) // 2]
    s2 = s2 + np.tril(s2, -1).T
    obs = sums[d + d * (d + 1) // 2:]
    mean = shift + s1 / n
    cov = (s2 - np.outer(s1, s1) / n) / max(n - 1.0, 1.0)
    nr, nc = n_real, n_complex
    re, im = slice(nr, nr + nc), slice(nr + nc, nr + 2 * nc)
    cov_c = (cov[re, re] + cov[im, im]) + 1j * (cov[im, re] - cov[re, im])
    return dict(mean_real=mean[:nr].copy(), mean_complex=mean[re] + 1j * mean[im], cov_real=cov[:nr, :nr].copy(),
                cov_complex=cov_c, observables_mean=obs / n, count=int(count))


_LIBRARY_COMMS = {}


def nccl_library_path():
    """The NCCL shared object the process already carries (torch's bundled copy), for me_comm_set_library."""
    import os
    try:
        import nvidia.nccl as nv
        base = list(nv.__path__)[0]
        cand = os.path.join(base, "lib", "libnccl.so.2")
        if os.path.exists(cand):
            return cand
    except Exception:
        pass
    return None


def library_comm(lib, device_index, group=None):
    """The library-side NCCL communicator (``me_comm``, include/me_b200.h) of this rank, created once per device:
    rank 0 draws the NCCL unique id inside the library, torch.distributed carries the 128 bytes to the other ranks,
    every rank joins with ``me_comm_create``.  Returns a ctypes handle (None when there is one rank or no CUDA
    process group) — ``me_allreduce_stats`` then runs the collective inside the library, stream-ordered, with no host
    round trip."""
    import ctypes
    import torch.distributed as dist
    rank, world_size = world(group)
    if world_size <= 1 or dist.get_backend(group) != "nccl":
        return None
    key = (device_index, id(group))
    if key in _LIBRARY_COMMS:
        return _LIBRARY_COMMS[key]
    path = nccl_library_path()
    if path:
        lib.me_comm_set_library(path.encode())
    buf = (ctypes.c_ubyte * 128)()
    if rank == 0:
        rc = lib.me_comm_unique_id(buf)
        if rc != 0:
            raise RuntimeError("me_comm_unique_id: " + lib.me_comm_last_error().decode())
    box = [bytes(buf)]
    dist.broadcast_object_list(box, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    ident = (ctypes.c_ubyte * 128).from_buffer_copy(box[0])
    comm = ctypes.c_void_p()
    rc = lib.me_comm_create(ident, world_size, rank, device_index, ctypes.byref(comm))
    if rc != 0:
        raise RuntimeError("me_comm_create: " + lib.me_comm_last_error().decode())
    connect_peer_windows(lib, comm, rank, world_size, device_index, group)
    _LIBRARY_COMMS[key] = comm
    return comm


# Vectors up to this many doubles go through the peer windows: the pooled-moment vectors of the fused engines (<= 601
# doubles, one chunk = one CTA).  The 16,656-double moment vector of the shared-covariance path stays on NCCL: its step kernel
# leaves one SM to the side stream and there NCCL's all-reduce measured faster at 8 ranks (bench c4: 1.60e10 against
# 1.35e10 chain-steps/s); ME_PEER_WINDOW_DOUBLES raises the limit (<= 32768).
PEER_WINDOW_DOUBLES = 1 << 10


def connect_peer_windows(lib, comm, rank, world_size, device_index, group=None):
    """Set up the one-shot NVLink all-reduce of a library communicator (``me_comm_peer_*``, include/me_b200.h): every rank
    allocates its window and exports a CUDA IPC handle, torch.distributed carries the handles, every rank opens its
    peers' windows, and only when ALL ranks succeeded are the windows switched on (otherwise — ranks on different
    boxes, IPC not permitted, ``ME_PEER_ALLREDUCE=0`` — the collectives stay on NCCL).  Returns whether they are on."""
    import ctypes
    import os
    import torch
    import torch.distributed as dist
    want = os.environ.get("ME_PEER_ALLREDUCE", "1") != "0"
    dev = torch.device("cuda", device_index)
    handle = (ctypes.c_ubyte * 64)()
    limit = int(os.environ.get("ME_PEER_WINDOW_DOUBLES", PEER_WINDOW_DOUBLES))
    ok = want and lib.me_comm_peer_init(comm, limit, handle) == 0
    mine = torch.tensor(list(bytes(handle)) + [1 if ok else 0], dtype=torch.uint8, device=dev)
    every = torch.empty((world_size, 65), dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(every, mine, group=group)
    every = every.cpu().numpy()
    ok = bool(every[:, 64].all())
    if ok:
        handles = (ctypes.c_ubyte * (64 * world_size)).from_buffer_copy(every[:, :64].tobytes())
        ok = lib.me_comm_peer_connect(comm, handles) == 0
    flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
    ok = int(flag.item()) == 1
    if ok:
        ok = lib.me_comm_peer_enable(comm, 1) == 0
    _PEER_WINDOWS[comm.value] = ok
    return ok


_PEER_WINDOWS = {}


def peer_windows_on(comm):
    """Whether the collectives of this library communicator run over the NVLink peer windows."""
    return bool(comm is not None and _PEER_WINDOWS.get(comm.value, False))
