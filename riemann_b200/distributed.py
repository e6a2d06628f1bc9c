"""
Multi-GPU plumbing: chains shard across ranks (each rank owns K/G chains and the Philox
substreams of its global chain ids); the only exchange is the per-batch diagnostics
all-reduce of a (6 + 3 nd)-double block (SURVEY.md section 8e).  torch.distributed
(NCCL on GPUs, gloo in the CPU tests) carries it.
"""
import numpy as np


def rank_world():
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(), dist.get_world_size()
    except Exception:
        pass
    return 0, 1


def shard_chains(K_total, rank=None, world=None):
    """Contiguous split of K_total chains: returns (chain_offset, K_local) for this rank."""
    if rank is None or world is None:
        rank, world = rank_world()
    base, rem = divmod(int(K_total), int(world))
    k_local = base + (1 if rank < rem else 0)
    offset = rank * base + min(rank, rem)
    return offset, k_local


def shard_rows(N_total, rank=None, world=None):
    """Contiguous split of the N data rows of a row-sharded model: (row_offset, N_local) for this rank."""
    return shard_chains(N_total, rank, world)


def exchange_unique_id(make_id, nbytes=128):
    """Rank 0 calls make_id(buffer, nbytes) (rmn_nccl_unique_id) and the bytes go to every rank of the
    torch.distributed group (any backend; a single process needs no group).  Returns a ctypes buffer."""
    import ctypes
    rank, world = rank_world()
    buf = ctypes.create_string_buffer(nbytes)
    if rank == 0:
        make_id(buf, nbytes)
    if world > 1:
        import torch.distributed as dist
        box = [buf.raw if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        buf = ctypes.create_string_buffer(box[0], nbytes)
    return buf


def reduce_block(blk):
    """Sum a diagnostics block over ranks (no-op without an initialised process group)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(blk, op=dist.ReduceOp.SUM)
        # entries 1 and 4 (samples / steps per chain) are identical on every rank, not additive: undo the sum with ONE
        # strided in-place division (exact: W n / W == n in fp64) instead of index gathers / puts with host-built indices
        blk[1:5:3].div_(float(dist.get_world_size()))
    return blk


def reduce_counts(t):
    """Sum an int64 count tensor over ranks, exactly (no-op without an initialised process group)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


def summarize_block(b):
    """
    b = [K, n_samples, accepts, overflows, steps, -, sum_c m_c (nd), sum_c m_c^2 (nd), sum_c v_c (nd)].
    tau = n B / W with B the variance of the chain means and W the mean within-chain
    variance; ESS = K n / tau; R-hat from (n-1)/n W + B.
    """
    b = np.asarray(b, dtype=np.float64)
    H = 6
    nd = (len(b) - H) // 3
    K, n, steps = b[0], b[1], b[4]
    sm, sm2, sv = b[H:H + nd], b[H + nd:H + 2 * nd], b[H + 2 * nd:H + 3 * nd]
    mean = sm / K
    with np.errstate(divide="ignore", invalid="ignore"):
        B = (sm2 - sm * sm / K) / max(K - 1.0, 1.0)
        W = sv / K * (n / max(n - 1.0, 1.0))
        tau_s = np.where(W > 0, n * B / W, np.nan)          # in units of accumulated samples
        ess = np.where(tau_s > 0, K * n / tau_s, np.nan)     # = K W / B, independent of the thinning
        tau = tau_s * (steps / max(n, 1.0))                  # in MH steps
        rhat = np.sqrt(((n - 1.0) / n * W + B) / W)
    return {"chains": int(K), "steps": int(steps), "samples": int(n),
            "accept_rate": b[2] / max(K * steps, 1.0),
            "overflows": int(b[3]), "mean": mean, "var": W + B, "within_var": W,
            "between_var": B, "tau": tau, "ess": ess, "rhat": rhat,
            "min_ess": float(np.nanmin(ess)) if nd and np.any(np.isfinite(ess)) else float("nan")}


def summarize_split(block_a, block_b):
    """
    Split-chain diagnostics (Gelman et al., BDA3 / Stan's split-R-hat) from the diagnostics blocks of two
    consecutive windows of equal length: every chain's two halves are treated as separate chains, so a chain
    whose mean drifts between the halves raises R-hat even when all chains drift alike.  The blocks' chain sums
    are additive, so the 2K half-chains' between-variance B and within-variance W follow from the two blocks:
        tau = n_half B / W (in samples), ESS = 2K n_half / tau, R-hat = sqrt(((n-1)/n W + B) / W).
    Returns the same keys as summarize_block (`chains` = 2K half-chains, `steps` = half-window length).
    """
    a, b = np.asarray(block_a, dtype=np.float64), np.asarray(block_b, dtype=np.float64)
    if a.shape != b.shape or a[0] != b[0] or a[1] != b[1] or a[4] != b[4]:
        raise ValueError("summarize_split needs two blocks of the same chains and window length")
    c = a.copy()
    c[0] = a[0] + b[0]                     # 2K half-chains
    c[2] = a[2] + b[2]                     # accepts
    c[3] = a[3] + b[3]                     # overflow events
    H = 6
    c[H:] = a[H:] + b[H:]                  # sum m, sum m^2, sum v over the 2K half-chains
    out = summarize_block(c)
    out["accept_rate"] = c[2] / max(a[0] * (a[4] + b[4]), 1.0)
    return out
