"""
Multi-GPU: chains shard by rank with no per-iteration communication (SURVEY.md section 8e).  The collectives are the
merge of the per-rank Welford posterior moments and, when convergence diagnostics are requested, the partial sums of the split
R-hat -- two sum all-reduces each (NCCL over NVLink on GPUs; gloo in CPU tests) --, for the segmentation posterior, one sum
all-reduce of the integer label counts, for the Jacobian posterior two sum all-reduces of its per-voxel Welford moments, and
for the landmark posterior two fp64 sum all-reduces of its per-landmark moments.

The reference has no distributed code at all; the quantity computed here is its calc_posterior_statistics
(utils/util.py:114-120: mean and unbiased std over every kept sample of every chain).
"""
import torch
import torch.distributed as dist


def chain_shard(no_chains_total, rank=None, world_size=None):
    """contiguous block of global chain ids owned by `rank`: [offset, offset + count)"""
    if rank is None:
        rank = dist.get_rank() if dist.is_initialized() else 0
    if world_size is None:
        world_size = dist.get_world_size() if dist.is_initialized() else 1
    base, extra = divmod(no_chains_total, world_size)
    count = base + (1 if rank < extra else 0)
    offset = rank * base + min(rank, extra)
    return offset, count


def any_rank(flag, device=None, group=None):
    """logical OR of a host flag over all ranks (one tiny MAX all-reduce); the flag itself without torch.distributed"""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return bool(flag)
    t = torch.tensor([1 if flag else 0], device=device if dist.get_backend(group) == 'nccl' else 'cpu', dtype=torch.int32)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return bool(t.item())


def split_rhat_totals(n_seq_local, sums, between, group=None):
    """
    The two collective phases of the split R-hat (ops.split_rhat), in the pattern of merge_moments.
      sums     (2, E) fp64: this rank's S1 = sum_j mean_j and SW = sum_j M2_j / (n - 1) over its n_seq_local sequences
      between  callable (s1_total (E,) fp64, M) -> this rank's SB = sum_j (mean_j - s1_total / M)^2, (E,) fp64
    Phase A sum-all-reduces (M, S1, SW) as one buffer (the sequence count rides in front, padded to 2 doubles), phase B the SB
    partials.  Returns (M, sums (2, E), SB (E,)) -- the totals over all ranks, identical on every rank.  Pure torch on the
    partial-sum tensors: NCCL on GPUs, gloo in CPU tests.  One host read (M) between the phases.
    """
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return n_seq_local, sums, between(sums[0], n_seq_local)
    E = sums.shape[1]
    buf = torch.empty(2 + 2 * E, device=sums.device, dtype=torch.float64)
    buf[:2] = float(n_seq_local)
    buf[2:].view(2, E).copy_(sums)
    dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    M = int(round(float(buf[0].item())))
    total = buf[2:].view(2, E)
    sb = between(total[0], M)
    dist.all_reduce(sb, op=dist.ReduceOp.SUM, group=group)
    return M, total, sb


def merge_label_counts(n_local, counts, group=None):
    """
    The label counts of the segmentation posterior (ops.label_counts_update) summed over the ranks of `group`: one SUM
    all-reduce of one int32 buffer, the number of accumulated segmentations riding in front (padded to 4 ints so that the
    counts stay 16-byte aligned).  Integer sums: the result does not depend on how the chains are split over ranks.
    Returns (n_total, counts_total) as new tensors, identical on every rank; the local counts are left as they are, so sampling
    can go on after a query.  One host read (n_total).
    """
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return int(n_local), counts.clone()
    buf = torch.empty(4 + counts.numel(), device=counts.device, dtype=torch.int32)
    buf[:4] = int(n_local)
    buf[4:].view_as(counts).copy_(counts)
    dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    return int(buf[0].item()), buf[4:].view_as(counts)


def merge_jacobian_moments(n_local, folds, mean, m2, group=None):
    """
    The accumulators of the Jacobian posterior (ops.jacobian_update) over the ranks of `group`: Chan's merge with the per-voxel
    count n_v = n - folds of finite samples,
        n_v = sum_r n_v,r ;  mean = sum_r n_v,r mean_r / n_v ;  M2 = sum_r [ M2_r + n_v,r (mean_r - mean)^2 ]
    in two SUM all-reduces of fp32 buffers in the style of merge_moments: the first carries n in front (padded to 4 floats),
    n_v and n_v mean, the second the M2 terms.  Integer counts are exact in fp32 below 2^24 samples, so the folds come back
    exactly as n - sum n_v; mean is 0 where no rank has a finite sample.  Returns (n_total, folds, mean, m2) as new tensors,
    identical on every rank; the local accumulators are kept, so sampling can continue.  One host read (n_total).
    """
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return int(n_local), folds.clone(), mean.clone(), m2.clone()
    V = folds.numel()
    nv_local = (int(n_local) - folds).to(torch.float32)
    buf = torch.empty(4 + 2 * V, device=mean.device, dtype=torch.float32)
    buf[:4] = float(n_local)
    nv, s = buf[4:4 + V].view_as(mean), buf[4 + V:].view_as(mean)
    nv.copy_(nv_local.view_as(mean))
    torch.mul(mean, nv, out=s)
    dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    n_total = int(round(float(buf[0].item())))
    if n_total >= 1 << 24:
        raise ValueError(f'{n_total} samples: the Jacobian posterior counts are exact below 2^24')
    mean_t = torch.where(nv > 0, s / nv.clamp(min=1.0), torch.zeros_like(s))
    d = mean - mean_t
    m2_t = torch.addcmul(m2, d, d * nv_local.view_as(mean))
    dist.all_reduce(m2_t, op=dist.ReduceOp.SUM, group=group)
    folds_t = (n_total - nv.to(torch.int32)).view_as(folds)
    return n_total, folds_t, mean_t, m2_t


def merge_landmark_moments(n_local, acc, group=None):
    """
    The landmark accumulators acc (P, 11) fp64 (ops.landmark_update: mean (3), co-moments xx xy xz yy yz zz (6), TRE mean,
    TRE M2) over the ranks of `group`: Chan's merge with n_r samples on rank r,
        n = sum_r n_r ;  mean = sum_r n_r mean_r / n ;  M_ab = sum_r [ M_ab,r + n_r (mean_r - mean)_a (mean_r - mean)_b ]
    for the position and the same for the TRE, in two fp64 SUM all-reduces: the first carries n in front and the n_r-weighted
    means, the second the co-moment terms.  A rank without samples contributes nothing.  Returns (n_total, acc) with a new
    tensor, identical on every rank; the local accumulators are kept, so sampling can continue.  One host read (n_total).
    """
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return int(n_local), acc.clone()
    P = acc.shape[0]
    n_r = float(n_local)
    buf = torch.empty(1 + 4 * P, device=acc.device, dtype=torch.float64)
    buf[0] = n_r
    sums = buf[1:].view(P, 4)
    torch.mul(acc[:, [0, 1, 2, 9]], n_r, out=sums)
    dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    n_total = int(buf[0].item())
    if n_total < 1:
        return 0, torch.zeros_like(acc)
    mean = sums / float(n_total)
    d = acc[:, [0, 1, 2, 9]] - mean
    out = torch.empty_like(acc)
    out[:, [0, 1, 2, 9]] = mean
    a, b = [0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]
    out[:, 3:9] = acc[:, 3:9] + n_r * d[:, a] * d[:, b]
    out[:, 10] = acc[:, 10] + n_r * d[:, 3] * d[:, 3]
    m = out[:, [3, 4, 5, 6, 7, 8, 10]].contiguous()
    dist.all_reduce(m, op=dist.ReduceOp.SUM, group=group)
    out[:, 3:9] = m[:, :6]
    out[:, 10] = m[:, 6]
    return n_total, out


def merge_moments(n_local, moments, group=None):
    """
    Chan et al. parallel merge of Welford triples.  `moments` is a list of (mean, M2) tensor pairs that share the
    sample count n_local.  Returns (n_total, (mean, M2), ...) identical on every rank.
        mean = sum_r n_r mean_r / N ;   M2 = sum_r [ M2_r + n_r (mean_r - mean)^2 ]
    Two sum all-reduces of ONE packed fp32 buffer each (the payload in its own precision: 32 MiB per phase at 128^3);
    the sample count rides in the first buffer, so nothing returns to the host between the phases -- the only
    synchronisation is the final read of N.
    """
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return (n_local,) + tuple((m.clone(), m2.clone()) for m, m2 in moments)

    ref = moments[0][0]
    sizes = [m.numel() for m, _ in moments]
    total = sum(sizes)
    # element 0 carries n (exact in fp32 up to 2^24 samples per rank; the sum is formed in the all-reduce), padded to 4 floats
    # so that the payload views stay 16-byte aligned
    buf = torch.empty(4 + total, device=ref.device, dtype=torch.float32)
    buf[:4] = float(n_local)
    views, o = [], 4
    for (m, _), k in zip(moments, sizes):
        views.append(buf[o:o + k].view_as(m))
        torch.mul(m, float(n_local), out=views[-1])
        o += k
    dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    n_total = buf[0]                                    # device scalar
    means = [v / n_total for v in views]

    buf2 = torch.empty(total, device=ref.device, dtype=torch.float32)
    out, o = [], 0
    for (m, m2), mg, k in zip(moments, means, sizes):
        d = m - mg
        part = buf2[o:o + k].view_as(m2)
        torch.addcmul(m2, d, d, value=float(n_local), out=part)
        out.append((mg, part))
        o += k
    dist.all_reduce(buf2, op=dist.ReduceOp.SUM, group=group)
    return (int(round(float(n_total.item()))),) + tuple(out)
