"""ORACLE (test infrastructure): the attention operations themselves, in float64.

Unlike the rest of oracle/, this module is NOT a restatement of the reference's in-test functions.
It quantises nothing: softmax(Q K^T * q_scale * k_scale / sqrt(d)) V * v_scale computed in float64
from the fp8 / f32 values the kernels receive, with the paged-KV, causal and block-mask semantics of
the library's FP8 decode and prefill entry points. It is meant for the inputs of
synth/exact_scores.py, on which every quantisation step of the kernels is exact, so that a kernel
must agree with it up to one bf16 rounding of its output (`violations`).
"""
import math

import torch

BSA_BLOCK = 128


def _gather(cache, ids, seqlen):
    """cache [blocks, bs, Hkv, D] (any strides) -> float64 [Hkv, seqlen, D]."""
    hkv, d = cache.shape[2], cache.shape[3]
    return cache[ids.long()].reshape(-1, hkv, d)[:seqlen].transpose(0, 1).double()


def _gather_kscale(kscale, ids, seqlen):
    """per-token k scales f32 [blocks, bs/32, Hkv, 32] (or their fp8 view) -> float64 [Hkv, seqlen]."""
    ks = kscale.contiguous()
    if ks.element_size() == 1:
        ks = ks.view(torch.float32)
    hkv = ks.shape[2]
    return ks[ids.long()].permute(0, 1, 3, 2).reshape(-1, hkv)[:seqlen].transpose(0, 1).double()


def decode_visible(num_seq_q, seqlen, causal_shift=0):
    """bool [Sq, seqlen]: new token i (the last Sq tokens are the queries) sees kv positions
    j <= seqlen - Sq + i. `causal_shift` models a kernel whose window is off by that many keys."""
    j = torch.arange(seqlen)[None, :]
    i = torch.arange(num_seq_q)[:, None]
    return j <= seqlen - num_seq_q + i + causal_shift


def decode_log2_scores(q, kcache, block_ids, kv_lens_total, q_scale, k_scale, num_seq_q, bi,
                       k_per_token=False):
    """Scores of request `bi` in the kernels' log2 domain, S * q_scale * k_scale * log2(e)/sqrt(d):
    float64 [Hkv, Sq, group, seqlen] (all keys, visible or not)."""
    num_head_q, d = q.shape[1], q.shape[2]
    hkv, bs = kcache.shape[2], kcache.shape[1]
    g = num_head_q // hkv
    seqlen = int(kv_lens_total[bi])
    ids = block_ids[bi, :(seqlen + bs - 1) // bs]
    k = _gather(kcache, ids, seqlen)                                           # [Hkv, L, D]
    rows = slice(bi * num_seq_q, (bi + 1) * num_seq_q)
    qb = q[rows].double().reshape(num_seq_q, hkv, g, d).permute(1, 0, 2, 3)    # [Hkv, Sq, g, D]
    qs = q_scale.reshape(-1, num_head_q)[rows].double().reshape(num_seq_q, hkv, g).permute(1, 0, 2)
    s = torch.einsum("hsgd,hld->hsgl", qb, k) * (qs[..., None] * (math.log2(math.e) / math.sqrt(d)))
    if k_per_token:
        s = s * _gather_kscale(k_scale, ids, seqlen)[:, None, None, :]
    else:
        s = s * float(k_scale.reshape(-1)[0])
    return s


def decode(q, kcache, vcache, block_ids, kv_lens_total, q_scale, k_scale, v_scale, num_seq_q,
           k_per_token=False, causal_shift=0):
    """Paged FP8 decode attention (hpc.attention_decode_fp8) in float64.

      q [B*Sq, Hq, D] e4m3; kcache / vcache [blocks, 64, Hkv, D] (any strides);
      block_ids [B, max_blocks]; kv_lens_total [B] (includes the Sq new tokens);
      q_scale [B*Sq, Hq] f32, indexed per token;
      k_scale: [1] f32, or (k_per_token) the f32 scale rows [blocks, 2, Hkv, 32] (or fp8 view);
      v_scale: [1] f32, or (k_per_token) [Hkv] f32.
    Returns float64 [B*Sq, Hq, D]."""
    num_batch = kv_lens_total.shape[0]
    num_head_q, d = q.shape[1], q.shape[2]
    hkv, bs = kcache.shape[2], kcache.shape[1]
    g = num_head_q // hkv
    vs = v_scale.double().reshape(-1)
    vs = vs.reshape(hkv, 1, 1, 1) if k_per_token else vs[0]
    out = torch.empty(num_batch, num_seq_q, hkv, g, d, dtype=torch.float64)
    for bi in range(num_batch):
        seqlen = int(kv_lens_total[bi])
        ids = block_ids[bi, :(seqlen + bs - 1) // bs]
        x = decode_log2_scores(q, kcache, block_ids, kv_lens_total, q_scale, k_scale, num_seq_q, bi,
                               k_per_token)
        vis = decode_visible(num_seq_q, seqlen, causal_shift)[None, :, None, :]
        x = x.masked_fill(~vis, float("-inf"))
        w = torch.softmax(x * math.log(2.0), dim=-1)                            # [Hkv, Sq, g, L]
        y = torch.einsum("hsgl,hld->hsgd", w, _gather(vcache, ids, seqlen)) * vs
        out[bi] = y.permute(1, 0, 2, 3)
    return out.reshape(num_batch * num_seq_q, num_head_q, d)


def prefill_visible(seq_q, seq_kv, bmask_row=None, causal_shift=0):
    """bool [seq_q, seq_kv] for one (request, q head): query i (kv position seq_kv - seq_q + i) sees
    j <= seq_kv - seq_q + i + causal_shift; with a block mask row `bmask_row` bool [nrow, Kb] also
    only the 128x128 tiles set in it, plus the one tile right past the mask width (index Kb)."""
    j = torch.arange(seq_kv)[None, :]
    i = torch.arange(seq_q)[:, None]
    vis = j <= seq_kv - seq_q + i + causal_shift
    if bmask_row is not None:
        kb = bmask_row.shape[-1]
        t = torch.arange(seq_kv) // BSA_BLOCK
        qt = torch.arange(seq_q) // BSA_BLOCK
        on = torch.zeros(seq_q, seq_kv, dtype=torch.bool)
        inside = t < kb
        on[:, inside] = bmask_row.bool()[qt][:, t[inside]]
        on[:, t == kb] = True
        vis = vis & on
    return vis


def prefill(q, kcache, vcache, qscale, kscale, vscale, cu_seqlens_q, seqlens_kv, block_ids,
            block_mask=None, k_per_token=False, causal_shift=0):
    """Paged FP8 block-sparse / dense prefill (hpc.attention_with_kvcache_blocksparse_prefill_fp8,
    hpc.attention_with_kvcache_prefill_fp8) in float64.

      q [total, Hq, D] e4m3; caches [blocks, 64, Hkv, D]; qscale [B, Hq, pad] f32 (position in the
      request's queries); kscale [1] or f32 [blocks, 2, Hkv, 32]; vscale [1] or [Hkv];
      block_mask bool/u8 [B, Hq, nrow, Kb] or None.
    Returns float64 [total, Hq, D]; a row that sees no key at all is NaN, as the kernels return it."""
    total, num_head_q, d = q.shape
    hkv, bs = kcache.shape[2], kcache.shape[1]
    g = num_head_q // hkv
    out = torch.full((total, num_head_q, d), float("nan"), dtype=torch.float64)
    sc = math.log2(math.e) / math.sqrt(d)
    for bi in range(seqlens_kv.shape[0]):
        s0, s1 = int(cu_seqlens_q[bi]), int(cu_seqlens_q[bi + 1])
        nq, nkv = s1 - s0, int(seqlens_kv[bi])
        if nq == 0:
            continue
        ids = block_ids[bi, :(nkv + bs - 1) // bs]
        k = _gather(kcache, ids, nkv)
        v = _gather(vcache, ids, nkv)
        ks = _gather_kscale(kscale, ids, nkv) if k_per_token else None
        for h in range(num_head_q):
            hk = h // g
            x = (q[s0:s1, h].double() @ k[hk].t()) * (qscale[bi, h, :nq].double()[:, None] * sc)
            x = x * (ks[hk][None, :] if k_per_token else float(kscale.reshape(-1)[0]))
            bm = block_mask[bi, h] if block_mask is not None else None
            vis = prefill_visible(nq, nkv, bm, causal_shift)
            x = x.masked_fill(~vis, float("-inf"))
            w = torch.softmax(x * math.log(2.0), dim=-1)  # all -inf -> NaN row
            vsh = float(vscale.reshape(-1)[hk if k_per_token else 0])
            out[s0:s1, h] = (w @ v[hk]) * vsh
    return out


def violations(y, y64):
    """Elements of a kernel output y outside one bf16 rounding of the float64 result y64:
    |y - y64| > 2^-8 |y64| + 2^-12 max_row |y64| (row = the head dim of one token and head).
    NaN must coincide; NaN rows of y64 are otherwise ignored. Returns a bool tensor shaped like y."""
    y = y.double().cpu()
    y64 = y64.double().cpu()
    nan = torch.isnan(y64)
    rowmax = y64.abs().nan_to_num(0.0).amax(dim=-1, keepdim=True)
    bound = 2.0 ** -8 * y64.abs() + 2.0 ** -12 * rowmax
    bad = ~((y - y64).abs() <= bound)  # a NaN in y counts as a violation
    return torch.where(nan, ~torch.isnan(y), bad)


def rel_l2(y, y64):
    """Relative L2 error over the non-NaN elements of y64."""
    y = y.double().cpu()
    y64 = y64.double().cpu()
    keep = ~torch.isnan(y64)
    return float((y[keep] - y64[keep]).norm() / y64[keep].norm().clamp_min(1e-30))
