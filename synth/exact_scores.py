"""Inputs for the FP8 attention kernels on which every score is an exact integer in the kernels'
log2 domain, x = S * q_scale * k_scale * log2(e) / sqrt(128), with |x| <= 8.

Then P = 256 * 2^(x - m) is an exact power of two in e4m3 for whatever reference maximum m a kernel
uses (running maximum, lazy maximum, split-k chunk maximum), so P quantisation, chunking and tile
order drop out and a kernel must reproduce a plain float64 softmax (oracle/exact.py) up to one bf16
rounding. The construction:
  * q entries are +-1;
  * every K row has r nonzero entries of +-1, one in each of r disjoint ranges of 128 / r dims, so
    S = q . k is an integer in [-r, r] and the keys together still use all 128 dims;
  * q_scale[t, h] = 2^e * sqrt(128) / log2(e) / kappa with e in {0, 1} per (token, head), where
    kappa is the k scale per tensor, or the common factor of the per-token k scales kappa * {1, 2};
  * V is random e4m3; v scales are arbitrary (per tensor, or per kv head with per-token k scales).
The bound |x| <= r * 2 * (2 with per-token k scales) <= 8 keeps every visible key's weight at least
2^-16 of the row maximum's, far from where a kernel flushes P to zero (x - m < -17).
Unused slots of each request's last page are zero (API contract): their score 0 sits in the middle
of the range, so a kernel that failed to mask them would shift the output visibly.
"""
import math

import torch

from synth.prefill import generate_block_sparse_mask

HEAD_DIM = 128
BLOCK = 64
X_MAX = 8  # largest |x| the generator may produce
LOG2E = math.log2(math.e)


def nonzeros_per_key(k_per_token):
    """r: nonzero entries per K row (|S| <= r); per-token k scales double x once more."""
    return 2 if k_per_token else 4


def _check_bound(k_per_token):
    r = nonzeros_per_key(k_per_token)
    x_bound = r * 2 * (2 if k_per_token else 1)  # |S| * max 2^e * max per-key factor
    assert x_bound <= X_MAX, f"generator would produce |x| up to {x_bound} > {X_MAX}"


def _sign_rows(n, r, gen, dev):
    """[n, 128] float32: r entries of +-1 per row, one in each of r disjoint dim ranges."""
    span = HEAD_DIM // r
    cols = (torch.randint(0, span, (n, r), generator=gen, device=dev)
            + torch.arange(r, device=dev) * span)
    signs = torch.randint(0, 2, (n, r), generator=gen, device=dev).float() * 2 - 1
    return torch.zeros(n, HEAD_DIM, device=dev).scatter_(1, cols, signs)


def _signs(shape, gen, dev):
    return torch.randint(0, 2, shape, generator=gen, device=dev).float() * 2 - 1


def _q_scale(shape, denom, gen, dev):
    """2^e * sqrt(128) / log2(e) / denom, e in {0, 1}: x = S * 2^e (times the per-key factor)."""
    e = torch.randint(0, 2, shape, generator=gen, device=dev).double()
    return (torch.exp2(e) * math.sqrt(HEAD_DIM) / LOG2E / float(denom)).float()


def _fill_cache(num_blocks, rows, num_head_kv, r, gen, dev):
    """e4m3 [blocks, 2, rows, Hkv, 128]: K sign rows and random V in the first BLOCK rows."""
    kv = torch.zeros((num_blocks, 2, rows, num_head_kv, HEAD_DIM), dtype=torch.float8_e4m3fn,
                     device=dev)
    step = 128
    for b0 in range(0, num_blocks, step):
        n = min(step, num_blocks - b0)
        k = _sign_rows(n * BLOCK * num_head_kv, r, gen, dev).view(n, BLOCK, num_head_kv, HEAD_DIM)
        kv[b0:b0 + n, 0, :BLOCK] = k.to(torch.float8_e4m3fn)
        v = torch.randn((n, BLOCK, num_head_kv, HEAD_DIM), generator=gen, device=dev)
        kv[b0:b0 + n, 1, :BLOCK] = v.to(torch.float8_e4m3fn)
    return kv


def _page_table(kv_lens, num_blocks, gen, dev):
    """Random distinct pages per request: block_ids [B, max_blocks] int32 (cpu), pages per request."""
    nblk = [(int(L) + BLOCK - 1) // BLOCK for L in kv_lens]
    perm = torch.randperm(num_blocks, generator=gen, device=dev)[:sum(nblk)].to(torch.int32).cpu()
    block_ids = torch.zeros((len(nblk), max(nblk)), dtype=torch.int32)
    cu = 0
    for i, nb in enumerate(nblk):
        block_ids[i, :nb] = perm[cu:cu + nb]
        cu += nb
    return block_ids, nblk


def _zero_tails(kv, kv_lens, block_ids, nblk):
    """Unused slots of each request's last page: K and V zero (scale rows untouched)."""
    u8 = kv.view(torch.uint8)
    for i, L in enumerate(kv_lens):
        tail = int(L) % BLOCK
        if tail:
            u8[int(block_ids[i, nblk[i] - 1]), :, tail:BLOCK] = 0


def _per_token_kscale(num_blocks, num_head_kv, kappa, gen, dev):
    """f32 [blocks, BLOCK, Hkv] with values kappa * {1, 2}."""
    f = torch.randint(0, 2, (num_blocks, BLOCK, num_head_kv), generator=gen, device=dev).float()
    return torch.exp2(f) * kappa


def make_decode_inputs(num_batch, num_seq_q, kv_lens_total, num_head_kv, num_head_q,
                       k_per_token=False, seed=0, layout="NHD", device="cpu"):
    """Paged FP8 decode inputs with exact integer log2 scores, in the form of
    synth.decode.make_decode_fp8_inputs (kv per tensor) / make_decode_fp8_kpt_inputs (k per token:
    the f32 k scales in the cache allocation's extra rows, v scale per kv head). Both return
    kvcache, kcache, vcache, k_scale, v_scale, q [B*Sq, Hq, 128] e4m3, q_scale [B*Sq, Hq] f32,
    block_ids and kv_lens_total (which includes the Sq new tokens)."""
    _check_bound(k_per_token)
    dev = torch.device(device)
    gen = torch.Generator(device=dev).manual_seed(seed)
    lens = [int(L) for L in torch.as_tensor(kv_lens_total).reshape(-1)]
    assert len(lens) == num_batch and min(lens) >= num_seq_q
    total = sum((L + BLOCK - 1) // BLOCK for L in lens)
    num_blocks = total + total // 8 + 4
    srows = BLOCK * 4 // HEAD_DIM if k_per_token else 0
    kv = _fill_cache(num_blocks, BLOCK + srows, num_head_kv, nonzeros_per_key(k_per_token), gen, dev)
    q = _signs((num_batch * num_seq_q, num_head_q, HEAD_DIM), gen, dev).to(torch.float8_e4m3fn)
    if k_per_token:
        kappa = float(torch.rand(1, generator=gen, device=dev)) * 0.9 + 0.1
        ks = _per_token_kscale(num_blocks, num_head_kv, kappa, gen, dev)
        # bit-cast into the extra rows: row t // 32 of head h holds tokens [32 r, 32 r + 32)
        kv[:, 0, BLOCK:] = (ks.permute(0, 2, 1).contiguous().view(torch.float8_e4m3fn)
                            .reshape(num_blocks, num_head_kv, srows, HEAD_DIM).permute(0, 2, 1, 3))
        v_scale = torch.rand(num_head_kv, generator=gen, device=dev) * 0.9 + 0.1
        q_scale = _q_scale((num_batch * num_seq_q, num_head_q), kappa, gen, dev)
    else:
        k_scale = torch.rand(1, generator=gen, device=dev) * 0.95 + 0.05
        v_scale = torch.rand(1, generator=gen, device=dev) * 0.95 + 0.05
        q_scale = _q_scale((num_batch * num_seq_q, num_head_q), float(k_scale), gen, dev)
    block_ids, nblk = _page_table(lens, num_blocks, gen, dev)
    _zero_tails(kv, lens, block_ids, nblk)
    if layout == "HND":
        kv = kv.permute(0, 1, 3, 2, 4).contiguous().permute(0, 1, 3, 2, 4)
    d = dict(q=q, q_scale=q_scale, kvcache=kv, kcache=kv[:, 0, :BLOCK], vcache=kv[:, 1, :BLOCK],
             v_scale=v_scale.float(), block_ids=block_ids.to(dev),
             kv_lens_total=torch.tensor(lens, dtype=torch.int32, device=dev))
    d["k_scale"] = kv[:, 0, BLOCK:] if k_per_token else k_scale.float()
    return d


def make_prefill_inputs(q_lens, kv_lens, num_head_q, num_head_kv, skip_ratio, k_per_token, seed=0,
                        layout="nhd", device="cpu", mask_cols=None):
    """Paged FP8 prefill inputs with exact integer log2 scores, in the form of
    synth.prefill.make_inputs: q [total, Hq, 128] e4m3, caches [blocks, 64, Hkv, 128] (views),
    qscale f32 [B, Hq, pad], kscale [1] or f32 [blocks, 2, Hkv, 32] (per token), vscale [1] or
    [Hkv], cu_seqlens_q, seqlens_kv, block_ids, block_mask (None = dense) and max_q. The last
    seq_q[b] of the seq_kv[b] tokens of request b are its queries."""
    _check_bound(k_per_token)
    dev = torch.device(device)
    gen = torch.Generator(device=dev).manual_seed(seed)
    B = len(q_lens)
    assert all(0 < q <= k for q, k in zip(q_lens, kv_lens))
    total = sum(q_lens)
    max_q = max(q_lens)
    pad = (max_q + 127) // 128 * 128
    nb_total = sum((L + BLOCK - 1) // BLOCK for L in kv_lens)
    num_blocks = nb_total + nb_total // 8 + 4
    kv = _fill_cache(num_blocks, BLOCK, num_head_kv, nonzeros_per_key(k_per_token), gen, dev)
    q = _signs((total, num_head_q, HEAD_DIM), gen, dev).to(torch.float8_e4m3fn)
    if k_per_token:
        kappa = float(torch.rand(1, generator=gen, device=dev)) * 0.9 + 0.1
        ks = _per_token_kscale(num_blocks, num_head_kv, kappa, gen, dev)
        # a fresh allocation: .contiguous() would keep the odd strides of a size-1 head dim
        kscale = torch.empty((num_blocks, BLOCK // 32, num_head_kv, 32), device=dev)
        kscale.copy_(ks.view(num_blocks, BLOCK // 32, 32, num_head_kv).permute(0, 1, 3, 2))
        vscale = torch.rand(num_head_kv, generator=gen, device=dev) * 0.9 + 0.1
        qscale = _q_scale((B, num_head_q, pad), kappa, gen, dev)
    else:
        kscale = torch.rand(1, generator=gen, device=dev) * 0.95 + 0.05
        vscale = torch.rand(1, generator=gen, device=dev) * 0.95 + 0.05
        qscale = _q_scale((B, num_head_q, pad), float(kscale), gen, dev)
    block_ids, nblk = _page_table(kv_lens, num_blocks, gen, dev)
    _zero_tails(kv, kv_lens, block_ids, nblk)
    if layout == "hnd":
        kv = kv.permute(0, 1, 3, 2, 4).contiguous().permute(0, 1, 3, 2, 4)
    cu_q = torch.zeros(B + 1, dtype=torch.int32)
    cu_q[1:] = torch.cumsum(torch.tensor(q_lens), 0)
    mask = None
    if skip_ratio is not None:
        nrow = (max_q + 127) // 128
        ncol = mask_cols if mask_cols is not None else (max(kv_lens) + 127) // 128
        mask = generate_block_sparse_mask(B, num_head_q, nrow, ncol, skip_ratio, True, gen, dev)
    return dict(q=q, kcache=kv[:, 0], vcache=kv[:, 1], qscale=qscale, kscale=kscale.float(),
                vscale=vscale.float(), cu_seqlens_q=cu_q.to(dev),
                seqlens_kv=torch.tensor(kv_lens, dtype=torch.int32, device=dev),
                block_ids=block_ids.to(dev), block_mask=mask, max_q=max_q)
