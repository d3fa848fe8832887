"""Exact-score inputs (synth/exact_scores.py) and the float64 attention reference (oracle/exact.py),
CPU only.

* the generator keeps its promises: integer log2 scores, |x| <= 8, zero page tails;
* on these inputs the reference-semantics oracles (pinned to the reference's goldens) agree with
  the float64 softmax within one bf16 rounding, which ties the new reference to the pinned ones;
* kernels with plausible bugs (modelled by mutating the inputs or the mask) violate that tolerance,
  which is what lets the GPU tests built on it fail;
* the restatement of the decode bin walk finds the rotated-walk features the GPU tests rely on.
"""
import numpy as np
import pytest
import torch

from oracle import attention as oa
from oracle import decode_walk as dw
from oracle import exact as ox
from oracle import prefill as op
from oracle import taskmap as otm
from synth import exact_scores as xs

DECODE_CASES = [  # (Hkv, Hq, Sq, lens, layout)
    (2, 8, 1, [1, 63, 64, 65, 129, 300], "NHD"),
    (1, 8, 4, [4, 127, 128, 257], "HND"),
    (4, 32, 2, [2, 200, 700], "NHD"),
]


def _decode(kpt, case, seed=1):
    hkv, hq, sq, lens, layout = case
    lens = [max(L, sq) for L in lens]
    d = xs.make_decode_inputs(len(lens), sq, lens, hkv, hq, k_per_token=kpt, seed=seed, layout=layout)
    return d, sq


def _exact_decode(d, sq, kpt, **kw):
    return ox.decode(d["q"], d["kcache"], d["vcache"], d["block_ids"], d["kv_lens_total"],
                     d["q_scale"], d["k_scale"], d["v_scale"], sq, k_per_token=kpt, **kw)


def _oracle_decode(d, sq, kpt, **kw):
    f = oa.decode_fp8_kpertoken if kpt else oa.decode_fp8_kvpertensor
    return f(d["q"], d["kcache"], d["vcache"], d["block_ids"], d["kv_lens_total"], d["q_scale"],
             d["k_scale"], d["v_scale"], sq, **kw)


def _prefill(kpt, skip, seed=2, **kw):
    return xs.make_prefill_inputs([1, 130, 257, 64], [1, 130, 900, 1000], 8, 2, skip, kpt,
                                  seed=seed, **kw)


def _exact_prefill(d, kpt, **kw):
    return ox.prefill(d["q"], d["kcache"], d["vcache"], d["qscale"], d["kscale"], d["vscale"],
                      d["cu_seqlens_q"], d["seqlens_kv"], d["block_ids"], d["block_mask"], kpt, **kw)


def _oracle_prefill(d, kpt):
    return op.blocksparse_prefill(d["q"], d["kcache"], d["vcache"], d["qscale"], d["kscale"],
                                  d["vscale"], d["cu_seqlens_q"], d["seqlens_kv"], d["block_ids"],
                                  d["block_mask"], kpt)


def _fails(y, y64, tag):
    n = int(ox.violations(y, y64).sum())
    assert n > 0, f"{tag}: a kernel with this bug would pass (rel L2 {ox.rel_l2(y, y64):.4f})"


# ------------------------------------------------------------------------------------------------
# generator invariants
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kpt", [False, True])
@pytest.mark.parametrize("case", DECODE_CASES)
def test_decode_generator_invariants(kpt, case):
    d, sq = _decode(kpt, case)
    lens = d["kv_lens_total"].tolist()
    for bi, L in enumerate(lens):
        x = ox.decode_log2_scores(d["q"], d["kcache"], d["block_ids"], d["kv_lens_total"],
                                  d["q_scale"], d["k_scale"], sq, bi, k_per_token=kpt)
        assert (x - x.round()).abs().max() < 1e-5, "log2 scores are not integers"
        assert x.abs().max() <= xs.X_MAX + 1e-5
        assert x.round().abs().max() >= 2  # not degenerate
        nb = (L + 63) // 64
        last = int(d["block_ids"][bi, nb - 1])
        if L % 64:
            assert d["kcache"][last, L % 64:].view(torch.uint8).sum() == 0
            assert d["vcache"][last, L % 64:].view(torch.uint8).sum() == 0
    # q scale exponents vary per (token, head): a wrong index changes the temperature
    e = torch.log2(d["q_scale"].double() * float(d["q_scale"].min()) ** -1).round()
    assert set(e.unique().tolist()) == {0.0, 1.0}


@pytest.mark.parametrize("kpt", [False, True])
def test_prefill_generator_invariants(kpt):
    d = _prefill(kpt, None)
    sc = np.log2(np.e) / np.sqrt(128)
    for bi in range(4):
        s0, s1 = int(d["cu_seqlens_q"][bi]), int(d["cu_seqlens_q"][bi + 1])
        L = int(d["seqlens_kv"][bi])
        ids = d["block_ids"][bi, :(L + 63) // 64]
        k = ox._gather(d["kcache"], ids, L)
        ks = ox._gather_kscale(d["kscale"], ids, L) if kpt else None
        for h in (0, 7):
            x = (d["q"][s0:s1, h].double() @ k[h // 4].t()) * d["qscale"][bi, h, :s1 - s0].double()[:, None] * sc
            x = x * (ks[h // 4][None] if kpt else float(d["kscale"][0]))
            assert (x - x.round()).abs().max() < 1e-5 and x.abs().max() <= xs.X_MAX + 1e-5
        if L % 64:
            last = int(ids[-1])
            assert d["kcache"][last, L % 64:].view(torch.uint8).sum() == 0


# ------------------------------------------------------------------------------------------------
# the pinned reference-semantics oracles agree with the float64 softmax on these inputs
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kpt", [False, True])
@pytest.mark.parametrize("case", DECODE_CASES)
def test_pinned_decode_oracle_matches_float64(kpt, case):
    d, sq = _decode(kpt, case)
    y64 = _exact_decode(d, sq, kpt)
    bad = ox.violations(_oracle_decode(d, sq, kpt), y64)
    assert int(bad.sum()) == 0, f"{int(bad.sum())} elements outside one bf16 rounding"


@pytest.mark.parametrize("kpt", [False, True])
@pytest.mark.parametrize("skip", [None, 0.5])
def test_pinned_prefill_oracle_matches_float64(kpt, skip):
    d = _prefill(kpt, skip)
    y64 = _exact_prefill(d, kpt)
    y = _oracle_prefill(d, kpt)
    assert int(ox.violations(y, y64).sum()) == 0
    if skip is not None:
        assert torch.isnan(y64).any()  # the ragged masks leave some rows without any key


def test_float64_prefill_extra_tile_past_mask_width():
    d = xs.make_prefill_inputs([1024], [1024], 4, 1, 0.3, False, seed=5)
    d["block_mask"] = d["block_mask"][:, :, :, :5].contiguous()
    assert int(ox.violations(_oracle_prefill(d, False), _exact_prefill(d, False)).sum()) == 0


# ------------------------------------------------------------------------------------------------
# sensitivity: kernels with these bugs violate the tolerance
# ------------------------------------------------------------------------------------------------
def _roll_heads_in_group(t, group):
    """[rows, Hq, ...]: every q head takes its neighbour's data within its GQA group."""
    s = t.shape
    g = t.reshape(s[0], s[1] // group, group, *s[2:])
    return torch.roll(g.float(), 1, dims=2).to(t.dtype).reshape(s)


def _roll_tokens_in_request(t, sq):
    """[B*Sq, ...]: every token takes the neighbouring token's row within its request."""
    s = t.shape
    return torch.roll(t.float().reshape(-1, sq, *s[1:]), 1, dims=1).to(t.dtype).reshape(s)


@pytest.mark.parametrize("kpt", [False, True])
@pytest.mark.parametrize("case", DECODE_CASES)
def test_decode_mutations_violate_tolerance(kpt, case):
    d, sq = _decode(kpt, case)
    hq, hkv = d["q"].shape[1], d["kcache"].shape[2]
    y64 = _exact_decode(d, sq, kpt)
    _fails(_oracle_decode(dict(d, q=torch.zeros_like(d["q"].float()).to(d["q"].dtype)), sq, kpt),
           y64, "q = 0")
    _fails(_oracle_decode(dict(d, q=_roll_heads_in_group(d["q"], hq // hkv)), sq, kpt), y64,
           "neighbouring q head")
    _fails(_oracle_decode(dict(d, q_scale=_roll_heads_in_group(d["q_scale"], hq // hkv)), sq, kpt),
           y64, "q scale of the neighbouring head")
    _fails(_exact_decode(d, sq, kpt, causal_shift=-1).to(torch.bfloat16), y64,
           "dropped last visible key")
    if sq > 1:
        _fails(_oracle_decode(d, sq, kpt, per_token_qscale=False), y64, "q scale per batch")
        _fails(_oracle_decode(dict(d, q_scale=_roll_tokens_in_request(d["q_scale"], sq)), sq, kpt),
               y64, "q scale of the neighbouring token")
        _fails(_exact_decode(d, sq, kpt, causal_shift=1).to(torch.bfloat16), y64,
               "causal window off by one")
    if kpt:
        ks = d["k_scale"].contiguous().view(torch.float32)  # [blocks, 2, Hkv, 32]
        nb = ks.shape[0]
        tok = ks.permute(0, 1, 3, 2).reshape(nb, 64, hkv)
        rolled = torch.roll(tok, 1, dims=1).reshape(nb, 2, 32, hkv).permute(0, 1, 3, 2)
        _fails(_oracle_decode(dict(d, k_scale=rolled), sq, kpt), y64, "k scale of the neighbouring token")
        if hkv > 1:
            _fails(_oracle_decode(dict(d, k_scale=torch.roll(ks, 1, dims=2)), sq, kpt), y64,
                   "k scale of the neighbouring kv head")
    else:
        _fails(_oracle_decode(dict(d, k_scale=d["k_scale"] * 2), sq, kpt), y64, "k scale doubled")


@pytest.mark.parametrize("kpt", [False, True])
def test_prefill_mutations_violate_tolerance(kpt):
    d = _prefill(kpt, 0.5)
    y64 = _exact_prefill(d, kpt)
    _fails(_oracle_prefill(dict(d, q=torch.zeros_like(d["q"].float()).to(d["q"].dtype)), kpt), y64, "q = 0")
    _fails(_oracle_prefill(dict(d, q=_roll_heads_in_group(d["q"], 4)), kpt), y64, "neighbouring q head")
    _fails(_oracle_prefill(dict(d, qscale=torch.roll(d["qscale"], 1, dims=2)), kpt), y64,
           "q scale of the neighbouring token")
    _fails(_exact_prefill(d, kpt, causal_shift=1).to(torch.bfloat16), y64, "causal window off by one")
    _fails(_exact_prefill(d, kpt, causal_shift=-1).to(torch.bfloat16), y64, "dropped last visible key")
    _fails(_oracle_prefill(dict(d, block_mask=None), kpt), y64, "block mask ignored")
    if kpt:
        _fails(_oracle_prefill(dict(d, kscale=torch.roll(d["kscale"], 1, dims=3)), kpt), y64,
               "k scale of the neighbouring token")
        _fails(_oracle_prefill(dict(d, kscale=torch.roll(d["kscale"], 1, dims=2)), kpt), y64,
               "k scale of the neighbouring kv head")


# ------------------------------------------------------------------------------------------------
# bin-walk restatement on the scheduler's task maps (148 bins, the B200's SM count)
# ------------------------------------------------------------------------------------------------
def _host_map(lens, hkv, sq, mpl, ctas=148):
    m = otm.assign(lens, ctas, hkv, sq, 128, True, mpl).reshape(-1).copy()
    m[6] = sum((L + 127) // 128 for L in lens)  # tiles per kv head, as the device workspace holds it
    return m


def test_walk_visits_every_tile_once():
    for lens, hkv, sq, mpl in (([40000], 2, 2, 64), ([8192] * 64, 8, 1, 64),
                               ([3, 63, 64, 65, 257, 1000, 40000], 2, 3, 1024)):
        for w in dw.walks(_host_map(lens, hkv, sq, mpl)):
            seen = [(r, t) for r, tb, te in w.segments() for t in range(tb, te)]
            want = [(r, t) for r in range(len(w.rows)) for t in range(int(w.rows[r, 6]))]
            assert sorted(seen) == want and len(seen) == len(set(seen))


def test_walk_features_on_ragged_lengths():
    """Ragged lengths up to 40000 over two kv heads, MTP 2: splits (also of a task holding the
    causal tail), a bin across the head boundary, a short last bin."""
    lens = [2, 63, 64, 65, 127, 128, 129, 255, 256, 257, 1000, 2500, 40000, 2]
    ws = dw.walks(_host_map(lens, 2, 2, 1024))
    assert any(w.split for w in ws)
    assert any(w.straddles_heads for w in ws)
    assert any(w.short for w in ws)
    assert any(w.split and int(w.rows[w.ks, 8]) for w in ws)
