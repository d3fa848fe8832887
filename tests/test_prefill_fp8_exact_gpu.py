"""FP8 paged prefill (dense and block-sparse, both quant schemes) against a float64 softmax, on inputs
whose log2 scores are exact integers (synth/exact_scores.py): P = 256 * 2^(x - mref) is exact in
e4m3 for the kernel's lazy reference maximum too, so the output must equal the float64 result up to
one bf16 rounding (oracle.exact.violations), and the rows that see no key must be NaN exactly where
the reference has them."""
import os
import subprocess
import sys
from pathlib import Path

import pytest
import torch

from oracle import exact as ox
from synth import exact_scores as xs

pytestmark = pytest.mark.gpu

# ragged requests: one token, lengths off the 128 / 64 grid, q shorter than kv (chunked prefill
# over an existing cache), a request whose queries are its whole cache
Q_LENS = [1, 130, 257, 64, 384]
KV_LENS = [1, 130, 900, 1000, 384]


def _qt(hpc, kpt):
    return (hpc.QuantType.QPERTOKEN_PERHEAD_KPERTOKEN_PERHEAD_VPERHEAD if kpt
            else hpc.QuantType.QPERTOKEN_PERHEAD_KPERTENSOR_VPERTENSOR)


def _run(hpc, d, kpt, dense_entry=False):
    c = {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in d.items()}
    args = (c["q"], c["kcache"], c["vcache"], c["qscale"], c["kscale"], c["vscale"],
            c["cu_seqlens_q"], c["block_ids"], c["seqlens_kv"], d["max_q"])
    if dense_entry:
        return hpc.attention_with_kvcache_prefill_fp8(*args, quant_type=_qt(hpc, kpt))
    mask = c["block_mask"].to(torch.uint8).contiguous() if c["block_mask"] is not None else None
    return hpc.attention_with_kvcache_blocksparse_prefill_fp8(*args, quant_type=_qt(hpc, kpt),
                                                              block_mask=mask)


def _reference(d, kpt):
    c = {k: (v.cpu() if isinstance(v, torch.Tensor) else v) for k, v in d.items()}
    return ox.prefill(c["q"], c["kcache"], c["vcache"], c["qscale"], c["kscale"], c["vscale"],
                      c["cu_seqlens_q"], c["seqlens_kv"], c["block_ids"], c["block_mask"], kpt)


def _check(y, y64, d, tag):
    y = y.float().cpu()
    bad = ox.violations(y, y64)
    if bool(bad.any()):
        t, h, dim = (int(i) for i in bad.nonzero()[0])
        cu = d["cu_seqlens_q"].cpu().tolist()
        b = max(i for i in range(len(cu) - 1) if cu[i] <= t)
        pos = t - cu[b]
        pytest.fail(f"{tag}: {int(bad.sum())} elements outside one bf16 rounding or NaN pattern "
                    f"(rel L2 {ox.rel_l2(y, y64):.4f}); first at request {b}, query {pos} (Q tile "
                    f"{pos // 128}), q head {h}, dim {dim}: got {float(y[t, h, dim]):.6g}, want "
                    f"{float(y64[t, h, dim]):.6g}")


@pytest.mark.parametrize("kpt", [False, True], ids=["kv-per-tensor", "k-per-token"])
@pytest.mark.parametrize("layout", ["nhd", "hnd"])
@pytest.mark.parametrize("heads", [(8, 2), (4, 1)], ids=lambda h: f"{h[0]}-{h[1]}")
def test_prefill_fp8_exact_scores(hpc, heads, layout, kpt):
    """The dense entry point and block-sparse masks at skip 0 and 0.5 on ragged requests."""
    hq, hkv = heads
    seed = 100 * hq + 2 * (layout == "hnd") + kpt
    d = xs.make_prefill_inputs(Q_LENS, KV_LENS, hq, hkv, None, kpt, seed=seed, layout=layout,
                               device="cuda")
    y64 = _reference(d, kpt)
    _check(_run(hpc, d, kpt, dense_entry=True), y64, d, "dense entry point")
    _check(_run(hpc, d, kpt), y64, d, "block-sparse entry point without a mask")
    for skip in (0.0, 0.5):
        m = xs.make_prefill_inputs(Q_LENS, KV_LENS, hq, hkv, skip, kpt, seed=seed, layout=layout,
                                   device="cuda")
        _check(_run(hpc, m, kpt), _reference(m, kpt), m, f"mask skip {skip}")


@pytest.mark.parametrize("kpt", [False, True], ids=["kv-per-tensor", "k-per-token"])
def test_prefill_fp8_exact_scores_short_mask_and_empty_tiles(hpc, kpt):
    """A mask narrower than the causal extent (exactly one tile past its width is visited), and Q
    tiles whose mask rows are empty: those rows must be NaN, all others exact."""
    d = xs.make_prefill_inputs([1024, 300], [1024, 2000], 4, 1, 0.3, kpt, seed=5, device="cuda")
    d["block_mask"] = d["block_mask"][:, :, :, :5].contiguous()
    _check(_run(hpc, d, kpt), _reference(d, kpt), d, "mask width 5 of 8 / 16 tiles")
    d = xs.make_prefill_inputs([1024, 300], [1024, 2000], 4, 1, 0.5, kpt, seed=6, device="cuda")
    d["block_mask"][0, 1, 2] = False  # request 0, head 1, Q tile 2: no active KV tile
    d["block_mask"][1, 3, 0] = False
    y64 = _reference(d, kpt)
    assert torch.isnan(y64[256:384, 1]).all() and torch.isnan(y64[1024:1152, 3]).all()
    _check(_run(hpc, d, kpt), y64, d, "empty mask rows")


def _roll_heads_in_group(t, group):
    s = t.shape
    return torch.roll(t.float().reshape(s[0], s[1] // group, group, *s[2:]), 1, dims=2).to(t.dtype).reshape(s)


@pytest.mark.parametrize("kpt", [False, True], ids=["kv-per-tensor", "k-per-token"])
def test_prefill_fp8_exact_scores_negative_control(hpc, kpt):
    """Real kernel output with the q heads rolled within each GQA group, and with the q scale of the
    neighbouring token, must fail the comparison with the unmutated reference."""
    d = xs.make_prefill_inputs(Q_LENS, KV_LENS, 8, 2, 0.5, kpt, seed=9, device="cuda")
    y64 = _reference(d, kpt)
    assert not bool(ox.violations(_run(hpc, d, kpt).float().cpu(), y64).any())
    for name, mut in (("q heads rolled", dict(q=_roll_heads_in_group(d["q"], 4))),
                      ("q scale of the wrong token", dict(qscale=torch.roll(d["qscale"], 1, dims=2)))):
        y = _run(hpc, dict(d, **mut), kpt).float().cpu()
        assert int(ox.violations(y, y64).sum()) > 0, f"{name}: the comparison did not notice"


@pytest.mark.skipif(os.environ.get("HPC_B200_PREFILL_POLY") is not None,
                    reason="already running under a fixed exponential mix")
@pytest.mark.parametrize("poly", ["0", "4"])
def test_prefill_fp8_exact_scores_exp2_mix(hpc, poly):
    """The share of exponentials taken by the polynomial exp2 is read once per process, so this
    file runs again in a child process with none (0) and half (4) of them on the polynomial. At
    integer inputs the polynomial gives 2^n * 0.99993, which rounds to the exact e4m3 code, so the
    tolerance holds unchanged."""
    here = Path(__file__).resolve()
    env = dict(os.environ, HPC_B200_PREFILL_POLY=poly)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [
        "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider", str(here), "-k", "not exp2_mix"]
    r = subprocess.run(cmd, cwd=str(here.parents[1]), env=env, capture_output=True, text=True,
                       timeout=1200)
    assert r.returncode == 0, f"HPC_B200_PREFILL_POLY={poly}:\n{r.stdout[-4000:]}\n{r.stderr[-2000:]}"
    assert " passed" in r.stdout and "skipped" not in r.stdout.splitlines()[-1], r.stdout[-2000:]
