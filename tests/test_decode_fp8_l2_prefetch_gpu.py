"""Page-wide L2 prefetch of the FP8 decode kernel (csrc/decode_attn_fp8.cu, producer warp): it only
moves bytes into L2 ahead of the loads, so every output must be bit-identical to the same call with
HPC_B200_KV_PREFETCH=0, at every prefetch distance, and on caches whose layout turns it off."""
import pytest
import torch

from synth.decode import make_decode_fp8_inputs, make_decode_fp8_kpt_inputs

pytestmark = pytest.mark.gpu

DISTANCES = [None, "0", "2", "37"]  # None: the shipped default; 37 reaches past a 16-tile id group


def _qt(hpc, kpt):
    return (hpc.QuantType.QPERTOKEN_PERHEAD_KPERTOKEN_PERHEAD_VPERHEAD if kpt
            else hpc.QuantType.QPERTOKEN_PERHEAD_KPERTENSOR_VPERTENSOR)


def _inputs(B, sq, lens, hkv, hq, kpt, layout="NHD", seed=5):
    if kpt:
        return make_decode_fp8_kpt_inputs(B, sq, lens, hkv, hq, seed=seed, layout=layout, device="cuda")
    d = make_decode_fp8_inputs(B, sq, lens, hkv, hq, seed=seed, layout=layout, device="cuda")
    return dict(d, kcache=d["kvcache"][:, 0], vcache=d["kvcache"][:, 1])


def _run(hpc, d, hkv, sq, kpt, mpl):
    tm = None
    if mpl is not None:
        lens = d["kv_lens_total"]
        tm = hpc.get_attention_decode_task_workspace(lens.numel(), int(lens.max()), hkv, mpl)
        hpc.assign_attention_decode_task(lens, tm, hkv, sq, True, mpl)
    y = hpc.attention_decode_fp8(d["q"], d["kcache"], d["vcache"], d["block_ids"],
                                 d["kv_lens_total"], d["q_scale"], d["k_scale"], d["v_scale"],
                                 mtp=sq - 1, new_kv_included=True, quant_type=_qt(hpc, kpt),
                                 task_map=tm)
    torch.cuda.synchronize()
    return y


def _check_on_off(hpc, monkeypatch, d, hkv, sq, kpt, mpl):
    monkeypatch.setenv("HPC_B200_KV_PREFETCH", "0")
    ref = _run(hpc, d, hkv, sq, kpt, mpl)
    assert bool(torch.isfinite(ref.float()).all())
    monkeypatch.setenv("HPC_B200_KV_PREFETCH", "1")
    for dist in DISTANCES:
        if dist is None:
            monkeypatch.delenv("HPC_B200_KV_PREFETCH_DIST", raising=False)
        else:
            monkeypatch.setenv("HPC_B200_KV_PREFETCH_DIST", dist)
        assert torch.equal(_run(hpc, d, hkv, sq, kpt, mpl), ref), f"prefetch distance {dist}"
    return ref


@pytest.mark.parametrize("kpt", [False, True], ids=["kv-per-tensor", "k-per-token"])
def test_prefetch_c2(hpc, monkeypatch, kpt):
    """BASELINE config C2: 64 requests x 8192 tokens, GQA 32/8, token-major cache."""
    B, hkv, hq, S = 64, 8, 32, 8192
    _check_on_off(hpc, monkeypatch, _inputs(B, 1, [S] * B, hkv, hq, kpt), hkv, 1, kpt, 64)


@pytest.mark.parametrize("mpl", [None, 64, 1024])
@pytest.mark.parametrize("sq", [1, 2])
@pytest.mark.parametrize("kpt", [False, True], ids=["kv-per-tensor", "k-per-token"])
def test_prefetch_ragged(hpc, monkeypatch, kpt, sq, mpl):
    """Ragged lengths, one request shorter than a tile and one shorter than a page, Sq 1 and 2."""
    hkv, hq = 8, 32
    lens = [max(L, sq) for L in (1, 100, 129, 200, 1000, 2500, 4097, 8192, 12000, 333)]
    d = _inputs(len(lens), sq, lens, hkv, hq, kpt, seed=11 + sq)
    _check_on_off(hpc, monkeypatch, d, hkv, sq, kpt, mpl)


@pytest.mark.parametrize("kpt", [False, True], ids=["kv-per-tensor", "k-per-token"])
def test_prefetch_hnd(hpc, monkeypatch, kpt):
    """Head-major cache: the prefetch is off, the knob changes nothing."""
    hkv, hq = 8, 32
    lens = [3000, 64, 8192, 777]
    _check_on_off(hpc, monkeypatch, _inputs(len(lens), 1, lens, hkv, hq, kpt, layout="HND"),
                  hkv, 1, kpt, 64)


def test_prefetch_strided_cache(hpc, monkeypatch):
    """Token rows padded to 10 heads: the walk still rotates but a page is not one contiguous range,
    so the prefetch is off. The output equals that of the dense cache holding the same values."""
    hkv, hq = 8, 32
    lens = [5000, 130, 8192, 2048]
    d = _inputs(len(lens), 1, lens, hkv, hq, False, seed=3)
    kv = d["kvcache"]
    padded = torch.zeros(kv.shape[:3] + (hkv + 2, 128), dtype=kv.dtype, device=kv.device)
    padded[:, :, :, :hkv] = kv
    padded = padded[:, :, :, :hkv]
    assert padded.stride(2) == (hkv + 2) * 128
    dense = _check_on_off(hpc, monkeypatch, d, hkv, 1, False, 64)
    ds = dict(d, kvcache=padded, kcache=padded[:, 0], vcache=padded[:, 1])
    assert torch.equal(_check_on_off(hpc, monkeypatch, ds, hkv, 1, False, 64), dense)
