"""FP8 paged decode (both quant types) against a float64 softmax, on inputs whose log2 scores are
exact integers (synth/exact_scores.py): every quantisation step of the kernel is then exact and its
output must equal the float64 result up to one bf16 rounding (oracle.exact.violations). Unlike the
reference-distribution tests, these see the Q operand, the q / k scales and their indexing, the GQA
head mapping, the causal tail and every tile of the rotated bin walk (csrc/decode_common.cuh),
whose coverage is asserted from the task maps themselves."""
import pytest
import torch

from oracle import decode_walk as dw
from oracle import exact as ox
from synth import exact_scores as xs

pytestmark = pytest.mark.gpu

HEADS = [(1, 8), (2, 8), (4, 32), (8, 32)]  # group 8 at Sq 4 / 3 is rows 32 / 24: NQ = 32
RAGGED = [1, 63, 64, 65, 127, 128, 129, 255, 256, 257, 1000, 2500, 40000]
MODES = [("device schedule", None), ("device-assigned", 64), ("device-assigned", 1024),
         ("cpu-assigned", 64), ("cpu-assigned", 1024)]


def _qt(hpc, kpt):
    return (hpc.QuantType.QPERTOKEN_PERHEAD_KPERTOKEN_PERHEAD_VPERHEAD if kpt
            else hpc.QuantType.QPERTOKEN_PERHEAD_KPERTENSOR_VPERTENSOR)


def _lens(sq):
    # every boundary length, a tail of exactly Sq tokens (the whole cache is the causal window)
    return [max(L, sq) for L in RAGGED] + [sq]


def _task_map(hpc, d, hkv, sq, mode, mpl):
    if mpl is None:
        return None
    lens = d["kv_lens_total"]
    tm = hpc.get_attention_decode_task_workspace(lens.numel(), int(lens.max()), hkv, mpl)
    hpc.assign_attention_decode_task(lens.cpu() if mode == "cpu-assigned" else lens, tm, hkv, sq,
                                     True, mpl)
    return tm


def _run(hpc, d, hkv, sq, kpt, tm):
    return hpc.attention_decode_fp8(d["q"], d["kcache"], d["vcache"], d["block_ids"],
                                    d["kv_lens_total"], d["q_scale"], d["k_scale"], d["v_scale"],
                                    mtp=sq - 1, new_kv_included=True, quant_type=_qt(hpc, kpt),
                                    task_map=tm)


def _reference(d, sq, kpt):
    c = {k: v.cpu() for k, v in d.items()}
    return ox.decode(c["q"], c["kcache"], c["vcache"], c["block_ids"], c["kv_lens_total"],
                     c["q_scale"], c["k_scale"], c["v_scale"], sq, k_per_token=kpt)


def _rotates(hkv, hq, sq, layout):
    """The launcher's condition for the rotated walk on these (256-byte aligned) caches."""
    return layout == "NHD" and hkv % 2 == 0 and (hq // hkv) * sq <= 16


def _report(y, y64, sq, hkv, tm, rotate, tag):
    """'' if y is within tolerance, else the coordinates of the first bad element and the tasks
    that cover its (batch, kv head)."""
    bad = ox.violations(y, y64)
    if not bool(bad.any()):
        return ""
    n = int(bad.sum())
    row, h, dim = (int(i) for i in bad.nonzero()[0])
    b, s = divmod(row, sq)
    g = y.shape[1] // hkv
    msg = (f"{tag}: {n} elements outside one bf16 rounding (rel L2 {ox.rel_l2(y, y64):.4f}); first "
           f"at batch {b}, query row {s}, q head {h}, dim {dim}: got {float(y[row, h, dim]):.6g}, "
           f"want {float(y64[row, h, dim]):.6g}")
    if tm is not None:
        m = tm.view(torch.int32).cpu().numpy()
        msg += f"; tasks of (batch {b}, kv head {h // g}): " + dw.tasks_of(m, b, h // g, rotate)
    return msg


@pytest.mark.parametrize("kpt", [False, True], ids=["kv-per-tensor", "k-per-token"])
@pytest.mark.parametrize("layout", ["NHD", "HND"])
@pytest.mark.parametrize("sq", [1, 2, 3, 4])
@pytest.mark.parametrize("heads", HEADS, ids=lambda h: f"{h[0]}-{h[1]}")
def test_decode_fp8_exact_scores(hpc, monkeypatch, heads, sq, layout, kpt):
    """Ragged and boundary lengths incl. one 40000-token request, every task-map mode, min_process_len
    64 (many chunks through the combine) and 1024 (tasks that are their request's only chunk write
    the output directly), the bin walk rotated and front to back."""
    hkv, hq = heads
    lens = _lens(sq)
    d = xs.make_decode_inputs(len(lens), sq, lens, hkv, hq, k_per_token=kpt, layout=layout,
                              seed=1000 * hkv + 10 * sq + kpt, device="cuda")
    y64 = _reference(d, sq, kpt)
    errors = []
    for rot in ("0", "1"):
        monkeypatch.setenv("HPC_B200_DECODE_ROTATE", rot)
        rotated = rot == "1" and _rotates(hkv, hq, sq, layout)
        for mode, mpl in MODES:
            tm = _task_map(hpc, d, hkv, sq, mode, mpl)
            y = _run(hpc, d, hkv, sq, kpt, tm).float().cpu()
            e = _report(y, y64, sq, hkv, tm, rotated,
                        f"mode {mode}, mpl {mpl}, HPC_B200_DECODE_ROTATE={rot} (walk rotated: {rotated})")
            if e:
                errors.append(e)
    assert not errors, "\n".join(errors)


def test_decode_fp8_exact_scores_c2_full(hpc, monkeypatch):
    """BASELINE config C2 (64 requests x 8192 tokens, GQA 32/8, NHD, min_process_len 64): all 64
    requests against the float64 reference, rotated and front to back."""
    B, hkv, hq, S = 64, 8, 32, 8192
    d = xs.make_decode_inputs(B, 1, [S] * B, hkv, hq, seed=64, device="cuda")
    y64 = _reference(d, 1, False)
    errors = []
    for rot in ("1", "0"):
        monkeypatch.setenv("HPC_B200_DECODE_ROTATE", rot)
        tm = _task_map(hpc, d, hkv, 1, "device-assigned", 64)
        if rot == "1":  # this is the shape the rotation was built for: it must split tasks here
            assert sum(w.split for w in dw.walks(tm.view(torch.int32).cpu().numpy())) > 100
        y = _run(hpc, d, hkv, 1, False, tm).float().cpu()
        e = _report(y, y64, 1, hkv, tm, rot == "1", f"C2, HPC_B200_DECODE_ROTATE={rot}")
        if e:
            errors.append(e)
    assert not errors, "\n".join(errors)


def test_decode_rotated_walk_coverage(hpc):
    """The rotated cases of test_decode_fp8_exact_scores contain each situation the rotated walk
    handles: a walk that starts inside a task (state saved, restored at the end of the walk), a bin
    across a kv-head boundary, a short last bin walked front to back, and a split task that holds
    the causal tail (Sq > 1). Read from the device workspaces, with the CPU-assigned maps equal."""
    found = dict(split=0, straddle=0, short=0, causal_split=0)
    for hkv, hq in HEADS:
        for sq in (1, 2, 3, 4):
            if not _rotates(hkv, hq, sq, "NHD"):
                continue
            lens = torch.tensor(_lens(sq), dtype=torch.int32, device="cuda")
            d = dict(kv_lens_total=lens)
            for mpl in (64, 1024):
                m = _task_map(hpc, d, hkv, sq, "device-assigned", mpl).view(torch.int32).cpu().numpy()
                mc = _task_map(hpc, d, hkv, sq, "cpu-assigned", mpl).view(torch.int32).cpu().numpy()
                n = (1 + int(m[0]) * int(m[1])) * dw.TASK_INTS
                assert (m[:2] == mc[:2]).all() and m[6] == mc[6] and (m[12:n] == mc[12:n]).all()
                for w in dw.walks(m):
                    seen = sorted((r, t) for r, tb, te in w.segments() for t in range(tb, te))
                    assert seen == [(r, t) for r in range(len(w.rows)) for t in range(int(w.rows[r, 6]))]
                    found["split"] += w.split
                    found["straddle"] += w.straddles_heads
                    found["short"] += w.short
                    found["causal_split"] += w.split and sq > 1 and bool(w.rows[w.ks, 8])
    assert all(v > 0 for v in found.values()), found


def _roll_heads_in_group(t, group):
    s = t.shape
    return torch.roll(t.float().reshape(s[0], s[1] // group, group, *s[2:]), 1, dims=2).to(t.dtype).reshape(s)


def _roll_tokens_in_request(t, sq):
    s = t.shape
    return torch.roll(t.float().reshape(-1, sq, *s[1:]), 1, dims=1).to(t.dtype).reshape(s)


@pytest.mark.parametrize("kpt", [False, True], ids=["kv-per-tensor", "k-per-token"])
def test_decode_fp8_exact_scores_negative_control(hpc, monkeypatch, kpt):
    """Real kernel output with the q heads rolled within each GQA group, and with the q scale of the
    neighbouring token, must fail the comparison with the unmutated reference."""
    hkv, hq, sq = 2, 8, 2
    lens = _lens(sq)
    monkeypatch.setenv("HPC_B200_DECODE_ROTATE", "1")
    d = xs.make_decode_inputs(len(lens), sq, lens, hkv, hq, k_per_token=kpt, seed=7, device="cuda")
    y64 = _reference(d, sq, kpt)
    tm = _task_map(hpc, d, hkv, sq, "device-assigned", 64)
    assert not _report(_run(hpc, d, hkv, sq, kpt, tm).float().cpu(), y64, sq, hkv, tm, True, "clean")
    for name, mut in (("q heads rolled", dict(q=_roll_heads_in_group(d["q"], hq // hkv))),
                      ("q scale of the wrong token", dict(q_scale=_roll_tokens_in_request(d["q_scale"], sq)))):
        y = _run(hpc, dict(d, **mut), hkv, sq, kpt, tm).float().cpu()
        assert int(ox.violations(y, y64).sum()) > 0, f"{name}: the comparison did not notice"
