"""A/B of the page-wide L2 prefetch of the fp8 decode kernel (csrc/decode_attn_fp8.cu) at the C2 shape
(bs 64, GQA 32/8, d 128, token-major cache, 64-token pages), plus the SM-side floor of the kernel.
HPC_B200_KV_PREFETCH, HPC_B200_KV_PREFETCH_DIST and HPC_B200_KV_PROMO are read at every launch, so
one process times all variants, alternating them, on the same box. GPU box only.

    python tools/decode_prefetch_ab.py [--reps 3] [--out profiles/decode_prefetch_ab.json]

Cases:
  equal    C2, every request 8192 tokens (the bench.py workload and seed)
  ragged   64 requests of 1024..8192 tokens
  floor    C2 with every request's page table pointing at the same 128 pages: 16 MB of K+V that
           stays in L2, so the kernel time is what the SM side (TMA issue, MMA, softmax) needs
For each variant: the attention kernel alone (CUDA events over `iters` launches) and the whole call
(attention + combine), and whether its output is bit-identical to the prefetch-off output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
from pathlib import Path

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "hpc-ops_b200"))
sys.path.insert(0, str(REPO / "tools"))
import torch  # noqa: E402

import hpc  # noqa: E402
from hpc import _ffi  # noqa: E402
from hpc import attention as hatt  # noqa: E402
from bench_extras import time_eager  # noqa: E402
from synth.decode import make_decode_fp8_inputs  # noqa: E402

KNOBS = ("HPC_B200_KV_PREFETCH", "HPC_B200_KV_PREFETCH_DIST", "HPC_B200_KV_PROMO")
DISTANCES = (0, 1, 2, 4)


def variants():
    v = []
    for promo_name, promo in (("promo256", "3"), ("promo128", "2"), ("promo64", "1")):
        v.append((f"off_{promo_name}", {"HPC_B200_KV_PREFETCH": "0", "HPC_B200_KV_PROMO": promo}))
        for dist in DISTANCES:
            v.append((f"d{dist}_{promo_name}", {"HPC_B200_KV_PREFETCH": "1",
                                                "HPC_B200_KV_PREFETCH_DIST": str(dist),
                                                "HPC_B200_KV_PROMO": promo}))
    return v


def set_env(env):
    for k in KNOBS:
        if env.get(k) is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = env[k]


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"query": q, "value": r.stdout.strip().splitlines()[0] if r.returncode == 0 else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--out", type=Path, default=None)
    a = ap.parse_args()

    dev = torch.device("cuda")
    B, S, hkv, hq, mpl = 64, 8192, 8, 32, 64
    d = make_decode_fp8_inputs(B, 1, [S] * B, hkv, hq, seed=41, device=dev)
    kc, vc = d["kvcache"][:, 0], d["kvcache"][:, 1]
    g = torch.Generator().manual_seed(7)
    cases = {
        "equal": (d["kv_lens_total"], d["block_ids"]),
        "ragged": (torch.randint(1024, S + 1, (B,), generator=g, dtype=torch.int32).to(dev),
                   d["block_ids"]),
        "floor": (d["kv_lens_total"], d["block_ids"][:1].expand(B, -1).contiguous()),
    }
    out = {"gpu": gpu_info(), "iters": a.iters, "reps": a.reps, "cases": {}}
    for cname, (lens, ids) in cases.items():
        tm = hpc.get_attention_decode_task_workspace(B, S, hkv, mpl)
        hpc.assign_attention_decode_task(lens, tm, hkv, 1, True, mpl)
        y = torch.empty(B, hq, 128, device=dev, dtype=torch.bfloat16)

        def call():
            hpc.attention_decode_fp8(d["q"], kc, vc, ids, lens, d["q_scale"], d["k_scale"],
                                     d["v_scale"], mtp=0, new_kv_included=True, task_map=tm,
                                     output=y)

        _, args, keep = hatt._decode_fp8_prepare(d["q"], kc, vc, ids, lens, d["q_scale"],
                                                 d["k_scale"], d["v_scale"], 0, True, 1, True, tm,
                                                 None, y)

        def kernel():
            _ffi.lib.hpc_attention_decode_fp8_partial_async(*args)

        byts = 2 * int(lens.sum()) * hkv * 128
        ref = None
        rows = {}
        for _ in range(a.reps):
            for name, env in variants():
                set_env(env)
                ms_call = time_eager(call, a.iters)
                same = None
                if ref is None:
                    ref = y.clone()
                else:
                    same = bool(torch.equal(ref, y))
                ms_kern = time_eager(kernel, a.iters)
                r = rows.setdefault(name, {"kernel_ms": [], "call_ms": [], "bit_equal_to_off": []})
                r["kernel_ms"].append(round(ms_kern, 5))
                r["call_ms"].append(round(ms_call, 5))
                if same is not None:
                    r["bit_equal_to_off"].append(same)
        for name, r in rows.items():
            km = statistics.median(r["kernel_ms"])
            r["kernel_ms_median"] = km
            r["call_ms_median"] = statistics.median(r["call_ms"])
            r["kernel_gbs_median"] = round(byts / km / 1e6, 1)
        out["cases"][cname] = {"algorithmic_kv_bytes": byts, "variants": rows}
        del keep
    set_env({})
    # tiles per CTA (bin) of the equal / floor cases: the floor's time per tile on the SM side
    tiles = B * (S // 128) * hkv
    ctas = hatt._num_total_ctas(dev)
    out["tiles_per_cta"] = -(-tiles // ctas)
    fl = out["cases"]["floor"]["variants"]["off_promo256"]["kernel_ms_median"]
    out["floor_us_per_tile"] = round(fl * 1e3 / out["tiles_per_cta"], 4)
    line = json.dumps(out)
    print(line)
    if a.out is not None:
        a.out.parent.mkdir(parents=True, exist_ok=True)
        a.out.write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
