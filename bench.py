#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 build (contract: see the task statement / DESIGN.md §4).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (N=1): BASELINE.json configs[1] — FP8 paged decode attention, q per-token/head scales,
k/v per-tensor scales, bs=64, GQA 32/8, d=128, seq=8192, page 64, synthetic data.
A step = one decode-attention pass over that batch: task-map assign + split-k attention + combine.

  value      tokens/s with every input already resident in HBM (CUDA events, one region of K steps).
  e2e        the same through the public API with HOST inputs: per step the pinned host q, q scales,
             kv lengths and page table are copied H2D, the task map is assigned, attention runs, and
             the bf16 output is read back D2H (the paged KV cache is device-resident state, exactly
             as in the reference API where it is a CUDA tensor owned by the serving engine).
  roofline   the attention kernel alone: algorithmic bytes / its CUDA-event duration vs measured HBM.
  cpu_baseline  the torch CPU oracle on a bounded sample of the same workload.

  extra      the other BASELINE configs, each with its own roofline fraction and a sampled parity
             check against the CPU oracle (tools/bench_extras.py): FusedMoE C3, block-sparse prefill
             C4 (both quant schemes), the route GEMM, and the fused AllReduce+RMSNorm C5.

N>1: decode does not shard (SURVEY.md §8e "replicas only"): every rank runs the same decode workload
on its own GPU, no data-path collective; value = N * tokens / max-over-ranks time ("weak"). The ONE
sharded path, fuse_allreduce_rmsnorm, runs at W=N inside `extra.allreduce_c5` (high-throughput and
low-latency kernels over the NCCL-initialised symmetric buffers, CUDA-graph timed, max over ranks).
`--impl reference`: times the reference's own algorithm on the host cores (the torch CPU reference
path restated in oracle/, since the reference's sm_90a build cannot execute on sm_100).
`--dump-outputs DIR`: after the timed steps, rank 0 writes the bf16 attention output of the last
step as DIR/attention_decode_fp8_output.npy (float32, [64, 32, 128]). The inputs are seeded, so
two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "hpc-ops_b200"))

import torch  # noqa: E402

WORKLOAD = dict(num_batch=64, num_seq_q=1, num_head_kv=8, num_head_q=32, head_dim=128, seq=8192,
                block_size=64)
WORKLOAD_NAME = "fp8_decode_attn bs=64 GQA32/8 d=128 seq=8192 page=64 (BASELINE configs[1])"
LAUNCHES_PER_STEP = 3   # assign_task_kernel, decode_attn_fp8_kernel, decode_combine_kernel
EXTRA_BUDGET_S = 420    # the `extra` block must not delay the line beyond this
METRIC = "fp8_decode_attn_tokens_per_s"
UNIT = "tok/s"


MPL = 64  # reference benchmark default (benchmark/attention_decode/bench_attention_decode_fp8.py:710)


def config_dict(world):
    """`config` of the JSON line: identical in both arms."""
    return {"workload": WORKLOAD_NAME, "parallelism": f"replicas x{world}",
            "step": "task-map assign + split-k attention + combine", "min_process_len": MPL,
            "l2": "inputs (1.07 GB KV per step) exceed the 126 MB L2; no flush needed"}


def algorithmic_bytes(w):
    """SURVEY.md §8(d): K+V stream + Q + bf16 out + q scales, per call."""
    B, Hkv, Hq, D, S = w["num_batch"], w["num_head_kv"], w["num_head_q"], w["head_dim"], w["seq"]
    return B * Hkv * S * (D + D) + B * Hq * D * (1 + 2) + B * Hq * 4


def measured_peaks():
    f = REPO / "MEASURED_PEAKS.json"
    if f.exists():
        try:
            return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "power_w_max": max(pw) if pw else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_oracle_sample(w, d, nreq, gpu_out=None):
    """cpu_baseline leg (the one place the measured arm touches oracle/): time the torch CPU
    reference path on the first `nreq` requests of the batch the GPU just processed and, since the
    result is there anyway, check the GPU output of those requests against it."""
    from oracle import attention as oa

    sub = {k: (v[:nreq * w["num_seq_q"]] if k in ("q", "q_scale") else v[:nreq] if k in
               ("block_ids", "kv_lens_total") else v).cpu() for k, v in d.items()}
    args = (sub["q"], sub["kvcache"][:, 0], sub["kvcache"][:, 1], sub["block_ids"],
            sub["kv_lens_total"], sub["q_scale"], sub["k_scale"], sub["v_scale"], w["num_seq_q"])
    oa.decode_fp8_kvpertensor(*args)  # warm-up (thread pool, page faults)
    times = []
    for _ in range(3):
        t0 = time.perf_counter()
        gt = oa.decode_fp8_kvpertensor(*args)
        times.append(time.perf_counter() - t0)
    dt = sorted(times)[1]  # median of 3 (SURVEY.md 8d)
    err = None
    if gpu_out is not None:
        err = (gpu_out[:nreq * w["num_seq_q"]].float().cpu() - gt.float()).abs().max().item()
        # tolerance of reference tests/test_attention_decode_qpertoken_perhead_kvpertensor_fp8.py
        assert err < 0.2, f"bench parity check failed: max abs err {err}"
    return nreq * w["num_seq_q"] / dt, dt, err


def run_reference(a, rank, world):
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    w = WORKLOAD
    nreq = 8  # bounded sample per step: 8 of the 64 requests (each request is independent)
    from oracle import attention as oa
    from synth.decode import make_decode_fp8_inputs

    d = make_decode_fp8_inputs(nreq, 1, [w["seq"]] * nreq, w["num_head_kv"], w["num_head_q"],
                               seed=41, device="cpu")
    args = (d["q"], d["kvcache"][:, 0], d["kvcache"][:, 1], d["block_ids"], d["kv_lens_total"],
            d["q_scale"], d["k_scale"], d["v_scale"], 1)
    for _ in range(a.warmup):
        oa.decode_fp8_kvpertensor(*args)
    t0 = time.perf_counter()
    for _ in range(a.steps):
        oa.decode_fp8_kvpertensor(*args)
    dt = time.perf_counter() - t0
    val = nreq * a.steps / dt
    sample = f"{nreq} of 64 requests per step (requests are independent), torch CPU oracle"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3,
        "ms_per_full_batch_extrapolated": dt / a.steps * 1e3 * (64 / nreq),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp8_e4m3 (fp32 accumulate)", "data": "synthetic", "config": config_dict(world),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(),
                         "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-extra", action="store_true", help="skip the `extra` block (C3/C4/C5/route GEMM)")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path, default=None,
                    help="write the attention output of the last timed step to DIR as .npy")
    a = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if a.impl == "reference":
        if a.dump_outputs is not None:
            ap.error("--dump-outputs applies to --impl b200")
        a.steps = a.steps or 3
        a.warmup = 1 if a.warmup is None else a.warmup
        run_reference(a, rank, world)
        return
    a.steps = a.steps or 2000
    a.warmup = 20 if a.warmup is None else max(a.warmup, 3)

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    import hpc
    from hpc import attention as hatt
    from hpc import _ffi
    from synth.decode import make_decode_fp8_inputs

    w = WORKLOAD
    B, Sq, Hkv, Hq, S = w["num_batch"], w["num_seq_q"], w["num_head_kv"], w["num_head_q"], w["seq"]
    d = make_decode_fp8_inputs(B, Sq, [S] * B, Hkv, Hq, seed=41 + rank, device=dev)
    kc, vc = d["kvcache"][:, 0], d["kvcache"][:, 1]
    task_map = hpc.get_attention_decode_task_workspace(B, S, Hkv, MPL)
    hpc.assign_attention_decode_task(d["kv_lens_total"], task_map, Hkv, Sq, True, MPL)
    out = torch.empty((B * Sq, Hq, 128), dtype=torch.bfloat16, device=dev)

    def step_resident():
        hpc.assign_attention_decode_task(d["kv_lens_total"], task_map, Hkv, Sq, True, MPL)
        hpc.attention_decode_fp8(d["q"], kc, vc, d["block_ids"], d["kv_lens_total"], d["q_scale"],
                                 d["k_scale"], d["v_scale"], mtp=Sq - 1, new_kv_included=True,
                                 task_map=task_map, output=out)

    step_resident()  # first call (lazy one-time setup) outside every timed region
    torch.cuda.synchronize()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # ---------------- value: inputs resident in HBM ----------------
    # One timed region of exactly K steps between barrier + synchronize.
    for _ in range(a.warmup):
        step_resident()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        step_resident()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / a.steps
    value = world * B * Sq / (ms_per_step * 1e-3)
    if a.dump_outputs is not None and rank == 0:
        import numpy as np

        a.dump_outputs.mkdir(parents=True, exist_ok=True)
        np.save(a.dump_outputs / "attention_decode_fp8_output.npy", out.float().cpu().numpy())

    # ---------------- roofline: the attention kernel alone ----------------
    y, args, keep = hatt._decode_fp8_prepare(
        d["q"], kc, vc, d["block_ids"], d["kv_lens_total"], d["q_scale"], d["k_scale"],
        d["v_scale"], Sq - 1, True, 1, True, task_map, None, out)
    nk = max(50, min(a.steps, 500))
    for _ in range(5):
        _ffi.check(_ffi.lib.hpc_attention_decode_fp8_partial_async(*args))
    torch.cuda.synchronize()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0.record()
    for _ in range(nk):
        _ffi.lib.hpc_attention_decode_fp8_partial_async(*args)
    k1.record()
    torch.cuda.synchronize()
    kern_ms = k0.elapsed_time(k1) / nk
    alg = algorithmic_bytes(w)
    peak, peak_src = measured_peaks()
    achieved = alg / (kern_ms * 1e-3) / 1e9
    traffic = None
    tf = REPO / "profiles" / "decode_attn_traffic.json"
    if tf.exists():
        try:
            traffic = json.loads(tf.read_text()).get("dram_bytes_per_launch")
        except Exception:
            traffic = None

    # ---------------- e2e: host inputs through the public API ----------------
    # The step's host inputs live in ONE pinned staging buffer (256-B aligned segments), as a
    # serving engine would stage them: one H2D copy per step, device tensors are views of it.
    names = ("q", "q_scale", "kv_lens_total", "block_ids")
    segs, total = {}, 0
    for k in names:
        nb = d[k].numel() * d[k].element_size()
        segs[k] = (total, nb)
        total += (nb + 255) // 256 * 256
    host_buf = torch.empty(total, dtype=torch.uint8).pin_memory()
    dev_buf = torch.empty(total, dtype=torch.uint8, device=dev)
    for k in names:
        off, nb = segs[k]
        host_buf[off:off + nb].copy_(d[k].cpu().contiguous().view(-1).view(torch.uint8))

    def dev_view(k):
        off, nb = segs[k]
        return dev_buf[off:off + nb].view(d[k].dtype).view(d[k].shape)

    dq, dqs, dl, dbi = (dev_view(k) for k in names)
    host_out = torch.empty(out.shape, dtype=out.dtype).pin_memory()
    h2d = sum(nb for _, nb in segs.values())
    d2h = host_out.numel() * host_out.element_size()

    def step_e2e():
        dev_buf.copy_(host_buf, non_blocking=True)
        hpc.assign_attention_decode_task(dl, task_map, Hkv, Sq, True, MPL)
        y2 = hpc.attention_decode_fp8(dq, kc, vc, dbi, dl, dqs, d["k_scale"], d["v_scale"],
                                      mtp=Sq - 1, new_kv_included=True, task_map=task_map,
                                      output=out)
        host_out.copy_(y2, non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the engine consumes the result on the host

    # e2e parity: the staged inputs must reproduce the resident result bit for bit
    step_e2e()
    ref_out = out.clone()
    step_resident()
    torch.cuda.synchronize()
    assert torch.equal(ref_out, out), "e2e path differs from the resident path"

    e2e_steps = max(20, min(a.steps, 300))
    for _ in range(3):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(e2e_steps):
        step_e2e()
    g1.record()
    barrier()
    wall = (time.perf_counter() - t0) * 1e3
    ems = max(g0.elapsed_time(g1), 0.0)
    te = torch.tensor([max(ems, wall)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms = float(te.item()) / e2e_steps
    e2e_val = world * B * Sq / (e2e_ms * 1e-3)

    clocks = sampler.stop() if rank == 0 else None

    line = None
    if rank == 0:
        # CPU baseline on a bounded sample (torch oracle == the reference's CPU-runnable path)
        torch.set_num_threads(os.cpu_count() or 1)
        nreq = 16
        step_resident()
        torch.cuda.synchronize()
        cpu_val, cpu_dt, cpu_err = cpu_oracle_sample(w, d, nreq, out)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp8_e4m3 (fp32 accumulate)",
            "data": "synthetic", "config": config_dict(world),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": "profiles/decode_attn_traffic.json (one ncu --set full capture)",
                         "kernel": "decode_attn_fp8_kernel<16,4>", "kernel_ms": kern_ms,
                         "algorithmic_bytes": alg, "peak_source": peak_src},
            "cpu_baseline": {"value": cpu_val, "unit": UNIT, "cores": torch.get_num_threads(),
                             "kind": "port",
                             "sample": f"{nreq} of 64 requests, median of 3 passes after a warm-up, "
                                       f"{cpu_dt:.2f} s per pass",
                             "gpu_vs_cpu_max_abs_err": cpu_err},
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "steps": e2e_steps,
                    "note": "paged KV cache is device-resident engine state; per-step host inputs "
                            "(q, q scales, kv lengths, page table) staged in one pinned buffer, "
                            "one H2D copy; bf16 output read back"},
            "gpu_launches": LAUNCHES_PER_STEP * a.steps,
            "clocks": clocks,
        }

    # The headline numbers are final here. A watchdog prints the line if anything below hangs.
    printed = threading.Event()

    def emit():
        if not printed.is_set():
            printed.set()
            if rank == 0:
                print(json.dumps(line), flush=True)

    def watchdog():
        if not printed.wait(EXTRA_BUDGET_S):
            if line is not None:
                line.setdefault("extra", {})["error"] = f"extra block exceeded {EXTRA_BUDGET_S} s; line emitted by watchdog"
            emit()
            os._exit(0)

    threading.Thread(target=watchdog, daemon=True).start()

    # free the decode tensors before the extras (the MoE weights alone are 22.6 GB)
    del d, kc, vc, out, task_map, dev_buf, host_buf, y, args, keep
    torch.cuda.empty_cache()

    extra = {}
    if not a.no_extra:
        sys.path.insert(0, str(REPO / "tools"))
        import bench_extras as bx

        def leg(name, fn):
            t0 = time.perf_counter()
            smp = ClockSampler(local_rank) if rank == 0 else None  # clocks / throttle reasons of this leg
            if smp:
                smp.start()
            try:
                r = fn()
                if isinstance(r, dict):
                    r["wall_s"] = time.perf_counter() - t0
                extra[name] = r
            except Exception as ex:  # noqa: BLE001  (a failed leg is reported, not hidden)
                extra[name] = {"error": repr(ex)[:400]}
            if smp:
                extra[name]["clocks"] = smp.stop()

        if world == 1:
            leg("moe_c3", lambda: bx.moe_c3(hpc, dev))
            leg("prefill_c4_kv_per_tensor", lambda: bx.prefill_c4(hpc, dev, kpt=False))
            leg("prefill_c4_k_per_token", lambda: bx.prefill_c4(hpc, dev, kpt=True))
            leg("route_gemm", lambda: bx.route_gemm(hpc, dev))
        leg("allreduce_c5", lambda: bx.allreduce_c5(hpc, dev, rank, world, dist))
        extra["peaks"] = bx.peaks()
    if rank == 0:
        line["extra"] = extra
    emit()
    if dist is not None:
        try:
            dist.barrier()  # ranks > 0 wait for rank 0 instead of tearing NCCL down early
            dist.destroy_process_group()
        except Exception:  # noqa: BLE001
            pass
        sys.stdout.flush()
        # with several ranks, symmetric-memory handles and NCCL teardown order must not turn a
        # finished run into a hang; a single process returns normally
        os._exit(0)


if __name__ == "__main__":
    main()
