"""Generate the golden fixtures in tests/golden/ from the REFERENCE's own code.

Needs a checkout of the original hpc-ops sources; the tests only read the stored fixtures:
    python tests/golden/make_golden.py <hpc-ops checkout>

* attention: the reference keeps its ground truth as pure-torch functions inside its test files.
  Those files `import hpc` at module level (needs their CUDA build), so we AST-extract the
  reference function's source text and exec it unmodified on CPU tensors.
* task map: outputs of the real reference CPU scheduler compiled in place (oracle/_ref, see
  oracle/Makefile `make ref`). Pad ints 9..11 of each row are uninitialised stack bytes in the
  reference (assign_task.cu:424 `TaskScheduleInfo task_info;`) and are stored zeroed.
"""
import ast
import json
import math
import re
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parents[2]
REF = None  # the original project's checkout, from the command line
OUT = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

from oracle import attention as oa  # noqa: E402
from oracle import taskmap as otm  # noqa: E402


def extract(path: Path, name: str):
    src = path.read_text()
    tree = ast.parse(src)
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name == name:
            code = ast.get_source_segment(src, node)
            ns = {"torch": torch, "math": math, "F": torch.nn.functional}
            exec(compile(code, str(path), "exec"), ns)
            return ns[name]
    raise KeyError(name)


def u8(t):
    return t.contiguous().view(torch.uint8).numpy()


def decode_fp8_case(tag, num_batch, kv_lens, hkv, hq, seed, layout):
    fn = extract(REF / "tests/test_attention_decode_qpertoken_perhead_kvpertensor_fp8.py",
                 "ref_attn_with_paged_kvcache_func")
    d = oa.make_decode_fp8_inputs(num_batch, 1, kv_lens, hkv, hq, seed=seed, layout=layout)
    lens = d["kv_lens_total"]
    nblocks = (lens + 63) // 64
    seqlenq = torch.ones(num_batch, dtype=torch.int32)
    kdummy = torch.empty(num_batch, hkv, 128)
    gt = fn(d["q"], kdummy, kdummy, d["kvcache"], d["block_ids"], nblocks, seqlenq, None,
            lens - 1, d["q_scale"], d["k_scale"], d["v_scale"])
    np.savez_compressed(
        OUT / f"decode_fp8_{tag}.npz", q=u8(d["q"]), q_scale=d["q_scale"].numpy(),
        kvcache=u8(d["kvcache"].contiguous()), k_scale=d["k_scale"].numpy(),
        v_scale=d["v_scale"].numpy(), block_ids=d["block_ids"].numpy(), kv_lens_total=lens.numpy(),
        out=gt.float().numpy(), meta=np.array([num_batch, 1, hkv, hq, 128, 64]),
        layout=np.array([0 if layout == "NHD" else 1]))
    print("wrote", tag, gt.shape)


def decode_fp8_kpt_case(tag, num_batch, kv_lens, hkv, hq, seed, layout):
    """k-per-token variant: the reference's own ref function on the in-cache scale layout."""
    fn = extract(REF / "tests/test_attention_decode_qkpertoken_perhead_vperhead_fp8.py",
                 "ref_attn_with_paged_kvcache_func")
    d = oa.make_decode_fp8_kpt_inputs(num_batch, 1, kv_lens, hkv, hq, seed=seed, layout=layout)
    lens = d["kv_lens_total"]
    nblocks = (lens + 63) // 64
    seqlenq = torch.ones(num_batch, dtype=torch.int32)
    kdummy = torch.empty(num_batch, hkv, 128)
    gt = fn(d["q"], kdummy, kdummy, d["kvcache"][:, :, :64], d["block_ids"], nblocks, seqlenq, None,
            lens - 1, d["q_scale"], d["k_scale"].contiguous(), d["v_scale"])
    np.savez_compressed(
        OUT / f"decode_fp8_kpt_{tag}.npz", q=u8(d["q"]), q_scale=d["q_scale"].numpy(),
        kvcache=u8(d["kvcache"].contiguous()), v_scale=d["v_scale"].numpy(),
        block_ids=d["block_ids"].numpy(), kv_lens_total=lens.numpy(), out=gt.float().numpy(),
        meta=np.array([num_batch, 1, hkv, hq, 128, 64]),
        layout=np.array([0 if layout == "NHD" else 1]))
    print("wrote kpt", tag, gt.shape)


def _bf16_bits(t):
    return t.to(torch.bfloat16).contiguous().view(torch.int16).numpy()


def rope_case(tag, num_req, is_prefill, mtp, hq, hkv, policy, seed):
    """reference tests/test_rope.py `rope_norm_ref` (with its helpers) on seeded CPU inputs
    (16-token pages keep the fixture small; bf16 tensors are stored as their bit patterns)."""
    from synth import rope as sr
    ns = extract_many(REF / "tests/test_rope.py", {"apply_rms_norm_reference",
                                                    "apply_rotary_pos_emb_neox_reference", "rope_norm_ref"})
    d = sr.make_inputs(num_req, is_prefill, mtp, hq, hkv, 128, kv_block_size=16, max_num_kv_blocks=24,
                       max_rope_position=128, seed=seed, len_range=(10, 60), pad_decode=False)
    kc, vc = d["kcache"].clone(), d["vcache"].clone()
    q = ns["rope_norm_ref"](kc, vc, d["qkv"], d["cos_sin"], d["num_seqlen"], d["q_index"],
                            d["kv_indices"], d["q_norm_w"], d["k_norm_w"], policy)
    np.savez_compressed(
        OUT / f"rope_{tag}.npz", qkv=_bf16_bits(d["qkv"]), num_seqlen=d["num_seqlen"].numpy(),
        q_index=d["q_index"].numpy(), kv_indices=d["kv_indices"].numpy(),
        kcache_in=_bf16_bits(d["kcache"]), vcache_in=_bf16_bits(d["vcache"]),
        q_norm_w=d["q_norm_w"].numpy(), k_norm_w=d["k_norm_w"].numpy(), cos_sin=d["cos_sin"].numpy(),
        out_q=_bf16_bits(q), kcache_out=_bf16_bits(kc), vcache_out=_bf16_bits(vc),
        meta=np.array([num_req, int(is_prefill), -1 if mtp is None else mtp, hq, hkv, policy]))
    print("wrote rope", tag, q.shape)


def decode_bf16_case(tag, num_batch, num_seq_q, kv_lens, hkv, hq, block_size, seed, layout):
    """head-dim-128 bf16 decode: the reference's own ref function (tests/test_attention_decode_bf16.py:15)."""
    fn = extract(REF / "tests/test_attention_decode_bf16.py", "ref_attn_with_paged_kvcache_func")
    d = oa.make_decode_bf16_inputs(num_batch, num_seq_q, kv_lens, hkv, hq, block_size=block_size,
                                   seed=seed, layout=layout, extra_blocks=2)
    lens = d["kv_lens_total"]
    nblocks = (lens + block_size - 1) // block_size
    seqlenq = torch.full((num_batch,), num_seq_q, dtype=torch.int32)
    kdummy = torch.empty(num_batch * num_seq_q, hkv, 128)
    gt = fn(d["q"], kdummy, kdummy, d["kvcache"], d["block_ids"], nblocks, seqlenq, None,
            lens - num_seq_q)
    np.savez_compressed(
        OUT / f"decode_bf16_{tag}.npz", q=_bf16_bits(d["q"]), kvcache=_bf16_bits(d["kvcache"].contiguous()),
        block_ids=d["block_ids"].numpy(), kv_lens_total=lens.numpy(), out=gt.float().numpy(),
        meta=np.array([num_batch, num_seq_q, hkv, hq, 128, block_size]),
        layout=np.array([0 if layout == "NHD" else 1]))
    print("wrote decode_bf16", tag, gt.shape)


def decode_bf16_c1():
    """BASELINE config 0: test_attention_decode_bf16 bs=2 h=4 d=64 seq=128 on the torch CPU path."""
    fn = extract(REF / "tests/test_attention_decode_bf16.py", "ref_attn_with_paged_kvcache_func")
    torch.manual_seed(41)
    B, Hkv, Hq, D, bs = 2, 1, 4, 64, 64
    lens = torch.randint(1, 128, (B,), dtype=torch.int32) + 1
    nblocks = (lens + bs - 1) // bs
    q = (torch.randn(B, Hq, D) / math.sqrt(D)).to(torch.bfloat16)
    kvcache = (torch.randn(8, 2, bs, Hkv, D) / math.sqrt(D)).to(torch.bfloat16)
    block_ids = torch.zeros(B, int(nblocks.max()), dtype=torch.int32)
    perm = torch.randperm(8)
    cu = 0
    for i in range(B):
        block_ids[i, : nblocks[i]] = perm[cu:cu + int(nblocks[i])]
        cu += int(nblocks[i])
    seqlenq = torch.ones(B, dtype=torch.int32)
    kd = torch.empty(B, Hkv, D)
    gt = fn(q, kd, kd, kvcache, block_ids, nblocks, seqlenq, None, lens - 1)
    np.savez_compressed(OUT / "decode_bf16_c1.npz", q=q.float().numpy(),
                        kvcache=kvcache.float().numpy(), block_ids=block_ids.numpy(),
                        kv_lens_total=lens.numpy(), out=gt.float().numpy())
    print("wrote decode_bf16_c1", gt.shape)


def taskmap_cases():
    assert otm.ref_lib() is not None, "run `make -C oracle ref` first"
    rng = np.random.default_rng(7)
    cases = []
    cfgs = [(1, 1, 1, 128, 148, 1024, 4096), (16, 4, 2, 128, 148, 1024, 4096),
            (200, 4, 4, 128, 148, 1024, 1024), (64, 8, 1, 128, 148, 64, 8193),
            (200, 1, 3, 64, 592, 1024, 4096), (33, 8, 4, 128, 148, 512, 300),
            (7, 2, 4, 128, 148, 64, 40000), (500, 8, 2, 64, 296, 2048, 700)]
    for i, (B, H, sq, tilen, ctas, mpl, mx) in enumerate(cfgs):
        lens = (rng.integers(1, mx, size=B) + sq).astype(np.int32)
        ref = otm.assign_ref(lens, ctas, H, sq, tilen, True, mpl)
        ref[1:1 + (ref[0, 0] * ctas), 9:] = 0
        cases.append(dict(lens=lens, cfg=np.array([B, H, sq, tilen, ctas, mpl]), out=ref))
    np.savez_compressed(OUT / "taskmap_ref.npz",
                        **{f"{k}_{i}": v for i, c in enumerate(cases) for k, v in c.items()},
                        n=np.array([len(cases)]))
    print("wrote taskmap_ref", len(cases))


def taskmap_random_cases():
    """Random configurations with the new token included. Their task maps come to ~15M rows, so
    each is stored as its row count and `taskmap_digest`; `lens` holds the cases' lengths back to
    back, `cfg` rows are [B, H, sq, tilen, ctas, mpl]."""
    assert otm.ref_lib() is not None, "oracle/_ref not built"
    sys.path.insert(0, str(OUT.parent))
    from test_oracle_taskmap import _random_cases, taskmap_digest
    lens, cfg, rows, sha = [], [], [], []
    for ln, ctas, H, sq, tilen, inc, mpl in _random_cases(300, 2):
        if inc:
            ref = otm.assign_ref(ln, ctas, H, sq, tilen, inc, mpl)
            lens.append(np.asarray(ln, np.int32))
            cfg.append([len(ln), H, sq, tilen, ctas, mpl])
            rows.append(ref.shape[0])
            sha.append(taskmap_digest(ref))
    np.savez_compressed(OUT / "taskmap_ref_random.npz", lens=np.concatenate(lens),
                        cfg=np.array(cfg, np.int32), rows=np.array(rows), sha256=np.stack(sha))
    print("wrote taskmap_ref_random", len(cfg))


def schemas():
    """Schema of every in-scope op, parsed out of the reference's `m.def("name(...) -> ...")`."""
    sys.path.insert(0, str(OUT.parent))
    from test_api_surface import IN_SCOPE_OPS
    out = {}
    for f in sorted(REF.glob("src/**/*.cc")):
        text = f.read_text(errors="ignore")
        for m in re.finditer(r"m\.def\(\s*((?:\"(?:[^\"\\]|\\.)*\"\s*)+)[,)]", text):
            schema = "".join(re.findall(r"\"((?:[^\"\\]|\\.)*)\"", m.group(1)))
            if "(" in schema:
                out[schema.split("(", 1)[0].strip()] = schema
    keep = {n: out[n] for n in IN_SCOPE_OPS if n in out}
    (OUT / "reference_schemas.json").write_text(json.dumps(keep, indent=1) + "\n")
    print("wrote reference_schemas", len(keep))


class _TorchCPU:
    """`torch` stand-in for exec'ing reference test functions that hard-code device="cuda"."""

    def __getattr__(self, name):
        attr = getattr(torch, name)
        if callable(attr) and not isinstance(attr, type):
            def wrapped(*a, **k):
                if k.get("device", None) == "cuda":
                    k["device"] = "cpu"
                return attr(*a, **k)
            return wrapped
        return attr


def extract_many(path: Path, names):
    src = path.read_text()
    tree = ast.parse(src)
    ns = {"torch": _TorchCPU(), "math": math, "F": torch.nn.functional, "Tuple": tuple}
    from typing import Tuple
    ns["Tuple"] = Tuple
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in names:
            exec(compile(ast.get_source_segment(src, node), str(path), "exec"), ns)
    return ns


def moe_blockwise_case(tag, T, K, H, I, E_total, size_ep, rank_ep, shared, seed):
    from oracle import moe as om
    ns = extract_many(REF / "tests/test_fuse_moe_blockwise.py",
                      {"naive_gather_expert_inputs", "naive_group_gemm",
                       "naive_act_mul_and_blockwise_quant", "naive_reduce",
                       "naive_fuse_moe_blockwise_fp8"})
    d = om.make_moe_blockwise_inputs(T, K, H, I, E_total, size_ep, shared, seed)
    gt = ns["naive_fuse_moe_blockwise_fp8"](
        d["x"], d["x_scale"], d["gate_up_weight"], d["gate_up_weight_scale"], d["down_weight"],
        d["down_weight_scale"], d["topk_ids"], d["topk_scale"], rank_ep, E_total,
        d["shared_output"])
    g = ns["naive_gather_expert_inputs"](d["x"], d["x_scale"], d["topk_ids"], E_total // size_ep, rank_ep)
    np.savez_compressed(
        OUT / f"moe_blockwise_{tag}.npz", x=u8(d["x"]), x_scale=d["x_scale"].numpy(),
        guw=u8(d["gate_up_weight"]), guws=d["gate_up_weight_scale"].numpy(),
        dw=u8(d["down_weight"]), dws=d["down_weight_scale"].numpy(),
        topk_ids=d["topk_ids"].numpy(), topk_scale=d["topk_scale"].numpy(),
        shared=(d["shared_output"].float().numpy() if shared else np.zeros(0, np.float32)),
        out=gt.float().numpy(), topk_pos=g[2].numpy(), counts=g[3].numpy(), cu=g[4].numpy(),
        meta=np.array([T, K, H, I, E_total, size_ep, rank_ep, int(shared)]))
    print("wrote moe_blockwise", tag, gt.shape)


def moe_pertensor_case(tag, T, K, H, I, E_total, size_ep, rank_ep, seed):
    ns = extract_many(REF / "tests/test_fuse_moe_pertensor.py",
                      {"naive_gather_expert_inputs", "naive_group_gemm", "naive_act_mul_and_quant",
                       "naive_reduce", "naive_fuse_moe_pertensor_fp8"})
    g = torch.Generator().manual_seed(seed)
    E = E_total // size_ep
    topk_ids = torch.multinomial(torch.ones((T, E_total)), K, replacement=False, generator=g).to(torch.int32)
    topk_ids, _ = torch.sort(topk_ids, dim=1)
    topk_scale = torch.rand((T, K), generator=g)
    x = torch.randn((T, H), generator=g).to(torch.float8_e4m3fn)
    guw = torch.randn((E, 2 * I, H), generator=g).to(torch.float8_e4m3fn)
    dw = torch.randn((E, H, I), generator=g).to(torch.float8_e4m3fn)
    gus = torch.rand((E,), generator=g) * 0.02
    ds = torch.rand((E,), generator=g) * 0.02
    acts = torch.rand((1,), generator=g) + 0.5
    gt = ns["naive_fuse_moe_pertensor_fp8"](x, guw, dw, gus, ds, acts, topk_ids, topk_scale, rank_ep, None)
    np.savez_compressed(OUT / f"moe_pertensor_{tag}.npz", x=u8(x), guw=u8(guw), dw=u8(dw),
                        gus=gus.numpy(), ds=ds.numpy(), acts=acts.numpy(), topk_ids=topk_ids.numpy(),
                        topk_scale=topk_scale.numpy(), out=gt.float().numpy(),
                        meta=np.array([T, K, H, I, E_total, size_ep, rank_ep]))
    print("wrote moe_pertensor", tag, gt.shape)


def prefill_case(tag, k_per_token, seq, Hq, Hkv, skip, layout, seed):
    from oracle import prefill as op
    if k_per_token:
        path = REF / "tests/test_attention_blocksparse_qkpertoken_perhead_vperhead_fp8.py"
        name = "naive_attn_with_kvcache_qkpv_sparse_fixed_pscale"
    else:
        path = REF / "tests/test_attention_blocksparse_qpertoken_perhead_kvpertensor_fp8.py"
        name = "naive_attn_with_kvcache_sparse_fixed_pscale"
    ns = extract_many(path, {name})
    ns["BSA_BLOCK"] = 128
    B = 2
    d = op.make_inputs([seq] * B, [seq] * B, Hq, Hkv, skip, k_per_token, seed=seed, layout=layout)
    gt = ns[name](d["q"].reshape(B, seq, Hq, 128), d["kcache"], d["vcache"], d["qscale"], d["kscale"],
                  d["vscale"], d["seqlens_kv"], d["block_ids"], block_mask=d["block_mask"], causal=True)
    kvc = torch.stack([d["kcache"], d["vcache"]], dim=1).contiguous()
    np.savez_compressed(
        OUT / f"prefill_{tag}.npz", q=u8(d["q"]), kv=u8(kvc), qscale=d["qscale"].numpy(),
        kscale=d["kscale"].numpy(), vscale=d["vscale"].numpy(), block_ids=d["block_ids"].numpy(),
        mask=(d["block_mask"].numpy() if d["block_mask"] is not None else np.zeros(0, bool)),
        out=gt.reshape(-1, Hq, 128).float().numpy(),
        meta=np.array([B, seq, Hq, Hkv, int(k_per_token), 0 if layout == "nhd" else 1]))
    print("wrote prefill", tag, gt.shape)


def act_case(tag, rows, half_cols, seed):
    """tests/test_act.py:20-28 `_act_mul_and_quant`, executed unmodified on CPU."""
    fn = extract(REF / "tests/test_act.py", "_act_mul_and_quant")
    sys.path.insert(0, str(REPO))
    from oracle import act as oact
    gate_up, scale = oact.make_act_inputs(rows, half_cols, seed)
    gt = fn(gate_up, scale)
    np.savez_compressed(OUT / f"act_{tag}.npz", gate_up=gate_up.float().numpy(),
                        scale=scale.numpy(), gt=u8(gt))
    print("wrote act", tag, gt.shape)


def allreduce_case(tag, world, n, hidden, seed):
    """tests/test_fuse_allreduce_rmsnorm_high_throughput.py:15-29 `ref_allreduce_rmsnorm` (+ `rmsnorm`),
    executed unmodified on CPU."""
    ns = extract_many(REF / "tests/test_fuse_allreduce_rmsnorm_high_throughput.py",
                      {"rmsnorm", "ref_allreduce_rmsnorm"})
    from oracle import allreduce as oar
    xs, residual, weight, n_pad = oar.make_inputs(world, n, hidden, seed)
    res, out = ns["ref_allreduce_rmsnorm"](xs, residual, weight, 1e-6)
    np.savez_compressed(OUT / f"allreduce_{tag}.npz", meta=np.array([world, n, hidden, seed]),
                        out_residual=res.float().numpy(), out=out.float().numpy())
    print("wrote allreduce", tag, out.shape)


def group_gemm_cases():
    """tests/test_group_gemm_pertensor.py:20-44 and tests/test_group_gemm_blockwise.py:20-47, executed
    unmodified on CPU (torch._scaled_mm has a CPU kernel in torch 2.11)."""
    g = torch.Generator().manual_seed(7)
    G, per, n, k = 4, 24, 256, 256
    seqlens = torch.tensor([24, 0, 7, 16], dtype=torch.int32)
    cu = torch.arange(G, dtype=torch.int32) * per  # groups start at multiples of `per` (padded m)
    m = G * per
    x = torch.randn((m, k), generator=g).to(torch.float8_e4m3fn)
    w = torch.randn((G, n, k), generator=g).to(torch.float8_e4m3fn)
    scale = torch.tensor(0.37, dtype=torch.float32)
    fn = extract(REF / "tests/test_group_gemm_pertensor.py", "naive_group_gemm_pertensor_fp8")
    y_pt = fn(x, w, seqlens, cu, scale)
    xscale = torch.rand((k // 128, m), generator=g) + 0.5
    wscale = torch.rand((G, n // 128, k // 128), generator=g) + 0.5
    fn2 = extract(REF / "tests/test_group_gemm_blockwise.py", "naive_group_gemm")
    y_bw = fn2(x, w, seqlens, cu, xscale, wscale)
    np.savez_compressed(OUT / "group_gemm_a.npz", x=u8(x), w=u8(w), seqlens=seqlens.numpy(),
                        cu=cu.numpy(), scale=scale.numpy(), xscale=xscale.numpy(),
                        wscale=wscale.numpy(), y_pertensor=y_pt.float().numpy(),
                        y_blockwise=y_bw.float().numpy(), per=np.array([per]))
    print("wrote group_gemm a", y_pt.shape)


if __name__ == "__main__":
    REF = Path(sys.argv[1]).resolve()
    subprocess.run(["make", "-C", str(REPO / "oracle"), "ref", f"REF={REF}"], check=True)
    allreduce_case("w4", 4, 13, 512, 10001)
    group_gemm_cases()
    act_case("a", 64, 256, 41)
    prefill_case("kvpt", False, 384, 4, 1, 0.5, "nhd", 10086)
    prefill_case("kpertoken", True, 320, 4, 2, 0.5, "hnd", 10086)
    moe_blockwise_case("a", 24, 4, 256, 128, 8, 2, 1, True, 41)
    moe_blockwise_case("b", 48, 8, 256, 256, 8, 1, 0, False, 7)
    moe_pertensor_case("a", 32, 4, 256, 128, 8, 1, 0, 5)
    decode_fp8_case("b2_nhd", 2, [100, 129], 1, 8, 41, "NHD")
    decode_fp8_case("b5_hnd", 5, [1, 64, 65, 300, 515], 2, 16, 10086, "HND")
    decode_fp8_kpt_case("b3_nhd", 3, [70, 129, 200], 1, 8, 41, "NHD")
    decode_fp8_kpt_case("b4_hnd", 4, [1, 64, 65, 300], 2, 8, 10086, "HND")
    rope_case("prefill_p2", 3, True, None, 4, 1, 2, 1)
    rope_case("decode_p1", 5, False, 1, 8, 2, 1, 2)
    decode_bf16_c1()
    decode_bf16_case("b3_bs16_nhd", 3, 2, [70, 129, 300], 1, 8, 16, 41, "NHD")
    decode_bf16_case("b4_bs64_hnd", 4, 1, [1, 64, 65, 260], 2, 8, 64, 10086, "HND")
    taskmap_cases()
    taskmap_random_cases()
    schemas()
