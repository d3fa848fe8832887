"""Drop-in surface (SURVEY.md §8b): the in-scope `torch.ops.hpc.*` operators exist with the reference's
schemas and the `hpc` package exports the reference's public functions. CPU only (no compute).

The reference's schemas are stored in tests/golden/reference_schemas.json, parsed out of its
TORCH_LIBRARY_FRAGMENT blocks by tests/golden/make_golden.py, and compared one by one."""
import json
import re
from pathlib import Path

import torch

GOLD = Path(__file__).resolve().parent / "golden" / "reference_schemas.json"

IN_SCOPE_OPS = [
    "assign_attention_decode_task", "attention_decode_fp8", "attention_decode_bf16",
    "attention_with_kvcache_blocksparse_prefill_fp8", "attention_with_kvcache_prefill_fp8",
    "fuse_moe", "fuse_moe_pertensor_fp8", "fuse_moe_blockwise", "fuse_moe_blockwise_fp8",
    "count_and_gather", "reduce",
    "group_gemm_fp8", "group_gemm_pertensor_fp8", "group_gemm_blockwise_fp8", "reformat_x_scale",
    "group_gemm_fp8_cp_async", "group_gemm_fp8_scatter_cp_async",
    "act_mul_and_quant", "scaled_fp8_quant",
    "gemm_bf16xfp32",
    "fuse_allreduce_rmsnorm_high_throughput", "fuse_allreduce_rmsnorm_low_latency",
    "version", "built_json",
]

PUBLIC_FUNCS = [
    "QuantType", "assign_attention_decode_task", "attention_decode_fp8", "attention_decode_bf16",
    "attention_with_kvcache_blocksparse_prefill_fp8", "attention_with_kvcache_prefill_fp8",
    "get_attention_decode_task_workspace",
    "print_attention_decode_task",
    "count_and_gather", "fuse_moe", "fuse_moe_blockwise", "fuse_moe_blockwise_fp8",
    "fuse_moe_pertensor_fp8", "reduce",
    "group_gemm_blockwise_fp8", "group_gemm_fp8", "group_gemm_pertensor_fp8", "reformat_x_scale",
    "gemm_bf16xfp32", "get_gemm_bf16xfp32_workspace",
    "empty_multimem", "fuse_allreduce_rmsnorm_high_throughput", "fuse_allreduce_rmsnorm_low_latency",
    "MulticastHandle", "MulticastCommunicator",
    "act_mul_and_quant", "scaled_fp8_quant",
]


def test_ops_registered(hpc):
    for name in IN_SCOPE_OPS:
        assert hasattr(torch.ops.hpc, name), f"torch.ops.hpc.{name} missing"
        getattr(torch.ops.hpc, name)  # resolves the overload packet


def test_public_functions_exported(hpc):
    missing = [n for n in PUBLIC_FUNCS if not hasattr(hpc, n)]
    assert not missing, missing
    assert isinstance(hpc.__version__, str) and isinstance(hpc.__built_json__, str)


def _canon(schema) -> str:
    """Canonical text of a schema with alias / mutation annotations removed: this build marks the
    tensors its Python impls write (`Tensor(a!)`) where the reference's C++ registrations leave
    them unannotated; names, types, order, defaults and returns must be identical."""
    text = str(torch._C.parse_schema(schema) if isinstance(schema, str) else schema)
    return re.sub(r"\(\$?\w+!?( -> [^)]*)?\)", "", text)


def test_schemas_match_reference(hpc):
    ref = json.loads(GOLD.read_text())
    checked = 0
    for name in IN_SCOPE_OPS:
        if name not in ref:  # version / built_json are registered from function signatures
            continue
        mine = _canon(getattr(torch.ops.hpc, name).default._schema)
        want = _canon("hpc::" + ref[name])
        assert mine == want, f"{name}:\n  mine {mine}\n  ref  {want}"
        checked += 1
    assert checked >= 20
