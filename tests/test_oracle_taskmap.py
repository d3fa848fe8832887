"""Task-map parity on CPU: oracle (C restatement) vs the reference's golden outputs, vs the real
reference code on random configurations, and the product's CPU scheduler vs the oracle (bit-exact)."""
import ctypes
import hashlib
from pathlib import Path

import numpy as np

from oracle import taskmap as otm

GOLD = Path(__file__).resolve().parent / "golden" / "taskmap_ref.npz"
GOLD_RANDOM = GOLD.with_name("taskmap_ref_random.npz")


def product_cpu(lib_path, lens, ctas, H, sq, tilen, inc, mpl):
    lib = ctypes.CDLL(str(lib_path))
    lib.hpc_assign_attention_decode_task_host_bytes.restype = ctypes.c_int64
    lens = np.ascontiguousarray(lens, dtype=np.int32)
    p = lens.ctypes.data_as(ctypes.c_void_p)
    nb = lib.hpc_assign_attention_decode_task_host_bytes(p, ctas, len(lens), H, sq, tilen, int(inc), mpl)
    out = np.zeros(nb // 4, dtype=np.int32)
    rc = lib.hpc_assign_attention_decode_task_sync(p, ctas, len(lens), H, sq, tilen, int(inc), mpl,
                                                   out.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(nb))
    assert rc == 0
    return out.reshape(-1, 12)


def golden_cases():
    z = np.load(GOLD)
    for i in range(int(z["n"][0])):
        yield z[f"lens_{i}"], z[f"cfg_{i}"], z[f"out_{i}"]


def test_oracle_matches_reference_golden():
    for lens, cfg, ref in golden_cases():
        B, H, sq, tilen, ctas, mpl = map(int, cfg)
        got = otm.assign(lens, ctas, H, sq, tilen, True, mpl)
        assert got.shape == ref.shape
        assert np.array_equal(got, ref), (cfg, np.argwhere(got != ref)[:4])


def test_product_cpu_matches_reference_golden(lib_path):
    for lens, cfg, ref in golden_cases():
        B, H, sq, tilen, ctas, mpl = map(int, cfg)
        got = product_cpu(lib_path, lens, ctas, H, sq, tilen, True, mpl)
        assert np.array_equal(got, ref), cfg


def _random_cases(n, seed):
    rng = np.random.default_rng(seed)
    for _ in range(n):
        B = int(rng.choice([1, 2, 3, 16, 64, 200, 500, 2048]))
        H = int(rng.choice([1, 2, 4, 8]))
        sq = int(rng.choice([1, 2, 3, 4]))
        tilen = int(rng.choice([64, 128]))
        ctas = int(rng.choice([1, 4, 132, 148, 296, 592]))
        mpl = int(rng.choice([64, 512, 1024, 2048]))
        mx = int(rng.choice([5, 130, 1024, 4096, 40000]))
        inc = bool(rng.integers(0, 2))
        lens = rng.integers(1, mx, size=B) + (sq if inc else 0)
        yield lens, ctas, H, sq, tilen, inc, mpl


def test_product_cpu_matches_oracle_random(lib_path):
    for args in _random_cases(400, 1):
        a = otm.assign(*args)
        p = product_cpu(lib_path, *args)
        assert np.array_equal(a, p), args[1:]


def test_edge_cases(lib_path):
    cases = [
        ([1], 148, 1, 1, 128, True, 64),              # single token
        ([128], 148, 1, 1, 128, True, 64),            # exactly one tile
        ([129], 148, 8, 4, 128, True, 64),            # tail shorter than num_seq_q -> spill back
        ([130] * 7, 4, 2, 4, 64, True, 64),           # spill back across bins
        ([0, 5, 0, 9], 148, 2, 1, 128, False, 64),    # empty caches before the new token
        ([40000], 148, 1, 1, 128, True, 64),          # one pair split over every bin
        ([8192] * 64, 148, 8, 1, 128, True, 64),      # BASELINE config C2
    ]
    for lens, ctas, H, sq, tilen, inc, mpl in cases:
        a = otm.assign(lens, ctas, H, sq, tilen, inc, mpl)
        p = product_cpu(lib_path, lens, ctas, H, sq, tilen, inc, mpl)
        assert np.array_equal(a, p), (lens[:4], ctas, H, sq)
    # C2 shape facts used by DESIGN.md / bench: 32768 tiles over 148 bins -> 222 per bin
    a = otm.assign([8192] * 64, 148, 8, 1, 128, True, 64)
    assert a[0, 0] == 223 and a[0, 1] == 148


def taskmap_digest(tm):
    """SHA-256 of a packed task map with ints 9..11 of its task rows zeroed: those are
    uninitialised stack bytes in the reference."""
    tm = np.array(tm, dtype="<i4")
    tm[1:1 + tm[0, 0] * tm[0, 1], 9:] = 0
    return np.frombuffer(hashlib.sha256(tm.tobytes()).digest(), np.uint8)


def test_oracle_matches_real_reference_random():
    """Random configurations of `_random_cases(300, 2)` with the new token included, against the
    real reference scheduler's task maps (stored as row count and digest)."""
    z = np.load(GOLD_RANDOM)
    lens = np.split(z["lens"], np.cumsum(z["cfg"][:-1, 0]))
    for cfg, ln, rows, sha in zip(z["cfg"], lens, z["rows"], z["sha256"]):
        B, H, sq, tilen, ctas, mpl = map(int, cfg)
        a = otm.assign(ln, ctas, H, sq, tilen, True, mpl)
        assert a.shape[0] == rows, cfg
        assert np.array_equal(taskmap_digest(a), sha), cfg
