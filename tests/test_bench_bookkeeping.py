"""bench.py bookkeeping that needs no GPU: the per-kernel source hash that ties an ncu capture (profiles/traffic_r2.json) to
the build it was taken on ignores comments and blank lines, follows the code, and the committed capture carries it."""
import importlib.util
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_code_only_strips_comments_and_blank_lines():
    b = _bench()
    a = "int x = 1;   // one\n\n// a comment line\nint y = 2;\n"
    c = "int x = 1;\nint y = 2;   // two\n"
    assert b._code_only(a) == b._code_only(c) == "int x = 1;\nint y = 2;"


def test_kernel_sources_hash_follows_code_not_comments():
    b = _bench()
    d = os.path.join(ROOT, "transformer-mm-explainability_b200", "csrc")
    real = lambda f: open(os.path.join(d, f)).read()
    base = b.kernel_sources_hash("gemm_f16x3")
    assert base == b.kernel_sources_hash("gemm_f16x3", real)
    commented = lambda f: real(f) + "\n// a trailing remark\n"
    assert b.kernel_sources_hash("gemm_f16x3", commented) == base
    changed = lambda f: real(f) + ("\nint extra;\n" if f == "gemm_epilogue.cuh" else "")
    assert b.kernel_sources_hash("gemm_f16x3", changed) != base
    assert b.kernel_sources_hash("avg_heads", changed) == b.kernel_sources_hash("avg_heads")     # not one of its sources


def test_dump_outputs_float32_and_seeded_sample_under_limit(tmp_path):
    import numpy as np
    import torch
    b = _bench()
    small = {"R_text": torch.randn(3, 4, 4, dtype=torch.float64), "R_image": np.arange(6).reshape(3, 2)}
    b.dump_outputs(str(tmp_path / "small"), small)
    for k, v in small.items():
        got = np.load(tmp_path / "small" / f"{k}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, np.asarray(v, dtype=np.float32))
    b.DUMP_LIMIT_BYTES = 100_000                          # this module instance only
    n = 600
    big = {"a": np.random.default_rng(1).random((n, 10, 10)), "b": np.arange(n, dtype=np.float32)[:, None]}
    assert sum(v.size * 4 for v in big.values()) > b.DUMP_LIMIT_BYTES
    for d in ("big1", "big2"):
        b.dump_outputs(str(tmp_path / d), big)
    a1, b1 = (np.load(tmp_path / "big1" / f"{k}.npy") for k in ("a", "b"))
    assert a1.nbytes + b1.nbytes <= b.DUMP_LIMIT_BYTES and a1.shape[0] == b1.shape[0] > 0
    keep = b1[:, 0].astype(int)                          # the same samples of every array, in order
    assert np.all(np.diff(keep) > 0) and np.array_equal(a1, big["a"][keep].astype(np.float32))
    assert np.array_equal(a1, np.load(tmp_path / "big2" / "a.npy"))


def test_committed_traffic_capture_is_tied_to_kernel_sources():
    b = _bench()
    with open(os.path.join(ROOT, "profiles", "traffic_r2.json")) as f:
        d = json.load(f)
    for key in ("gemm_f16x3", "avg_heads"):
        rec = d[key]
        assert rec["dram_bytes"] > 0 and rec["sources_hash"] and list(rec["sources"]) == list(b.KERNEL_SOURCES[key])
        traffic, info = b.captured_traffic(key)
        assert traffic == rec["dram_bytes"] and isinstance(info["build_matches"], bool)
