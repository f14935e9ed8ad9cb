"""not-gpu: libktb200.so loads, exports every symbol include/ktb200.h declares, and the host-only
entry points (shard bounds, pack layout, argument validation) behave without a GPU."""
import ctypes
import os
import re

import pytest
import torch

from conftest import REPO
from kubetorch_b200.device import lib as L


def _declared_symbols():
    text = open(os.path.join(REPO, "include", "ktb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ktb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = L.load()
    names = _declared_symbols()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} declared in ktb200.h but not exported"
        assert n in L._SIGNATURES, f"{n} has no ctypes prototype"
    assert lib.ktb_version() == 100


def test_library_is_sm100a_only():
    import subprocess

    from __graft_entry__ import cuda_tool

    out = subprocess.run([cuda_tool("cuobjdump"), "-lelf", L.lib_path()], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_mlp_kernels_issue_tcgen05_and_tma_without_waterfall_loops():
    """The shipped MLP kernels (layer-1 form, generic CTA-pair kernel, fused layer 2 + head) are tcgen05 / TMA kernels whose
    single-lane instructions are issued from converged warps through elect.sync: no UTCHMMA / UTMALDG / UTMASTG sits in
    an ELECT + R2UR.BROADCAST + BRA.U.ANY loop (that form issued one MMA per ~177 cycles instead of 128)."""
    import subprocess

    from __graft_entry__ import cuda_tool

    sass = subprocess.run([cuda_tool("cuobjdump"), "-sass", L.lib_path()], capture_output=True, text=True).stdout
    funcs = sass.split("Function : ")[1:]
    wanted = {"gemm_bf16_tn_2sm_bres_kernel": 0, "gemm_bf16_tn_2sm_kernel": 0, "mlp_l2_head_fused_kernel": 0}
    for f in funcs:
        name = f.split("\n", 1)[0]
        for key in wanted:
            if key + "I" in name:          # mangled: <name>I<template args>
                wanted[key] += 1
                assert "UTCHMMA.2CTA" in f and "UTMALDG" in f and "LDTM" in f, name
                assert "BRA.U.ANY" not in f, name      # the loop-back branch of the waterfall
    assert all(v >= 1 for v in wanted.values()), wanted


@pytest.mark.parametrize("n,world", [(0, 1), (1, 4), (3, 4), (5, 4), (1003, 4), (1000, 3), (64, 8), (2**26, 8), (7, 7)])
def test_shard_bounds_equal_torch_chunk(n, world):
    x = torch.arange(n)
    chunks = x.chunk(world) if n else ()
    for r in range(world):
        b, e = ctypes.c_size_t(), ctypes.c_size_t()
        L.call("ktb_shard_bounds", n, world, r, ctypes.byref(b), ctypes.byref(e))
        from kubetorch_b200.device import ops

        assert ops.shard_bounds(n, world, r) == (b.value, e.value)   # the Python twin agrees with the C entry
        want = chunks[r] if r < len(chunks) else x[:0]
        assert e.value - b.value == want.numel()
        if want.numel():
            assert (b.value, e.value - 1) == (int(want[0]), int(want[-1]))
    with pytest.raises(L.KtbError):
        L.call("ktb_shard_bounds", 10, 0, 0, ctypes.byref(b), ctypes.byref(e))


def test_pack_layout_is_256_aligned_and_ordered():
    sizes = [1, 0, 255, 256, 257, 4096, 3, 10**6]
    offs = (ctypes.c_size_t * len(sizes))()
    total = ctypes.c_size_t()
    L.call("ktb_pack_layout", L.arr(ctypes.c_size_t, sizes), len(sizes), offs, ctypes.byref(total))
    off = 0
    for o, s in zip(offs, sizes):
        assert o == off and o % 256 == 0
        off += -(-s // 256) * 256
    assert total.value == off


def test_calls_fail_loudly_without_registered_device():
    buf = (ctypes.c_float * 8)()
    with pytest.raises(L.KtbError) as ei:
        L.call("ktb_map", 0, L.OP_SCALE, L.F32, buf, buf, 8, 2.0, 0.0, 0, 0)
    assert ei.value.status == L.ERR_STATE and "ktb_init" in str(ei.value)
    if not torch.cuda.is_available():
        with pytest.raises(L.KtbError):
            L.call("ktb_init", 1, L.arr(ctypes.c_int, [0]))


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_device_backend_has_no_cpu_fallback():
    import kubetorch_b200 as kt
    from oracle import cases

    from conftest import mapped_copy

    double = mapped_copy(cases.double, "scale", alpha=2.0)
    with pytest.raises(Exception) as ei:
        kt.fn(double, name="no-gpu").to(kt.Compute(gpus=1))
    assert "CUDA" in str(ei.value) or "cuda" in str(ei.value)
    from kubetorch_b200.device import ops

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.ensure_init([0])
    with pytest.raises(ValueError, match="must be a CUDA tensor"):
        ops.map_tensor(torch.ones(4), "scale", 2.0)


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under kubetorch_b200/ may import it."""
    for root, _, files in os.walk(os.path.join(REPO, "kubetorch_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(root, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), os.path.join(root, f)


def test_bench_reference_arm_emits_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): one JSON line with the contract's keys."""
    import json
    import subprocess
    import sys

    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=REPO)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["value"] > 0 and line["config"].get("workload")
    # the unmodified reference when baseline/_ref travelled with the repo (install_reference.py), else the oracle port
    want_kind = "reference" if os.path.isdir(os.path.join(REPO, "baseline", "_ref", "kubetorch")) else "port"
    assert line["cpu_baseline"]["kind"] == want_kind and line["cpu_baseline"]["cores"] == os.cpu_count()
    assert line["config"]["parallelism"] == "dp1" and "64 MiB arg" in line["cpu_baseline"]["sample"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
