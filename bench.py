#!/usr/bin/env python
"""bench.py — parallel-map throughput of the kubetorch remote-map path on B200.

Workload (BASELINE.json configs[1]): x → 2x over 64 Mi fp32 elements (256 MiB arg + 256 MiB result)
sharded `x.chunk(N)` across N GPUs; a "step" is ONE remote call (scatter → exec → gather).

  value   arg+result GB/s, device-timed, args/results resident in the root GPU's HBM
          (N=1: one kernel on HBM; N>1: one process per GPU, each rank's kernel pulls its shard
          from rank 0's arena over NVLink via CUDA IPC and pushes its result back — strong scaling)
  e2e     the same metric through the public API (kt.fn(...).to(kt.Compute(gpus=N)) → remote(x))
          with HOST buffers: every step copies the args host→device and the results device→host
  roofline / cpu_baseline / clocks / gpu_launches: see the driver contract in DESIGN.md §Measurement.
  extra keys at every N (time-boxed, never fail the headline): `parity` (golden + ragged cases over the REAL
  peers against the oracle, before anything is timed), `small_calls` and `c5` (BASELINE configs[4]: calls/s and
  GB/s at 1 KiB / 1 MiB / 1 GiB through the public API), `c4_rollout` (configs[3]), `c3_ddp` (configs[2]).

`--impl reference` times the reference's own CPU dispatch path on the host cores: the UNMODIFIED reference
runtime from baseline/_ref (FastAPI app → supervisor → spawned ProcessWorkers, `kind: "reference"`) with
N = --gpus ranks on a 64 MiB sample of the same workload; when baseline/_ref is absent, the oracle port.

`--dump-outputs DIR` writes what the timed path returned in its last timed step: `DIR/result_sample.npy`, the
results at a fixed, seeded sample of 4 Mi positions (float32, 16 MiB; the full result is 256 MiB).  The input is
generated from a fixed seed, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

# the tree may be read-only: no bytecode caches from this process or the rank processes it starts
sys.dont_write_bytecode = True
os.environ["PYTHONDONTWRITEBYTECODE"] = "1"

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)


def _clone(fn):
    """A copy of an oracle callable to decorate (the shared function object stays undecorated)."""
    import types

    return types.FunctionType(fn.__code__, fn.__globals__, fn.__name__, fn.__defaults__, fn.__closure__)


N_ELEMS = 1 << 26  # 64 Mi fp32 = 256 MiB
METRIC = "parallel_map_arg_plus_result_GBps"
UNIT = "GB/s"
REF_SAMPLE_ELEMS = 1 << 24   # 64 MiB arg per reference call (the reference needs seconds per call; 256 MiB exceeds its
                             # nginx body cap anyway, SURVEY.md §8(d))
REF_DIR = os.path.join(REPO, "baseline", "_ref")
INPUT_SEED = 0
DUMP_SAMPLE = 1 << 22        # result positions written by --dump-outputs
DUMP_SEED = 1234


def timed_input():
    """The timed call's argument: 64 Mi fp32 drawn on the host from a fixed seed (the same on every device and run)."""
    import torch

    return torch.randn(N_ELEMS, dtype=torch.float32, generator=torch.Generator().manual_seed(INPUT_SEED))


def dump_index(device):
    """The fixed, seeded sample of result positions --dump-outputs writes, sorted."""
    import torch

    idx = torch.randint(0, N_ELEMS, (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(DUMP_SEED))
    return idx.sort().values.to(device)


def workload_config(n_gpus: int) -> dict:
    """Identical in both arms (the driver compares them): what is computed, not how."""
    return {
        "workload": "configs[1]: parallel map x->2x over 64Mi fp32 (256 MiB arg + 256 MiB result), x.chunk(N) shards "
                    "over N ranks, rank-ordered results",
        "n_elems": N_ELEMS, "parallelism": f"dp{n_gpus}",
    }


def _peaks():
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int = 0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)   # the sampler never outlives the benchmark, even when a section fails
            self._t = threading.Thread(target=self._read, daemon=True)
            self._t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ts, line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                mhz = float(parts[1])
                smax = float(parts[2])
            except ValueError:
                continue
            if t0 - 0.05 <= ts <= t1 + 0.15:
                sm.append(mhz)
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                     parts[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        if not sm:  # region shorter than one sample: use the nearest samples
            for ts, line in self.lines[-3:]:
                parts = [p.strip() for p in line.split(",")]
                try:
                    sm.append(float(parts[1]))
                    smax = float(parts[2])
                except (ValueError, IndexError):
                    pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# =========================================================================================================
# reference arm / cpu baseline
# =========================================================================================================
def have_reference() -> bool:
    return os.path.isdir(os.path.join(REF_DIR, "kubetorch"))


def time_reference_runtime(shape: str, steps: int, warmup: int, n_ranks: int, n_elems: int, timeout: float = 1500.0):
    """The UNMODIFIED reference runtime (baseline/_ref) in a child process.  Returns the runner's JSON."""
    work = tempfile.mkdtemp(prefix="kt_ref_")
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "LOCAL_WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "GROUP_RANK",
              "ROLE_RANK", "TORCHELASTIC_RUN_ID"):
        env.pop(k, None)            # the reference sets its own rank environment
    env["PYTHONPATH"] = os.pathsep.join([REF_DIR, REPO])
    env["HOME"] = work
    env["PYTHONDONTWRITEBYTECODE"] = "1"
    env["CUDA_VISIBLE_DEVICES"] = ""   # the reference arm is the CPU dispatch path: host cores only
    cmd = [sys.executable, os.path.join(REPO, "baseline", "ref_runner.py"), "--shape", shape, "--ranks", str(n_ranks),
           "--elems", str(n_elems), "--steps", str(steps), "--warmup", str(warmup)]
    p = subprocess.run(cmd, env=env, cwd=work, capture_output=True, text=True, timeout=timeout)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("REFRESULT ")]
    if p.returncode != 0 or not lines:
        raise RuntimeError(f"reference runner failed (rc={p.returncode}): {p.stderr[-1500:]}")
    return json.loads(lines[-1][len("REFRESULT "):])


def time_port(steps: int, warmup: int, n_ranks: int, n_elems: int):
    """The oracle port of the reference's dispatch path (pickle → base64 → JSON → one queue hop per rank → decode →
    run → encode → gather) on spawned rank processes."""
    import torch

    from oracle.ref_dispatch import OracleRuntime

    x = torch.randn(n_elems, dtype=torch.float32)
    per = []
    with OracleRuntime("oracle.cases", "double", n_ranks, "spmd", extra_path=REPO) as rt:
        for _ in range(max(1, warmup)):
            out = rt.call(x, serialization="pickle")
        ok = bool(torch.equal(torch.cat(out), x * 2))
        for _ in range(steps):
            t0 = time.perf_counter()
            rt.call(x, serialization="pickle")
            per.append(time.perf_counter() - t0)
    return {"shape": f"oracle port, {n_ranks} ranks", "per_call_s": per, "ok": ok, "elems": n_elems, "ranks": n_ranks}


def _summarise(r: dict) -> dict:
    mean = sum(r["per_call_s"]) / len(r["per_call_s"])
    nbytes = r["elems"] * 4
    return {"value": 2 * nbytes / mean / 1e9, "ms_per_step": mean * 1e3, "calls_per_sec": 1.0 / mean,
            "sample": f"x->2x over {r['elems']} fp32 ({nbytes >> 20} MiB arg + {nbytes >> 20} MiB result), {r['shape']}, "
                      f"{len(r['per_call_s'])} timed calls", "ok": r.get("ok")}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = max(1, args.gpus)
    cores = os.cpu_count() or 1
    steps, warmup = args.steps, max(args.warmup, 1)
    kind = "reference" if have_reference() else "port"
    if kind == "reference":
        main = _summarise(time_reference_runtime("testclient", steps, warmup, n, REF_SAMPLE_ELEMS))
    else:
        main = _summarise(time_port(steps, warmup, n, REF_SAMPLE_ELEMS))
    extras = {}
    try:   # second leg: the port on the same sample (the arm the GPU box can always run)
        if kind == "reference":
            extras["port"] = _summarise(time_port(3, 1, n, REF_SAMPLE_ELEMS))
    except Exception as e:  # noqa: BLE001
        extras["port"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    try:   # the N-pods x 1-rank shape of BASELINE.md §3 (real HTTP between uvicorn pods), small time box
        if kind == "reference":
            extras["reference_pods"] = _summarise(time_reference_runtime("pods", 3, 1, n, 1 << 22, timeout=600))
    except Exception as e:  # noqa: BLE001
        extras["reference_pods"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    line = {
        "impl": "reference", "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "calls_per_sec": main["calls_per_sec"],
        "config": workload_config(args.gpus),
        "reference_arm": {"what": "the reference's CPU dispatch path (pickle/base64/JSON/HTTP app/queues/spawned rank "
                                  "processes) on the host cores, bounded sample of the workload per step",
                          "ranks": n, "sample": main["sample"], "results_checked": main["ok"]},
        "cpu_baseline": {"value": main["value"], "unit": UNIT, "cores": cores, "kind": kind, "sample": main["sample"]},
        "e2e": {"value": main["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, **extras,
    }
    print(json.dumps(line), flush=True)


# =========================================================================================================
# our arm
# =========================================================================================================
def _timeboxed(fn, label):
    """Auxiliary sections never fail the headline measurement."""
    t0 = time.perf_counter()
    try:
        out = fn()
    except Exception as e:  # noqa: BLE001
        out = {"error": f"{type(e).__name__}: {e}"[:400]}
    if isinstance(out, dict):
        out["section_seconds"] = round(time.perf_counter() - t0, 2)
    return out


PARITY_CASES = [
    # (name, dtype, shape, op, alpha, beta, byte offset of the arg in the arena)
    ("f32_1003_scale", "float32", (1003,), "scale", 2.0, 0.0, 0),
    ("f32_3_fewer_rows_than_ranks", "float32", (3,), "scale", 2.0, 0.0, 0),
    ("bf16_777_affine_inexact", "bfloat16", (777,), "affine", 1.7, -0.3, 0),
    ("f16_515_affine", "float16", (515,), "affine", 1.7, -0.3, 0),
    ("u8_1000_identity", "uint8", (1000,), "identity", 1.0, 0.0, 0),
    ("i64_130_affine", "int64", (130,), "affine", -5, 11, 0),
    ("i32_515_scale_wraps", "int32", (515,), "scale", 65537, 0, 0),
    ("f32_rows_10x37_ragged", "float32", (10, 37), "affine", 0.1, 0.3, 0),
    ("f32_1001_misaligned_by_4", "float32", (1001,), "scale", 0.1, 0.0, 4),
    ("f32_1M_plus_5", "float32", ((1 << 20) + 5,), "affine", 0.5, 1.5, 0),
]


def _parity_input(dtype_name, shape, seed):
    import torch

    g = torch.Generator().manual_seed(seed)
    dt = getattr(torch, dtype_name)
    if dt.is_floating_point:
        return torch.randn(shape, generator=g).to(dt)
    if dt is torch.uint8:
        return torch.randint(0, 256, shape, generator=g, dtype=dt)
    return torch.randint(-(2 ** 20), 2 ** 20, shape, generator=g, dtype=dt)


def _oracle_result(x, op, alpha, beta, world):
    """Rank-ordered concat of what the reference's ranks return (oracle restatement of the dispatch path)."""
    import torch

    from oracle import cases, ref_dispatch

    if op == "identity":
        out = ref_dispatch.spmd_call(cases.identity, x, num_proc=world, serialization="pickle")
    elif op == "scale":
        out = ref_dispatch.spmd_call(cases.scale, x, alpha, num_proc=world, serialization="pickle")
    else:
        out = ref_dispatch.spmd_call(cases.affine, x, alpha, beta, num_proc=world, serialization="pickle")
    return torch.cat([o.reshape(-1) for o in out]) if out else x.reshape(-1)[:0]


def run_ours(args):
    import ctypes

    import numpy as np
    import torch
    import torch.distributed as dist

    import kubetorch_b200 as kt
    from kubetorch_b200.device import lib as L
    from kubetorch_b200.device import ops
    from oracle import cases

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a B200"
    if world > 1:
        assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    dev = local_rank if world > 1 else 0
    torch.cuda.set_device(dev)
    cpu_group = None
    if world > 1:
        dist.init_process_group("cpu:gloo,cuda:nccl", device_id=torch.device(f"cuda:{dev}"))
        cpu_group = dist.new_group(backend="gloo")  # host-side waits must not spin on a GPU
    n_gpus = world if world > 1 else args.gpus
    K, W = args.steps, max(args.warmup, 3)
    lib = L.load()
    ops.ensure_init([dev])
    es = 4
    nbytes = N_ELEMS * es
    dtype_codes = {"float32": L.F32, "bfloat16": L.BF16, "float16": L.F16, "uint8": L.U8, "int64": L.I64, "int32": L.I32}
    op_codes = {"identity": L.OP_IDENTITY, "scale": L.OP_SCALE, "affine": L.OP_AFFINE}

    # ---- device-resident path -------------------------------------------------------------------------------
    # call_pull(n_elems, granule, dtype, op, alpha, beta, byte_off) / call_push(...): ONE remote call in each transfer
    # mode; the timed configuration is (N_ELEMS, 1, F32, SCALE, 2, 0, 0), the parity section replays other shapes
    # through the very same functions.
    TIMED = (N_ELEMS, 1, L.F32, L.OP_SCALE, 2.0, 0.0, 0)
    x = y = None
    x_src = timed_input() if rank == 0 else None
    if world == 1:
        devices = list(range(n_gpus))
        ops.ensure_init(devices)
        x = x_src.to("cuda:0")
        y = torch.empty_like(x)
        x_ptr, y_ptr = x.data_ptr(), y.data_ptr()
        c_devs = L.arr(ctypes.c_int, devices)

        def call_pull(n, gran, dt, op, a, b, off):
            streams = L.arr(L.c_uintptr, [ops.current_stream_handle(d) for d in devices])
            L.call("ktb_scatter_map_gather", op, dt, x_ptr + off, y_ptr + off, n, gran, float(a), float(b), n_gpus,
                   c_devs, 0, L.VARIANT_AUTO, streams)

        call_push = None
        if n_gpus > 1:
            session = ops.PushSession(devices, ops.shard_bounds(N_ELEMS, n_gpus, 0)[1] * es, n_chunks=args.push_chunks)
            names = {v: k for k, v in op_codes.items()}
            tdt = {L.F32: torch.float32, L.BF16: torch.bfloat16, L.F16: torch.float16, L.U8: torch.uint8,
                   L.I64: torch.int64, L.I32: torch.int32}

            def call_push(n, gran, dt, op, a, b, off):
                esz = torch.empty((), dtype=tdt[dt]).element_size()
                xv = x.view(torch.uint8)[off:off + n * esz].view(tdt[dt]).view(n // gran, gran)
                yv = y.view(torch.uint8)[off:off + n * esz].view(tdt[dt]).view(n // gran, gran)
                session.call(xv, yv, names[op], a, b)
    else:
        # rank 0 owns the arg/result arenas; every rank owns a control block and a staging arena; all are
        # cross-mapped through CUDA IPC.  Two transfer modes are timed (pull+push fused kernel, push/push
        # pipeline with in-kernel flags); `value` reports the faster one.
        n_chunks = args.push_chunks
        stride = (ops.shard_bounds(N_ELEMS, world, 0)[1] * es + 255) // 256 * 256
        ctrl = ops.Arena(dev, lib.ktb_push_control_bytes(), zero=True)
        stage = ops.Arena(dev, 2 * stride) if rank != 0 else None
        mine = {"ctrl": ctrl.export(), "stage": stage.export() if stage else None, "x": None, "y": None}
        if rank == 0:
            ax, ay = ops.Arena(dev, nbytes), ops.Arena(dev, nbytes)
            mine["x"], mine["y"] = ax.export(), ay.export()
            x, y = ax.tensor(torch.float32), ay.tensor(torch.float32)
            x.copy_(x_src)
            torch.cuda.synchronize()
            x_ptr, y_ptr = ax.ptr, ay.ptr
        everyone = [None] * world
        dist.all_gather_object(everyone, mine)
        if rank == 0:
            ctrl_ptrs = [ctrl.ptr] + [ops.ipc_open(dev, everyone[r]["ctrl"]) for r in range(1, world)]
            stage_ptrs = [0] + [ops.ipc_open(dev, everyone[r]["stage"]) for r in range(1, world)]
            c_stage = L.arr(ctypes.c_void_p, stage_ptrs)
            c_ctrl = L.arr(ctypes.c_void_p, ctrl_ptrs)
            ctrl_root_ptr = ctrl.ptr
        else:
            x_ptr = ops.ipc_open(dev, everyone[0]["x"])
            y_ptr = ops.ipc_open(dev, everyone[0]["y"])
            ctrl_root_ptr = ops.ipc_open(dev, everyone[0]["ctrl"])
        stream = torch.cuda.current_stream(dev).cuda_stream
        side = torch.cuda.Stream(dev)
        ev_fork, ev_join = torch.cuda.Event(), torch.cuda.Event()
        seq_box = [0]
        esize = {L.F32: 4, L.BF16: 2, L.F16: 2, L.U8: 1, L.I64: 8, L.I32: 4}

        def call_pull(n, gran, dt, op, a, b, off):
            bb, ee = ops.shard_bounds(n // gran, world, rank)
            if ee > bb:
                e_ = esize[dt]
                L.call("ktb_map", dev, op, dt, x_ptr + off + bb * gran * e_, y_ptr + off + bb * gran * e_,
                       (ee - bb) * gran, float(a), float(b), L.VARIANT_AUTO, stream)

        lanes = [torch.cuda.Stream(dev), torch.cuda.Stream(dev)] if rank == 0 else None

        def call_push(n, gran, dt, op, a, b, off, lane=None):
            """lane = None: on the current stream; 0/1: rank 0 issues on one of two alternating streams, so that the
            scatter of call k+1 overlaps the gather of call k (two calls in flight; staging and counters are per parity)."""
            seq_box[0] += 1
            seq = seq_box[0]
            e_ = esize[dt]
            bb, ee = ops.shard_bounds(n // gran, world, rank)
            if rank == 0:
                cur = torch.cuda.current_stream(dev) if lane is None else lanes[lane]
                st_ = cur.cuda_stream
                if ee > bb:   # the root's own shard maps on a side stream, forked and launched before the scatter
                    ev_fork.record(cur)
                    side.wait_event(ev_fork)
                    L.call("ktb_map", dev, op, dt, x_ptr + off + bb * gran * e_, y_ptr + off + bb * gran * e_,
                           (ee - bb) * gran, float(a), float(b), L.VARIANT_AUTO, side.cuda_stream)
                    ev_join.record(side)
                L.call("ktb_push_scatter", dev, x_ptr + off, n, gran, dt, world, 0, c_stage, stride, c_ctrl,
                       ctrl_root_ptr, n_chunks, seq, st_)
                L.call("ktb_push_wait", dev, ctrl_root_ptr, world, 0, seq, st_)
                if ee > bb:
                    cur.wait_event(ev_join)
            else:
                L.call("ktb_push_consume", dev, op, dt, stage.ptr, stride, y_ptr + off + bb * gran * e_,
                       (ee - bb) * gran, float(a), float(b), ctrl.ptr, ctrl_root_ptr, rank, n_chunks, seq, stream)

    def sync_all():
        if world == 1:
            for d in range(n_gpus):
                torch.cuda.synchronize(d)
        else:
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()

    # ---- real-peer parity BEFORE anything is timed: golden + ragged + misaligned shards vs the oracle -------------
    def parity_over_peers():
        report = {"cases": 0, "modes": ["pull_push_fused_kernel"] + (["push_push_flag_pipeline"] if call_push else []),
                  "oracle": "oracle.ref_dispatch.spmd_call on the same inputs; full torch.equal on the bytes"}
        for mode, fn in (("pull", call_pull), ("push", call_push)):
            if fn is None:
                continue
            for i, (name, dtn, shape, op, a, b, off) in enumerate(PARITY_CASES):
                xin = _parity_input(dtn, shape, 100 + i)
                n = xin.numel()
                gran = n // shape[0]
                nb = n * xin.element_size()
                if rank == 0:
                    x.view(torch.uint8)[off:off + nb].copy_(xin.reshape(-1).view(torch.uint8).cuda(dev))
                    y.view(torch.uint8)[off:off + nb + 64].zero_()
                sync_all()
                fn(n, gran, dtype_codes[dtn], op_codes[op], a, b, off)
                sync_all()
                if rank == 0:
                    got = y.view(torch.uint8)[off:off + nb].cpu()
                    want = _oracle_result(xin, op, a, b, n_gpus).reshape(-1).view(torch.uint8)
                    if got.numel() != want.numel() or not torch.equal(got, want):
                        raise SystemExit(f"PARITY FAILURE over real peers: case {name}, mode {mode}, N={n_gpus}")
                    report["cases"] += 1
        if rank == 0:   # restore the timed input
            x.copy_(x_src)
            torch.cuda.synchronize()
        sync_all()
        return report

    parity = parity_over_peers()

    def time_mode(fn):
        """W warm-up calls, then K timed calls bracketed by barrier + synchronize; device time, max over ranks."""
        for _ in range(W):
            fn(*TIMED)
        sync_all()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0w = time.time()
        ev0.record()
        for _ in range(K):
            fn(*TIMED)
        ev1.record()
        sync_all()
        t1w = time.time()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device=f"cuda:{dev}")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / K, t0w, t1w

    last_outputs = {}   # mode -> the dump sample of what that mode's last timed call returned

    def check_result(tag, mode):
        if rank == 0:
            idx = torch.randint(0, N_ELEMS, (4096,), device=x.device)
            assert torch.equal(y[idx], x[idx] * 2), f"{tag}: timed kernel produced wrong results"
            assert torch.equal(y[-1024:], x[-1024:] * 2), f"{tag}: tail wrong"
            if args.dump_outputs:
                last_outputs[mode] = y[dump_index(y.device)].cpu()
            y.zero_()
            torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def time_two_in_flight():
        """The push pipeline with TWO calls in flight (rank 0 alternates two streams): throughput of a caller that
        keeps the port busy both ways all the time.  Reported beside `value`, never as `value`."""
        for i in range(W + (W & 1)):
            call_push(*TIMED, lane=i & 1)
        sync_all()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        if rank == 0:
            for ln in lanes:
                ln.wait_event(ev0)
        for i in range(K):
            call_push(*TIMED, lane=i & 1)
        if rank == 0:
            for ln in lanes:
                e = torch.cuda.Event()
                e.record(ln)
                torch.cuda.current_stream(dev).wait_event(e)
        ev1.record()
        sync_all()
        ms = ev0.elapsed_time(ev1)
        t = torch.tensor([ms], device=f"cuda:{dev}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / K

    sampler = ClockSampler(dev)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    modes = {}
    ms_pull, t_wall0, t_wall1 = time_mode(call_pull)
    check_result("pull", "pull_push_fused_kernel")
    modes["pull_push_fused_kernel"] = ms_pull
    if n_gpus > 1 and call_push is not None:
        ms_push, t0b, t_wall1 = time_mode(call_push)
        check_result("push", "push_push_flag_pipeline")
        modes["push_push_flag_pipeline"] = ms_push
    two_in_flight = None
    if world > 1:
        # third mode: the SAME push/push pipeline with two calls in flight — rank 0 issues the K timed calls on two
        # alternating streams, so call k+1's scatter overlaps call k's gather and the root's port stays busy in both
        # directions (the protocol's per-parity staging halves and counters exist for exactly this).  Every call is a
        # complete scatter -> exec -> gather whose results are checked below; nothing is skipped, calls only overlap.
        try:
            ms2 = time_two_in_flight()
            check_result("push, two calls in flight", "push_push_flag_pipeline_two_calls_in_flight")
            modes["push_push_flag_pipeline_two_calls_in_flight"] = ms2
            two_in_flight = {"ms_per_step": ms2, "arg_plus_result_gbps": 2 * nbytes / (ms2 * 1e-3) / 1e9,
                             "root_port_gbps_per_direction": (n_gpus - 1) / n_gpus * nbytes / (ms2 * 1e-3) / 1e9,
                             "what": "push/push pipeline, rank 0 alternates two streams: call k+1's scatter overlaps call k's "
                                     "gather; ms_per_step is time per call at that throughput, per-call latency is the "
                                     "single-stream figure"}
        except Exception as e:  # noqa: BLE001
            two_in_flight = {"error": f"{type(e).__name__}: {e}"[:300]}
    # The timed region lasts a few milliseconds — shorter than one nvidia-smi sample — so the clocks are sampled over
    # an extended loop of the SAME call right after it (~0.6 s under load, all ranks take part).
    best_mode = min(modes, key=modes.get)
    if rank == 0 and args.dump_outputs:   # the mode `value` reports
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "result_sample.npy"), last_outputs[best_mode].numpy())
    if best_mode == "pull_push_fused_kernel" or call_push is None:
        probe_fn = call_pull
    elif best_mode.endswith("two_calls_in_flight"):
        lane_box = [0]

        def probe_fn(*a):
            lane_box[0] ^= 1
            call_push(*a, lane=lane_box[0])
    else:
        probe_fn = call_push
    t_probe0 = time.time()
    n_probe = 0
    while True:
        for _ in range(50):
            probe_fn(*TIMED)
        n_probe += 50
        if world == 1:
            torch.cuda.synchronize(0)
            if time.time() - t_probe0 >= 0.6:
                break
        else:
            torch.cuda.synchronize()
            flag = torch.tensor([1.0 if time.time() - t_probe0 < 0.6 else 0.0], device=f"cuda:{dev}")
            dist.broadcast(flag, src=0)          # rank 0's clock decides: every rank runs the same number of calls
            if flag.item() == 0.0:
                break
    sync_all()
    t_probe1 = time.time()
    clocks = sampler.stop(t_probe0, t_probe1) if rank == 0 else None
    if clocks is not None:
        clocks["window"] = f"extended loop of the timed call right after the timed region: {n_probe} calls"
    ms_per_step = modes[best_mode]
    value = 2 * nbytes / (ms_per_step * 1e-3) / 1e9
    # kernels launched inside the timed region, all ranks: fused mode = one map kernel per rank per call;
    # pipeline mode = root (scatter + own map + wait) + one consume kernel per other rank
    gpu_launches = K * (n_gpus if best_mode == "pull_push_fused_kernel" else 3 + (n_gpus - 1))

    # ---- roofline of the dominant kernel (map_vec_kernel<F32,SCALE,256-bit>) --------------------------------
    peak, peak_src = _peaks()
    shard_bytes = nbytes if n_gpus == 1 else (ops.shard_bounds(N_ELEMS, n_gpus, 0)[1]) * es
    traffic = _traffic(n_gpus)
    if n_gpus == 1:
        achieved = 2 * nbytes / (ms_per_step * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic.get("bytes"), "traffic_source": traffic.get("source"), "peak_source": peak_src,
                "kernel": "ktb::map_vec_kernel<F32,SCALE,32B>", "algorithmic_bytes_per_launch": 2 * nbytes}
    else:
        # root NVLink port: (N-1)/N of the arg leaves and of the result enters the root, full duplex
        link_bytes = (n_gpus - 1) * shard_bytes
        achieved = link_bytes / (ms_per_step * 1e-3) / 1e9
        roof = {"bound": "nvlink", "achieved": achieved, "peak": 770.0, "unit": "GB/s", "frac": achieved / 770.0,
                "traffic": traffic.get("bytes"), "traffic_source": traffic.get("source"),
                "peak_source": "measured peer copy per direction (B200_PROFILING.md)",
                "kernel": ("ktb::map_vec_kernel<F32,SCALE,32B> on peer pointers" if best_mode == "pull_push_fused_kernel"
                           else "ktb::push_scatter_kernel (root) + ktb::push_consume_kernel<F32,SCALE> (ranks)"),
                "algorithmic_bytes_per_launch": 2 * shard_bytes,
                "note": "bytes crossing the root GPU's NVLink port per direction per call / step time, both directions busy "
                        "at once. Measured ceiling of this duplex pattern with INDEPENDENT streams (no scatter->gather "
                        "dependency): 689 GB/s per direction at N=2, 618 at N=8 (profiles/r2_summary.md §1); one GPU "
                        "driving both directions caps at 489",
                "duplex_ceiling_gbps": 689.0 if n_gpus == 2 else 618.0,
                "frac_of_duplex_ceiling": achieved / (689.0 if n_gpus == 2 else 618.0)}

    # everything below runs on rank 0 as ONE controller process driving all N GPUs through the public API (the product's
    # launch mode); the other torchrun ranks release their arenas and wait on a CPU barrier
    e2e = small = c5 = c4 = c1 = None
    if world > 1:
        torch.cuda.synchronize()
    if rank == 0:
        double = kt.mapped("scale", alpha=2.0)(_clone(cases.double))

        # ---- real-peer parity through the PUBLIC API (single controller), both transfer modes + kt.put/get -----------
        def api_parity():
            rep = {"cases": 0}
            if n_gpus == 1:
                return rep
            fns = {"identity": kt.mapped("identity")(_clone(cases.identity)),
                   "scale": kt.mapped("scale", alpha="alpha")(_clone(cases.scale)),
                   "affine": kt.mapped("affine", alpha="alpha", beta="beta")(_clone(cases.affine))}
            for transfer in ("pull", "push"):
                for op, fn in fns.items():
                    remote = kt.fn(fn, name=f"bench-parity-{op}-{transfer}").to(
                        kt.Compute(gpus=n_gpus).distribute("b200", workers=1, num_proc=n_gpus, placement="ranks",
                                                           transfer=transfer))
                    try:
                        for i, (name, dtn, shape, cop, a, b, off) in enumerate(PARITY_CASES):
                            if cop != op:
                                continue
                            xin = _parity_input(dtn, shape, 100 + i)
                            extra = () if op == "identity" else ((a,) if op == "scale" else (a, b))
                            for resident in ("device", "host", "noncontiguous"):
                                if resident == "noncontiguous":
                                    if xin.dim() != 2:
                                        continue
                                    arg = xin.t().contiguous().t().cuda(0)
                                else:
                                    arg = xin.cuda(0) if resident == "device" else xin
                                got = remote(arg, *extra, serialization="pickle")
                                for d in range(n_gpus):
                                    torch.cuda.synchronize(d)
                                got = torch.cat([g.reshape(-1).cpu() for g in got])
                                want = _oracle_result(xin, op, a, b, n_gpus).reshape(-1)
                                if got.dtype != want.dtype or not torch.equal(got.view(torch.uint8), want.view(torch.uint8)):
                                    raise SystemExit(f"API PARITY FAILURE over real peers: {name} {transfer} {resident} N={n_gpus}")
                                rep["cases"] += 1
                    finally:
                        remote.teardown()
            # kt.put on cuda:0 -> kt.get on every other GPU, and a packed BroadcastWindow of a state dict
            src = torch.arange(1 << 16, dtype=torch.float32, device="cuda:0") * 0.5
            kt.put(key="bench/t", src=src)
            for d in range(1, n_gpus):
                dest = torch.zeros(1 << 16, device=f"cuda:{d}")
                kt.get(key="bench/t", dest=dest)
                torch.cuda.synchronize(d)
                if not torch.equal(dest.cpu(), src.cpu()):
                    raise SystemExit(f"kt.put/get PARITY FAILURE cuda:0 -> cuda:{d}")
                rep["cases"] += 1
            kt.rm("bench/t")
            sd = {"w": torch.randn(257, 33, device="cuda:0"), "b": torch.arange(33, device="cuda:0"),
                  "h": torch.randn(5, 7, device="cuda:0").bfloat16()}
            bw = kt.BroadcastWindow(world_size=n_gpus, timeout=60.0, group_id="bench-sd", pack=True)
            errs = []

            def getter(d):
                try:
                    with torch.cuda.device(d):
                        dest = {k: torch.zeros_like(v, device=f"cuda:{d}") for k, v in sd.items()}
                        kt.get(key="bench/sd", dest=dest, broadcast=bw)
                        torch.cuda.synchronize(d)
                        for k in sd:
                            assert torch.equal(dest[k].cpu(), sd[k].cpu()), k
                except BaseException as e:  # noqa: BLE001
                    errs.append(f"cuda:{d}: {type(e).__name__}: {e}")

            ths = [threading.Thread(target=getter, args=(d,)) for d in range(1, n_gpus)]
            [t.start() for t in ths]
            kt.put(key="bench/sd", src=sd, broadcast=bw)
            [t.join(timeout=120) for t in ths]
            if errs:
                raise SystemExit("BroadcastWindow PARITY FAILURE: " + "; ".join(errs)[:500])
            rep["cases"] += n_gpus - 1
            rep["store"] = "kt.put cuda:0 -> kt.get cuda:k and a packed BroadcastWindow state dict: bit-equal"
            return rep

        api_rep = api_parity()
        parity["public_api_cases"] = api_rep["cases"]
        if "store" in api_rep:
            parity["store"] = api_rep["store"]

        # ---- e2e: public API, host buffers ---------------------------------------------------------------------------
        remote = kt.fn(double, name="bench-double").to(
            kt.Compute(gpus=n_gpus).distribute("b200", workers=1, num_proc=n_gpus))
        # the caller's pinned buffer, allocated through the framework's NUMA-aware allocator (kt.pinned_empty): shard r's
        # pages live on GPU r's socket.  The result buffer is allocated per call by the framework the same way.
        xh = kt.pinned_empty((N_ELEMS,), torch.float32, module=remote)
        xh.normal_()
        e2e_steps = max(3, min(K, 10))
        for _ in range(3):
            out = remote(xh, serialization="pickle")
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            out = remote(xh, serialization="pickle")
        dt = (time.perf_counter() - t0) / e2e_steps
        cat = torch.cat(out)
        assert torch.equal(cat[:4096], xh[:4096] * 2) and torch.equal(out[-1][-4096:], xh[-4096:] * 2)
        idx = torch.randint(0, N_ELEMS, (65536,))
        assert torch.equal(cat[idx], xh[idx] * 2)
        e2e = {"value": 2 * nbytes / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": nbytes,
               "d2h_bytes_per_step": nbytes, "ms_per_step": dt * 1e3, "steps": e2e_steps,
               "path": "kt.fn(mapped).to(kt.Compute(gpus=N)) -> remote(pinned host tensor): per-rank chunked "
                       "H2D/kernel/D2H over each GPU's own PCIe link from per-GPU issue threads, NUMA-sharded pinned "
                       "buffers, host-clock timed"}
        del cat, out
        remote.teardown()

        # ---- calls/sec and the C5 sweep points through the public API (device-resident identity) ------------------------
        def api_rate(remote_fn, arg, n_calls):
            for _ in range(min(200, n_calls)):
                o = remote_fn(arg, serialization="pickle")
            for d in range(n_gpus):
                torch.cuda.synchronize(d)
            t0 = time.perf_counter()
            for _ in range(n_calls):
                o = remote_fn(arg, serialization="pickle")
            for d in range(n_gpus):
                torch.cuda.synchronize(d)
            return n_calls / (time.perf_counter() - t0), o

        def small_and_c5():
            ident = kt.mapped("identity")(_clone(cases.identity))
            r_id = kt.fn(ident, name="bench-c5").to(kt.Compute(gpus=n_gpus).distribute("b200", workers=1, num_proc=n_gpus))
            r_dbl = kt.fn(double, name="bench-small").to(kt.Compute(gpus=n_gpus).distribute("b200", workers=1, num_proc=n_gpus))
            pts = {}
            try:
                x1k = torch.randn(256, device="cuda:0")
                rate, o = api_rate(r_dbl, x1k, 20000)
                assert len(o) == n_gpus and torch.equal(torch.cat(o), x1k * 2)
                small_ = {"payload_bytes": 1024, "public_api_calls_per_sec": rate,
                          "path": "remote(x) small-call lane: one ctypes hop binds+launches on the caller's stream; under "
                                  "4 MiB every rank's shard maps on the root GPU in that one launch"}
                # device-level rates for context: one launch per call through the C-ABI, and a coalesced batch
                xs = [torch.randn(256, device="cuda:0") for _ in range(2048)]
                ys = [torch.empty_like(t) for t in xs]
                plan = ops.BatchPlan(xs, ys, "scale", 2.0)

                def dev_ms(fn, iters):
                    for _ in range(3):
                        fn()
                    torch.cuda.synchronize()
                    a, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    for _ in range(iters):
                        fn()
                    b2.record()
                    torch.cuda.synchronize()
                    return a.elapsed_time(b2) / iters

                # the same 2048 small calls through the PUBLIC API in one go: remote.map(xs) -> one segmented launch
                for _ in range(3):
                    outs = r_dbl.map(xs, serialization="pickle")
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(10):
                    outs = r_dbl.map(xs, serialization="pickle")
                torch.cuda.synchronize()
                small_["public_api_map_calls_per_sec"] = 10 * len(xs) / (time.perf_counter() - t0)
                assert len(outs) == len(xs) and torch.equal(torch.cat(outs[5]), xs[5] * 2)
                small_["one_launch_per_call_calls_per_sec"] = 1e3 / dev_ms(
                    lambda: ops.map_tensor(xs[0], "scale", 2.0, out=ys[0]), 2000)
                small_["coalesced_batch_calls_per_sec"] = 2048 * 1e3 / dev_ms(plan.run, 20)
                small_["device_timed"] = True
                for label, nb_, calls in (("1KiB", 1 << 10, 20000), ("1MiB", 1 << 20, 5000), ("1GiB", 1 << 30, 20)):
                    xb = torch.empty(nb_, dtype=torch.uint8, device="cuda:0").random_(0, 256)
                    rate, o = api_rate(r_id, xb, calls)
                    assert sum(t.numel() for t in o) == nb_ and torch.equal(o[-1][-64:], xb[-64:])
                    pts[label] = {"calls_per_sec": rate, "arg_plus_result_gbps": 2 * nb_ * rate / 1e9}
                    del xb, o
                return small_, {"workload": "configs[4]: identity over uint8 tensors through the public API, device-"
                                            "resident on GPU 0, rank-ordered shard views returned", "points": pts}
            finally:
                r_id.teardown()
                r_dbl.teardown()

        sc = _timeboxed(small_and_c5, "small")
        if isinstance(sc, tuple):
            small, c5 = sc
        else:
            small = c5 = sc

        # ---- configs[3]: RL rollout, 4096 env-state shards through the bf16 policy MLP over N GPUs -----------------------
        def c4_rollout():
            shards, rows = 4096, 512
            M = shards * rows
            g = torch.Generator(device="cuda:0").manual_seed(0)
            obs = torch.randn(M, 256, device="cuda:0", generator=g).bfloat16()
            w1 = (torch.randn(1024, 256, device="cuda:0", generator=g) * 0.02).bfloat16()
            w2 = (torch.randn(1024, 1024, device="cuda:0", generator=g) * 0.02).bfloat16()
            w3 = (torch.randn(64, 1024, device="cuda:0", generator=g) * 0.02).bfloat16()
            policy = kt.mapped("mlp")(_clone(cases.mlp_policy))
            r = kt.fn(policy, name="bench-c4").to(kt.Compute(gpus=n_gpus).distribute("b200", workers=1, num_proc=n_gpus))
            try:
                for _ in range(3):
                    out = r(obs, w1, w2, w3, serialization="pickle")
                for d in range(n_gpus):
                    torch.cuda.synchronize(d)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                iters = 8
                e0.record()
                for _ in range(iters):
                    out = r(obs, w1, w2, w3, serialization="pickle")
                e1.record()
                for d in range(n_gpus):
                    torch.cuda.synchronize(d)
                ms = e0.elapsed_time(e1) / iters
                # the MLP is tensor-heavy enough to run into the board power cap: sample the SM clock under ~0.5 s of the
                # same calls (the timed region itself is shorter than one nvidia-smi sample)
                sampler = ClockSampler(0)
                sampler.start()
                time.sleep(0.12)
                tc0 = time.time()
                while time.time() - tc0 < 0.5:
                    for _ in range(4):
                        out = r(obs, w1, w2, w3, serialization="pickle")
                    for d in range(n_gpus):
                        torch.cuda.synchronize(d)
                c4_clocks = sampler.stop(tc0, time.time())
                logits = torch.cat(out)
                idx = torch.randint(0, M, (2048,), device="cuda:0")
                h = torch.relu(obs[idx].float() @ w1.float().t()).bfloat16()
                h = torch.relu(h.float() @ w2.float().t()).bfloat16()
                ref = (h.float() @ w3.float().t()).bfloat16()
                torch.testing.assert_close(logits[idx].float(), ref.float(), rtol=2 ** -7, atol=1e-2)
                flop = 2 * (256 * 1024 + 1024 * 1024 + 1024 * 64) * M
                nb_ = M * 256 * 2 + M * 64 * 2
                return {"workload": "configs[3]: 4096 env-state shards (512 x 256 bf16) through the bf16 policy MLP "
                                    "256->1024->1024->64 on tcgen05, obs resident on GPU 0, scatter/gather over N GPUs",
                        "ms_per_call": ms, "calls_per_sec": 1e3 / ms, "tflops": flop / ms / 1e9,
                        "arg_plus_result_gbps": nb_ / ms / 1e6,
                        "root_nvlink_egress_gbps": (n_gpus - 1) / n_gpus * (M * 256 * 2) / ms / 1e6 if n_gpus > 1 else 0.0,
                        "clocks_under_load": c4_clocks,
                        "parity": "2048 sampled rows vs an fp32 evaluation, rtol 2^-7 atol 1e-2: ok"}
            finally:
                r.teardown()
                del obs

        c4 = _timeboxed(c4_rollout, "c4")
        torch.cuda.empty_cache()

        # ---- configs[0]: hello_world via kt.fn/.to on kt.Compute(cpus='.1'), local in-process backend (plumbing, no GPU) ---
        def c1_hello():
            r = kt.fn(cases.hello_world, name="bench-hello").to(kt.Compute(cpus=".1"))
            try:
                assert r() == "Hello from Kubetorch!"
                for _ in range(2000):
                    r()
                t0 = time.perf_counter()
                for _ in range(20000):
                    r()
                return {"workload": "configs[0]: hello_world single remote call, kt.Compute(cpus='.1'), in-process backend",
                        "calls_per_sec": 20000 / (time.perf_counter() - t0)}
            finally:
                r.teardown()

        c1 = _timeboxed(c1_hello, "c1")

    if world > 1:
        dist.barrier(group=cpu_group)  # other ranks wait on the CPU while rank 0 drives all N GPUs

    # ---- configs[2]: DDP ResNet-50 step through the kt launcher, beside plain DDP on the bench's own ranks -----------------
    c3 = None
    if not args.no_c3:
        c3 = _c3_ddp(args, world, rank, n_gpus, cpu_group)

    # ---- CPU baseline (N=1 only), bounded sample: the unmodified reference runtime when it travelled with the repo ----------
    cpu = None
    if rank == 0 and n_gpus == 1 and not args.no_cpu_baseline:
        def cpu_leg():
            if have_reference():
                r = _summarise(time_reference_runtime("testclient", 4, 2, 1, REF_SAMPLE_ELEMS, timeout=600))
                kind = "reference"
            else:
                r = _summarise(time_port(4, 1, 1, REF_SAMPLE_ELEMS))
                kind = "port"
            return {"value": r["value"], "unit": UNIT, "cores": os.cpu_count() or 1, "kind": kind, "sample": r["sample"],
                    "calls_per_sec": r["calls_per_sec"], "ranks": 1}

        cpu = _timeboxed(cpu_leg, "cpu")

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "calls_per_sec": 1e3 / ms_per_step,
            "config": workload_config(n_gpus),
            "launch": {
                "residency": "args/results resident on GPU 0",
                "mode": "single controller" if world == 1 else "one process per GPU, CUDA-IPC peer arenas, calls "
                        "pipelined per rank",
                "transfer": best_mode, "ms_per_step_by_transfer": modes, "two_calls_in_flight": two_in_flight,
                "single_stream_ms_per_step": min(v for k, v in modes.items() if not k.endswith("two_calls_in_flight")),
                "l2": "inputs+outputs (512 MiB) exceed the 126 MB L2; no flush needed",
            },
            "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks, "parity": parity,
            "c1_hello_world": c1, "small_calls": small, "c5": c5, "c4_rollout": c4, "c3_ddp": c3,
            "gpu_launches": gpu_launches,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _c3_ddp(args, world, rank, n_gpus, cpu_group):
    """BASELINE configs[2]: `steps` DDP ResNet-50 steps (synthetic 224x224 batches, bf16 autocast, channels_last,
    batch 256 per GPU).  (a) plain DDP on the bench's own ranks (under torchrun: the torchrun world; at N=1: a
    one-rank group), (b) the same function launched through kt.Compute(gpus=N).distribute("pytorch", num_proc=N)."""
    import torch
    import torch.distributed as dist

    sys.path.insert(0, os.path.join(REPO, "tools"))
    import ddp_resnet50

    steps, warm, batch = 20, 5, 256
    out = {"workload": "configs[2]: torch DDP ResNet-50, synthetic 224x224, bf16 autocast, channels_last, batch 256/GPU, "
                       f"{steps} timed steps"}
    t_sec = time.perf_counter()
    try:
        own_group = False
        if world == 1:
            if n_gpus > 1:
                plain = None   # a single controller cannot be N DDP ranks; the launcher below is the N-rank job
            else:
                os.environ["LOCAL_RANK"] = "0"
                dist.init_process_group("nccl", init_method="tcp://127.0.0.1:29611", rank=0, world_size=1,
                                        device_id=torch.device("cuda:0"))
                own_group = True
                plain = ddp_resnet50.train_resnet50(steps, warm, batch)
        else:
            plain = ddp_resnet50.train_resnet50(steps, warm, batch)
        if plain is not None:
            t = torch.tensor([plain["images_per_sec"]], device="cuda")
            if world > 1:
                dist.all_reduce(t)
            out["plain_ddp_images_per_sec"] = float(t.item())
        if own_group:
            dist.destroy_process_group()
        torch.cuda.empty_cache()
    except Exception as e:  # noqa: BLE001
        out["plain_ddp_error"] = f"{type(e).__name__}: {e}"[:300]
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier(group=cpu_group)
    if rank == 0:
        try:
            import math

            import kubetorch_b200 as kt

            saved = {k: os.environ.pop(k) for k in list(os.environ)
                     if k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "LOCAL_WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT",
                              "GROUP_RANK", "ROLE_RANK") or k.startswith("TORCHELASTIC")}
            try:
                t0 = time.perf_counter()
                remote = kt.fn(ddp_resnet50.train_resnet50, name="bench-ddp-resnet50").to(
                    kt.Compute(gpus=n_gpus, launch_timeout=600).distribute("pytorch", workers=1, num_proc=n_gpus, port=29577))
                t_launch = time.perf_counter() - t0
                try:
                    results = remote(steps, warm, batch)
                finally:
                    remote.teardown()
            finally:
                os.environ.update(saved)
            assert [r["rank"] for r in results] == list(range(n_gpus))
            assert all(math.isfinite(r["loss"]) for r in results)
            assert len({round(r["param_checksum"], 3) for r in results}) == 1, "DDP replicas diverged"
            out["kt_launcher_images_per_sec"] = sum(r["images_per_sec"] for r in results)
            out["launch_seconds"] = t_launch
            out["replica_param_checksums_equal"] = True
            out["loss"] = results[0]["loss"]
        except Exception as e:  # noqa: BLE001
            out["kt_launcher_error"] = f"{type(e).__name__}: {e}"[:300]
    if world > 1:
        dist.barrier(group=cpu_group)
    out["section_seconds"] = round(time.perf_counter() - t_sec, 1)
    return out


def _traffic(n_gpus: int) -> dict:
    """DRAM (N=1) / NVLink (N>1) bytes per launch of the dominant kernel from the committed ncu capture — valid only
    while the kernel source is the one that was profiled (sha256 of ktb_map.cu + ktb_common.cuh stamped in the file)."""
    import hashlib

    try:
        with open(os.path.join(REPO, "profiles", "roofline_traffic.json")) as f:
            rec = json.load(f)
        from kubetorch_b200.device import lib as _L

        if rec.get("kernel_source_sha256") != _L.map_kernel_source_sha256():
            return {"bytes": None, "source": "stale: kernel source changed since the ncu capture in profiles/roofline_traffic.json"}
        if n_gpus == 1:
            return {"bytes": rec.get("dram_bytes_per_launch"), "source": rec.get("source")}
        nv = rec.get("nvlink") or {}
        if not nv:
            return {"bytes": None, "source": "no NVLink capture"}
        # bytes on the wire through the root's port per call, both directions: user bytes x the measured wire/user ratio
        # of the push kernels (N=2 capture; the ratio is a property of the 128-byte write packets, not of N)
        shard = -(-N_ELEMS // n_gpus) * 4
        user = (n_gpus - 1) * shard
        return {"bytes": int(2 * user * nv["wire_per_user"]),
                "source": nv["source"] + f"; scaled to N={n_gpus}: 2 directions x {user} user bytes x {nv['wire_per_user']:.4f}"}
    except Exception as e:  # noqa: BLE001
        return {"bytes": None, "source": f"unavailable: {type(e).__name__}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps (remote calls) of the headline measurement")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c3", action="store_true")
    ap.add_argument("--push-chunks", type=int, default=32, help="chunks per shard of the push/push flag pipeline")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a sample of the last timed step's result to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
