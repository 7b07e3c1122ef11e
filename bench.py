#!/usr/bin/env python
"""bench.py — MIG placement decisions/s of the B200 placement engine on the BASELINE configurations.

    python bench.py [--config c4] [--gpus N] [--steps K] [--warmup W] [--impl reference] [--min-age A] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR (configs c1-c4): after the timed steps, what the headline path computed in its last timed step, as float64 .npy
files: result_gpu / result_start / result_size / result_status (one entry per request, in request order) and occupancy (the final
occupancy byte of every GPU).  The workloads are seeded, so two builds of the project run with the same arguments can be compared
output for output.  c5 is not supported: how its requests are grouped into calls depends on the host clock.

--config (default c4, the configuration BASELINE.json's metric is quoted on; the others make every BASELINE config
driver-reachable with the same parity / cpu_baseline / roofline / e2e keys):
  c1    samples/test-pod.yaml: one 1g.5gb request on one emulated A100-40GB GPU           (isl_place_batch, the k_few path)
  c2    10 000 x 1g.10gb on 256 GPUs, first-fit                                            (one batch; scan-mode commit)
  c3    100 000 mixed-profile pods on 4 096 GPUs, first-fit (REF_EXACT parity)             (one batch; segment pipeline)
  c3bf  the same input, ISL_POLICY_BEST_FIT (extension, parity against the oracle's best-fit)
  c4    1M operations x 65 536 GPUs, 50/50 alloc/free churn, 16 batches                    (stream of batches; N > 1: partitioned)
  c5    vLLM-shaped replay (3g.20gb) at 10 000 req/s for 10 s on 4 096 GPUs — p50 / p99 submit -> result latency (native driver)

One "step" = one pass of the hot path over the whole workload of the config, starting from the same inventory (the reset of the
occupancy bytes is a 64 KiB device copy inside the timed region).

c4 in detail.  In the churn workload a FREE names an allocation an EARLIER batch placed, so a live caller cannot compose batch b
before it has seen the results of batch b - 1.  The headline therefore is STRICT CAUSAL (--min-age 1, the default): the original
config-4 stream with ONE batch in flight — every batch is resolved before the next one starts, exactly what the reconciler's per-pod
call sequence (instaslice_controller.go:192) implies.
  value         ALLOC decisions/s, requests and results resident in HBM; one device-side stream call with isl_set_causal_window(1):
                batch b does not start before every inventory stage has committed batch b - 1.  A batch's decisions are one exact
                recurrence over the inventory; the stages resolve it by speculative rounds (DESIGN.md 4.5)
  e2e           one synchronous isl_place_batch per batch with HOST buffers (H2D and D2H inside every call) — the call SURVEY 8d
                defines the metric on; e2e.open_stream_value: the same through isl_stream_open / _submit / _wait / _close
  causal_feed   the variant whose FREEs name allocations at least 2 batches old (Churn(min_age=2)) with TWO batches in flight
                (--min-age 2 makes it the headline).  At config 4's own churn rate the whole live set turns over every ~3.4 batches:
                depths beyond 3 are not sustainable
  replay_*      the original stream handed over in one call (all 16 batches up front) — the pipelining ceiling, not causally available
Every mode is checked byte for byte against the CPU oracle (ref_fast): results of every batch and the final occupancy.
N > 1: the inventory is partitioned over the ranks (contiguous GPU ranges); the stages of all ranks form one sequence and exchange the
per-round records of the speculative rounds through peer memory (stores into the other ranks' record memory over NVLink, inside the
running kernels); the PLACED records go straight into rank 0's result array (peer stores from the commit threads — no result
collective); the causal window is enforced across ranks by a per-chunk counter on rank 0 (peer atomics); the occupancy shards are
all-gathered with NCCL.  Strong scaling (the job is fixed).

The CPU oracle is used only for the parity gate, the cpu_baseline leg and --impl reference.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "placements_per_sec"
UNIT = "placements/s"
WORKLOADS = {
    "c1": "C1: samples/test-pod.yaml, one 1g.5gb request on 1 node x 1 empty A100-40GB GPU",
    "c2": "C2: 10000 x 1g.10gb on 32 nodes x 8 GPUs (256), H100-80GB table, first-fit",
    "c3": "C3: 100000 mixed-profile pods (1g 40 / 2g 25 / 3g 20 / 4g 10 / 7g 5 %) on 512 nodes x 8 GPUs (4096), first-fit, seed 42",
    "c3bf": "C3: 100000 mixed-profile pods on 4096 GPUs, best-fit with fragmentation score (extension), seed 42",
    "c4": "C4: 8192 nodes x 8 GPUs (65536), H100-80GB table, prefill 50%, 1e6 ops, 50/50 alloc/free, batches of 65536, seed 42",
    "c5": "C5: vLLM-shaped replay, Poisson 10000 req/s, 100% 3g.20gb, A100-40GB tables, 4096 GPUs, exp(30 s) lifetimes",
}


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(kernel="k_pipeline"):
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if one has been summarised."""
    try:
        with open(os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")) as f:
            d = json.load(f)
        return d.get("dram_bytes_per_launch") if d.get("kernel", "k_pipeline").startswith(kernel) else None
    except Exception:
        return None


def _device_view(torch, ptr: int, n: int, typestr="|u1"):
    """torch view of engine-owned device memory (no copy)."""
    class _Holder:
        pass
    h = _Holder()
    h.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3}
    return torch.as_tensor(h, device="cuda")


class Ctx:
    """What every config needs: torch, ranks, a timing helper, the clock sampler."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.rank, self.world, self.local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
        # NCCL's own log shows the communicator (ranks, NVLS / P2P): NCCL_DEBUG=INFO unless the caller asked for something else.  NCCL writes
        # to the process's stdout, which must end with rank 0's JSON line: file descriptor 1 points at stderr while the process group lives
        # (so the log lands on stderr, whole), the real stdout is restored for the one JSON line at the very end
        self.real_stdout = None
        if self.world > 1:
            if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
                os.environ["NCCL_DEBUG"] = "INFO"
            os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
            os.environ.pop("NCCL_DEBUG_FILE", None)
            sys.stdout.flush()
            self.real_stdout = os.dup(1)
            os.dup2(2, 1)
        if self.world != args.gpus and self.world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with torch.distributed.run (one rank per GPU)")
        torch.cuda.set_device(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        import __graft_entry__ as g
        if self.rank == 0:
            g.build()
        if self.world > 1:
            dist.barrier()
        self.stream = torch.cuda.Stream()           # a real (non-default) stream: the legacy default stream has handle 0
        torch.cuda.set_stream(self.stream)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")     # > 126 MB L2

    def timed(self, step_fn, steps, warmup, flush_l2=True):
        """W untimed steps, then K steps, each bracketed by CUDA events on the stream the engine launches on; barrier + synchronize on
        both sides; returns (total ms = MAX over ranks, wall seconds of this rank)."""
        torch, dist = self.torch, self.dist
        for _ in range(warmup):
            step_fn()
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        total_ms, wall = 0.0, 0.0
        for _ in range(steps):
            if flush_l2:
                self.flush.fill_(1)
                torch.cuda.synchronize()        # the host clock below must not see the flush
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            step_fn()
            e1.record()
            e1.synchronize()
            wall += time.perf_counter() - t0
            total_ms += e0.elapsed_time(e1)
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
            t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total_ms = float(t.item())
        return total_ms, wall


def dump_outputs(out_dir, results, occupancy):
    """--dump-outputs: every field of the result records and the final occupancy, as float64 (exact for every u8 / u16 / u32 value)."""
    arrays = {"result_" + f: results[f] for f in results.dtype.names}
    arrays["occupancy"] = occupancy
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > 64 << 20:
        raise SystemExit("--dump-outputs: %d bytes exceed the 64 MiB budget" % total)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def base_line(ctx, config, value, ms_per_step, config_extra, parity, launches, clocks, scaling="strong"):
    a = ctx.args
    cfg = {"workload": WORKLOADS[config], "l2": "flushed between timed steps (256 MiB write)", "timing": "cuda events per step on the launching stream, max over ranks",
           "quirks": "REF_EXACT"}
    cfg.update(config_extra)
    return {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ctx.world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": cfg,
            "parity": "bit-exact vs the CPU oracle (ref_fast): every result record and the final occupancy" if parity else "MISMATCH vs the CPU oracle",
            "gpu_launches": int(launches), "clocks": clocks}


# ---- CPU legs (the only places that execute oracle/) ----------------------------------------------------------------------
def fast_replay(oracle, node_off, rows, occ0, batches, policy=0, reps=5):
    """ref_fast on the whole job, best of `reps` (one core).  Returns (results per batch, final occupancy, best seconds)."""
    best, res, occ = 1e30, None, None
    for _ in range(reps):
        f = oracle.Fast(node_off, rows, 3, policy=policy)
        f.load(occ0)
        t0 = time.perf_counter()
        r = [f.place(b) for b in batches]
        dt = time.perf_counter() - t0
        if dt < best:
            best = dt
        res, occ = r, f.occupancy()
    return res, occ, best


def faithful_from_prefill(oracle, node_off, rows, prefill):
    """The reference's CR state that corresponds to a pre-filled inventory: one Allocations entry per pre-fill placement."""
    f = oracle.Faithful(node_off, rows)
    pod = 0
    for req, res in prefill:
        placed = (req["op"] == 0) & (res["status"] == 0)
        for g, s, z in zip(res["gpu"][placed].tolist(), res["start"][placed].tolist(), res["size"][placed].tolist()):
            f.add_allocation(g, s, z, pod)
            pod += 1
    return f


def cpu_baseline_batches(node_off, rows, occ0, batches, got, got_occ, policy=0, faithful=None, faithful_ops=None, faithful_note=""):
    """ref_fast on the whole job (best of 5) + parity verdicts; ref_faithful (the reference as written, one reconcile worker) on a
    bounded prefix when `faithful` (a prepared Faithful state) is given."""
    import oracle
    from instaslice_b200 import engine as E
    want, want_occ, t_fast = fast_replay(oracle, node_off, rows, occ0, batches, policy)
    ok = all(np.array_equal(a, b) for a, b in zip(got, want)) and (got_occ is None or np.array_equal(got_occ, want_occ))
    n_ops = sum(len(b) for b in batches)
    n_alloc = int(sum(int((b["op"] == E.OP_ALLOC).sum()) for b in batches))
    out = {"cores": 1, "kind": "port", "unit": UNIT,
           "ref_fast_value": n_alloc / t_fast, "ref_fast_ops_per_sec": n_ops / t_fast, "ref_fast_ms": t_fast * 1e3,
           "ref_fast_note": "bitmask restatement (oracle/ref_fast.cpp), whole job, 1 core, best of 5 — the strong CPU baseline",
           "parity_full_job_vs_ref_fast": bool(ok)}
    if faithful is not None:
        req = np.concatenate(batches)[:faithful_ops] if faithful_ops else np.concatenate(batches)
        # batch boundaries matter (FREEs first inside a batch): the prefix is cut inside batch 0 or spans whole batches
        pieces, off = [], 0
        for b in batches:
            if off >= len(req):
                break
            pieces.append(b[: len(req) - off])
            off += len(pieces[-1])
        t0 = time.perf_counter()
        fres = [faithful.place(p) for p in pieces]
        dt = time.perf_counter() - t0
        n_a = int(sum(int((p["op"] == E.OP_ALLOC).sum()) for p in pieces))
        # a prefix cut inside a batch is a batch of its own (only ITS FREEs are applied first): the checker replays the same pieces
        fcheck = oracle.Fast(node_off, rows, 3, policy=policy)
        fcheck.load(occ0)
        ok_f = all(np.array_equal(a, fcheck.place(p)) for a, p in zip(fres, pieces))
        out.update({"value": n_a / dt, "sample": "ref_faithful.cpp (the reference as written: string-keyed CRs, rescans per pod; 1 reconcile worker) on %s: %d ops = %d ALLOC decisions, %.1f s"
                                                  % (faithful_note, len(req), n_a, dt),
                    "parity_sample_faithful_vs_fast": bool(ok_f)})
        ok = ok and ok_f
    else:
        out.update({"value": n_alloc / t_fast, "sample": "ref_fast.cpp on the whole job (no reference-as-written counterpart for this policy)"})
    return out, bool(ok)


# ---- configs 1-3: one batch ------------------------------------------------------------------------------------------------
def run_single_batch(ctx, config):
    torch = ctx.torch
    from instaslice_b200 import engine as E
    from instaslice_b200 import workloads as W
    a = ctx.args
    policy = E.POLICY_BEST_FIT if config == "c3bf" else E.POLICY_FIRST_FIT
    node_off, occ0, rows, req = {"c1": W.config1, "c2": W.config2, "c3": W.config3, "c3bf": W.config3}[config]()
    G, n = len(occ0), len(req)
    eng = E.Engine(max_gpus=max(4096, G), max_batch=1 << 20, policy=policy)
    eng.set_stream(ctx.stream.cuda_stream)
    eng.load_profiles(rows)
    eng.load_inventory(node_off, occ0)
    d_occ0 = torch.from_numpy(occ0).cuda()
    occ_view = _device_view(torch, eng.device_occupancy(), G)
    d_in = torch.from_numpy(req.view(np.int64).copy()).cuda()
    d_out = torch.empty_like(d_in)
    h_in = torch.from_numpy(req.view(np.int64).copy()).pin_memory()
    h_out = torch.empty_like(h_in).pin_memory()

    eng.snapshot_occupancy()            # the reset of a step = isl_restore_occupancy: one async device copy on the engine's stream

    def step_device():
        eng.restore_occupancy()
        eng.place_batch_device(n, d_in.data_ptr(), d_out.data_ptr())

    def step_e2e():         # the call the reconciler makes: host buffers in, host buffers out, synchronous
        eng.restore_occupancy()
        eng.place_batch_ptr(n, h_in.data_ptr(), h_out.data_ptr())

    sampler = ClockSampler(ctx.local)
    if ctx.rank == 0:
        sampler.start()
    launches0 = eng.stats()["kernel_launches"]
    ms_dev, _ = ctx.timed(step_device, a.steps, a.warmup)
    launches = eng.stats()["kernel_launches"] - launches0
    got_dev = d_out.cpu().numpy().view(E.RESULT_DTYPE)
    occ_dev = eng.read_occupancy()
    ms_e2e, wall_e2e = ctx.timed(step_e2e, a.steps, a.warmup)
    clocks = sampler.stop() if ctx.rank == 0 else None
    got_e2e = h_out.numpy().view(E.RESULT_DTYPE).copy()
    n_alloc = int((req["op"] == E.OP_ALLOC).sum())

    # dominant kernel, timed live with CUDA events on the engine's own stream (timing mode)
    teng = E.Engine(max_gpus=max(4096, G), max_batch=1 << 20, policy=policy, timing=True)
    teng.load_profiles(rows)
    for _ in range(3):
        teng.load_inventory(node_off, occ0)
        teng.reset_stats()
        teng.place_batch_device(n, d_in.data_ptr(), d_out.data_ptr())
        teng.synchronize()
    st = teng.stats()
    teng.close()
    phases = {"prepare": st["ms_free"], "partition": st["ms_partition"], "sweep": st["ms_sweep"], "commit": st["ms_commit"], "total": st["ms_total"]}
    dom_name, dom_ms = max(((k, v) for k, v in phases.items() if k != "total"), key=lambda kv: kv[1])
    kernel = {"c1": "k_few", "c2": "k_sweep_scatter (scan-mode commit)", "c3": "k_pipeline", "c3bf": "k_bestfit"}[config]
    alg_bytes = 16 * n + 2 * G
    peak, how = measured_peak()
    achieved = alg_bytes / (max(dom_ms, 1e-6) / 1e3) / 1e9
    roofline = {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                "peak_source": how, "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": dom_ms, "dominant_phase": dom_name, "phase_ms_per_step": phases,
                "note": "integer / bitmask work; the inventory (%d B) is on-chip, the request / result arrays stream once; the exact commit is a sequential "
                        "recurrence over placements and bounds the step, not HBM" % G}
    parity, cpu = True, None
    if ctx.rank == 0:
        import oracle
        faithful = faithful_ops = None
        note = ""
        if policy == E.POLICY_FIRST_FIT:
            faithful = oracle.Faithful(node_off, rows)
            faithful.load_occupancy_as_dangling(occ0)
            faithful_ops = {"c1": None, "c2": None, "c3": 20000}[config]
            note = "the whole job" if faithful_ops is None else "the first %d requests of the job" % faithful_ops
        cpu, parity = cpu_baseline_batches(node_off, rows, occ0, [req], [got_dev], occ_dev, policy, faithful, faithful_ops, note)
        parity = parity and np.array_equal(got_e2e, got_dev)
    value = n_alloc * a.steps / (ms_dev / 1e3)
    e2e_ms = max(ms_e2e, wall_e2e * 1e3)
    line = base_line(ctx, config, value * ctx.world, ms_dev / a.steps,
                     {"requests_per_step": n, "gpus_in_inventory": G, "policy": "best-fit" if policy else "first-fit",
                      "parallelism": "1 GPU" if ctx.world == 1 else "%d independent replicas (a single batch does not shard: replicas only)" % ctx.world,
                      "ops_counted": "ALLOC decisions (placed or definitively no-capacity)"}, parity, launches, clocks,
                     scaling="strong" if ctx.world == 1 else "weak")
    line["e2e"] = {"value": n_alloc * a.steps / (e2e_ms / 1e3) * ctx.world, "unit": UNIT, "h2d_bytes_per_step": 8 * n, "d2h_bytes_per_step": 8 * n,
                   "ms_per_step": e2e_ms / a.steps, "api": "isl_place_batch (host buffers, synchronous); timed by the host clock around the call and by CUDA events, the larger is reported"}
    line["roofline"] = roofline
    if cpu:
        line["cpu_baseline"] = cpu
    if a.dump_outputs and ctx.rank == 0:
        dump_outputs(a.dump_outputs, got_dev, occ_dev)
    eng.close()
    return line, parity


# ---- config 5: latency replay -----------------------------------------------------------------------------------------------
def c5_trace(W, rate, seconds, mean_life=30.0):
    rng = W.SplitMix64(42)
    n = int(rate * seconds)
    u = (rng.next(n) >> np.uint64(11)).astype(np.float64) / float(1 << 53)
    arrivals = np.cumsum(-np.log1p(-u) / rate)
    life = -np.log1p(-(rng.next(n) >> np.uint64(11)).astype(np.float64) / float(1 << 53)) * mean_life
    return n, np.ascontiguousarray(arrivals), np.ascontiguousarray(life)


def c5_replay(place_fn_addr, ctx_handle, n, arrivals, life, profile):
    """instaslice_b200/host/replay_driver.cpp: the native open-loop driver (no Python between the clock and the call)."""
    from instaslice_b200 import engine as E
    host = C.CDLL(os.path.join(ROOT, "instaslice_b200", "libislhost.so"))
    fn = host.islh_replay_open_loop
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint8, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                   C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_double), C.POINTER(C.c_uint32)]
    cap, cap_calls = 4 * n + 1024, 2 * n + 1024
    lat = np.zeros(n)
    rec_req, rec_res = np.zeros(cap, dtype=E.REQUEST_DTYPE), np.zeros(cap, dtype=E.RESULT_DTYPE)
    rec_sizes = np.zeros(cap_calls, dtype=np.uint32)
    n_calls, n_rec, wall, placed = C.c_uint32(), C.c_uint32(), C.c_double(), C.c_uint32()
    p = lambda x: x.ctypes.data_as(C.c_void_p)
    rc = fn(C.c_void_p(place_fn_addr), ctx_handle, n, p(arrivals), p(life), profile, p(lat), p(rec_req), p(rec_res), cap, p(rec_sizes), cap_calls,
            C.byref(n_calls), C.byref(n_rec), C.byref(wall), C.byref(placed))
    if rc != 0:
        raise RuntimeError("islh_replay_open_loop: %d" % rc)
    sizes = rec_sizes[: n_calls.value]
    return lat, rec_req[: n_rec.value], rec_res[: n_rec.value], sizes, wall.value, placed.value


def latency_summary(lat):
    us = lat * 1e6
    return {k: float(np.percentile(us, q)) for k, q in (("p50", 50), ("p90", 90), ("p99", 99), ("p999", 99.9))} | {"max": float(us.max()), "mean": float(us.mean())}


def run_c5(ctx):
    from instaslice_b200 import engine as E, tables
    from instaslice_b200 import workloads as W
    a = ctx.args
    rate, seconds, G = 10000.0, float(a.seconds), 4096
    n, arrivals, life = c5_trace(W, rate, seconds)
    rows = E.make_profiles(tables.A100_40GB)
    node_off = W.node_offsets(G // 8, 8)
    prof = tables.profile_index(tables.A100_40GB, "3g.20gb")
    eng = E.Engine(max_gpus=G, max_batch=65536)
    eng.load_profiles(rows)
    eng.load_inventory(node_off, np.zeros(G, dtype=np.uint8))
    noop = np.array([(0, E.PROFILE_UNKNOWN, E.OP_NOOP, 0, 0)], dtype=E.REQUEST_DTYPE)
    for _ in range(max(200, a.warmup)):                    # warm the path (kernels loaded, buffers allocated)
        eng.place_batch(noop)
    lib = E.load_library()
    sampler = ClockSampler(ctx.local)
    sampler.start()
    launches0 = eng.stats()["kernel_launches"]
    lat, rreq, rres, sizes, wall, placed = c5_replay(C.cast(lib.isl_place_batch, C.c_void_p).value, eng._h, n, arrivals, life, prof)
    launches = eng.stats()["kernel_launches"] - launches0
    clocks = sampler.stop()
    occ_end = eng.read_occupancy()
    eng.close()
    # parity: everything that was submitted, call by call, through the oracle
    import oracle
    f = oracle.Fast(node_off, rows)
    f.load(np.zeros(G, dtype=np.uint8))
    ok, off = True, 0
    for m in sizes.tolist():
        ok = ok and np.array_equal(f.place(rreq[off:off + m]), rres[off:off + m])
        off += m
    ok = bool(ok and np.array_equal(occ_end, f.occupancy()))
    # CPU baseline: the same trace through the same native driver with ref_fast as the placer, and with the reference as written
    ol = oracle.lib()
    f2 = oracle.Fast(node_off, rows)
    f2.load(np.zeros(G, dtype=np.uint8))
    lat_fast, *_ = c5_replay(C.cast(ol.orc_fast_place, C.c_void_p).value, f2._h, n, arrivals, life, prof)
    n_f, arr_f, life_f = c5_trace(W, rate, min(seconds, 2.0))
    ff = oracle.Faithful(node_off, rows)
    lat_faith, _, _, sz_f, wall_f, _ = c5_replay(C.cast(ol.orc_f_place_batch, C.c_void_p).value, ff._h, n_f, arr_f, life_f, prof)
    s = latency_summary(lat)
    line = {"metric": "placement_latency_p50_us", "value": s["p50"], "unit": "us", "n_gpus": 1, "steps": 1, "warmup": a.warmup, "ms_per_step": wall * 1e3,
            "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOADS["c5"], "seconds": seconds, "requests": n, "calls": int(len(sizes)), "mean_batch": float(sizes.mean()), "placed": int(placed),
                       "driver": "native open-loop replay (instaslice_b200/host/replay_driver.cpp): every turn hands isl_place_batch the expired slices and the requests that arrived since the last call",
                       "timing": "host steady_clock, arrival -> result available (a latency metric: the call is synchronous, there is nothing to bracket with CUDA events)",
                       "l2": "n/a (latency of single small calls)"},
            "latency_us": s, "parity": "bit-exact vs the CPU oracle (ref_fast): every call's results and the final occupancy" if ok else "MISMATCH vs the CPU oracle",
            "gpu_launches": int(launches), "clocks": clocks,
            "e2e": {"value": s["p50"], "unit": "us", "p99": s["p99"], "h2d_bytes_per_step": int(8 * sizes.mean()), "d2h_bytes_per_step": int(8 * sizes.mean()),
                    "api": "isl_place_batch per driver turn (requests travel as kernel parameters, results through mapped pinned memory)"},
            "roofline": {"bound": "hbm", "kernel": "k_few", "achieved": None, "peak": measured_peak()[0], "unit": "GB/s", "frac": None, "traffic": None,
                         "note": "latency path: one launch of one CTA per call, ~16 B in and out; launch + synchronisation latency bounds it, not bandwidth"},
            "cpu_baseline": {"value": latency_summary(lat_fast)["p50"], "unit": "us", "cores": 1, "kind": "port",
                             "sample": "the same trace through the same native driver with oracle/ref_fast.cpp as the placer (p50 of arrival -> result)",
                             "ref_fast_latency_us": latency_summary(lat_fast),
                             "ref_faithful_latency_us": latency_summary(lat_faith),
                             "ref_faithful_note": "the reference as written on the first %.0f s of the trace (%d requests, %d calls, wall %.2f s): it resolves ~10^4 pods/s on 4096 GPUs, "
                                                  "so an open loop at 10^4 req/s keeps it saturated" % (min(seconds, 2.0), n_f, len(sz_f), wall_f),
                             "parity_full_job_vs_ref_fast": ok}}
    return line, ok


# ---- config 4: the churn stream ---------------------------------------------------------------------------------------------
def record_churn(E, W, min_age):
    """Generate config 4 through the engine (untimed, one isl_place_batch per batch).  Returns (churn, prefilled occupancy,
    churn batches, engine results per batch, [(pre-fill requests, results)])."""
    ch = W.Churn(min_age=min_age)
    eng = E.Engine(max_gpus=ch.G, max_batch=65536)
    eng.load_profiles(ch.rows)
    eng.load_inventory(ch.node_off, np.zeros(ch.G, dtype=np.uint8))
    results, snap = [], {}

    def placer(req):
        res = eng.place_batch(req)
        results.append(res)
        return res

    ch.generate(placer, after_prefill=lambda: snap.update(occ=eng.read_occupancy()))
    eng.close()
    nb = ch.n_prefill_batches
    return ch, snap["occ"], ch.batches[nb:], results[nb:], list(zip(ch.batches[:nb], results[:nb]))


def run_c4(ctx):
    torch, dist = ctx.torch, ctx.dist
    from instaslice_b200 import engine as E
    from instaslice_b200 import workloads as W
    a = ctx.args
    A = max(1, a.min_age)
    rank, world = ctx.rank, ctx.world
    ch, occ0, batches, rec, prefill = record_churn(E, W, A)
    nb, G = len(batches), ch.G
    sizes = np.array([len(b) for b in batches], dtype=np.uint32)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    n_ops = int(offs[-1])
    n_alloc = int(sum(int((b["op"] == E.OP_ALLOC).sum()) for b in batches))
    all_req = np.concatenate(batches).view(np.int64)

    eng = E.Engine(max_gpus=G, max_batch=1 << 20)
    eng.set_stream(ctx.stream.cuda_stream)
    eng.load_profiles(ch.rows)
    eng.load_inventory(ch.node_off, occ0)
    d_occ0 = torch.from_numpy(occ0).cuda()
    occ_view = _device_view(torch, eng.device_occupancy(), G)
    d_in_all = torch.from_numpy(all_req.copy()).cuda()            # the whole stream, batch after batch, resident in HBM
    d_res = _device_view(torch, eng.device_results(), n_ops, "<i8")      # the engine's own result array (rank 0: the ranks' records land here)
    h_in_all = torch.from_numpy(all_req.copy()).pin_memory()
    h_out_all = torch.zeros_like(h_in_all).pin_memory()

    def split(x):
        return [x[offs[i]:offs[i + 1]] for i in range(nb)]

    def results_of(t):
        return split(t.cpu().numpy().view(E.RESULT_DTYPE) if t.is_cuda else t.numpy().view(E.RESULT_DTYPE).copy())

    lines_extra, parity = {}, True
    sampler = ClockSampler(ctx.local)

    if world == 1:
        import oracle

        def load_variant(chv, occv, batchesv):
            reqv = np.concatenate(batchesv).view(np.int64)
            d_occ0.copy_(torch.from_numpy(occv))
            d_in_all.copy_(torch.from_numpy(reqv.copy()))
            h_in_all.copy_(torch.from_numpy(reqv.copy()))
            eng.load_inventory(chv.node_off, occv)

        def step_device():
            occ_view.copy_(d_occ0)
            eng.place_stream_ptr(sizes, d_in_all.data_ptr(), d_res.data_ptr(), device=True)

        def open_stream_step(window):
            def step():
                occ_view.copy_(d_occ0)
                try:
                    eng.set_causal_window(window)      # tells the engine how many batches this caller keeps in flight (1..3: speculative rounds)
                    eng.stream_open(nb)
                except E.EngineError:       # under ncu / compute-sanitizer (kernels serialised) an open stream cannot run: per-batch calls
                    for i in range(nb):
                        eng.place_batch_ptr(int(sizes[i]), h_in_all.data_ptr() + 8 * int(offs[i]), h_out_all.data_ptr() + 8 * int(offs[i]))
                    return
                t = []
                for b in range(nb):
                    if b >= window:
                        eng.stream_wait(t[b - window])         # the results of batch b - window are in host memory: batch b may be composed
                    t.append(eng.stream_submit_ptr(int(sizes[b]), h_in_all.data_ptr() + 8 * int(offs[b]), h_out_all.data_ptr() + 8 * int(offs[b])))
                for b in range(max(0, nb - window), nb):
                    eng.stream_wait(t[b])
                eng.stream_close()
                eng.set_causal_window(0)
            return step

        def step_per_batch():       # one synchronous isl_place_batch per batch, host buffers: the call SURVEY 8d defines the metric on
            occ_view.copy_(d_occ0)
            for i in range(nb):
                eng.place_batch_ptr(int(sizes[i]), h_in_all.data_ptr() + 8 * int(offs[i]), h_out_all.data_ptr() + 8 * int(offs[i]))

        def measure(chv, occv, batchesv, window, with_calls):
            """device stream with the causal window, open stream with `window` batches in flight, optionally per-batch calls; all checked"""
            load_variant(chv, occv, batchesv)
            want, want_occ, t_fast = fast_replay(oracle, chv.node_off, chv.rows, occv, batchesv)
            ok = lambda got, occ: all(np.array_equal(x, y) for x, y in zip(got, want)) and np.array_equal(occ, want_occ)
            n_al = int(sum(int((b["op"] == E.OP_ALLOC).sum()) for b in batchesv))
            out = {"n_alloc": n_al, "ref_fast_s": t_fast}
            eng.set_causal_window(window)
            eng.reset_stats()
            l0 = eng.stats()["kernel_launches"]
            ms, _ = ctx.timed(step_device, a.steps, a.warmup)
            st = eng.stats()
            out["launches"] = st["kernel_launches"] - l0
            out["spec"] = {"chunks": st["spec_chunks"], "rounds_per_chunk": st["spec_rounds"] / max(1, st["spec_chunks"]), "simulations_per_chunk": st["spec_sims"] / max(1, st["spec_chunks"])}
            out["got"], out["occ"] = results_of(d_res), eng.read_occupancy()
            out["dev_ms"] = ms / a.steps
            parity_ok = ok(out["got"], out["occ"])
            eng.set_causal_window(0)
            ms, wall = ctx.timed(open_stream_step(window), a.steps, a.warmup)
            out["open_ms"] = max(ms, wall * 1e3) / a.steps
            parity_ok &= ok(results_of(h_out_all), eng.read_occupancy())
            if with_calls:
                ms, wall = ctx.timed(step_per_batch, a.steps, a.warmup)
                out["calls_ms"] = max(ms, wall * 1e3) / a.steps
                parity_ok &= ok(results_of(h_out_all), eng.read_occupancy())
            out["parity"] = bool(parity_ok)
            return out

        sampler.start()
        head = measure(ch, occ0, batches, A, A == 1)
        clocks = sampler.stop()
        per = lambda m, ms: m["n_alloc"] / (ms / 1e3)
        parity = head["parity"]

        # dominant kernel (k_pipeline), timed live with CUDA events on the engine's own stream in timing mode, same causal window
        teng = E.Engine(max_gpus=G, max_batch=1 << 20, timing=True)
        teng.load_profiles(ch.rows)
        teng.set_causal_window(A)
        for _ in range(3):
            teng.load_inventory(ch.node_off, occ0)
            teng.reset_stats()
            teng.place_stream_ptr(sizes, d_in_all.data_ptr(), d_res.data_ptr(), device=True)
            teng.synchronize()
        st = teng.stats()
        teng.close()
        ms_pipe = st["ms_commit"]
        alg_bytes = 16 * n_ops + 2 * G * nb                   # B_alg = 16 R + 2 G per batch (SURVEY 8d), whole stream = one launch
        peak, how = measured_peak()
        achieved = alg_bytes / (ms_pipe / 1e3) / 1e9
        roofline = {"bound": "hbm", "kernel": "k_pipeline", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": ncu_traffic(), "peak_source": how, "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": ms_pipe, "launches": 1,
                    "note": "latency-bound: a batch's decisions are ONE exact recurrence over the inventory (first-fit in arrival order); with one batch in flight the "
                            "inventory stages resolve it by speculative rounds (every stage simulates its segment from predicted queue heads, commits when certified). "
                            "Inventory, queues and candidates are shared-memory / L2 resident by construction, so DRAM traffic stays below the algorithmic bytes",
                    "speculative_rounds": head["spec"],
                    "phase_ms_per_step": {"prepare": st["ms_free"], "partition": st["ms_partition"], "pipeline": st["ms_commit"], "total": st["ms_total"]}}

        faithful = faithful_from_prefill(oracle, ch.node_off, ch.rows, prefill)
        cpu, ok_cpu = cpu_baseline_batches(ch.node_off, ch.rows, occ0, batches, head["got"], head["occ"], 0, faithful, a.faithful_ops,
                                           "the first %d operations of the churn stream on the pre-filled 65536-GPU inventory (SURVEY 8d prefix)" % a.faithful_ops)
        parity = parity and ok_cpu

        # ---- beside the headline: the other causal depth, and the replay ceiling on the original stream
        other_A = 2 if A == 1 else 1
        cho, occo, batcheso, _, _ = record_churn(E, W, other_A)
        assert np.array_equal(np.array([len(b) for b in batcheso], dtype=np.uint32), sizes)
        other = measure(cho, occo, batcheso, other_A, other_A == 1)
        parity = parity and other["parity"]
        if A == 1:
            ch1, occ1, batches1 = ch, occ0, batches
        else:
            ch1, occ1, batches1 = cho, occo, batcheso
        load_variant(ch1, occ1, batches1)
        want1, want1_occ, _ = fast_replay(oracle, ch1.node_off, ch1.rows, occ1, batches1)
        check1 = lambda got, occ: all(np.array_equal(x, y) for x, y in zip(got, want1)) and np.array_equal(occ, want1_occ)
        n_alloc1 = int(sum(int((b["op"] == E.OP_ALLOC).sum()) for b in batches1))
        eng.set_causal_window(0)
        ms_r_dev, _ = ctx.timed(step_device, a.steps, 3)
        extra_ok = check1(results_of(d_res), eng.read_occupancy())

        def step_replay_e2e():
            occ_view.copy_(d_occ0)
            eng.place_stream_ptr(sizes, h_in_all.data_ptr(), h_out_all.data_ptr(), device=False)
        ms_r_e2e, wall_r = ctx.timed(step_replay_e2e, a.steps, 3)
        extra_ok &= check1(results_of(h_out_all), eng.read_occupancy())
        parity = parity and bool(extra_ok)

        def block(m, Ax):
            d = {"batches_in_flight": Ax, "value": per(m, m["dev_ms"]), "ms_per_step": m["dev_ms"], "open_stream_e2e_value": per(m, m["open_ms"]), "open_stream_e2e_ms_per_step": m["open_ms"],
                 "ref_fast_value": m["n_alloc"] / m["ref_fast_s"], "unit": UNIT, "parity_vs_ref_fast": m["parity"], "speculative_rounds": m["spec"]}
            if "calls_ms" in m:
                d["per_batch_calls_value"] = per(m, m["calls_ms"]); d["per_batch_calls_ms_per_step"] = m["calls_ms"]
            return d
        strict, feed = (head, other) if A == 1 else (other, head)
        lines_extra = {
            "strict_causal": dict(block(strict, 1), workload="the original config-4 stream (a FREE may name any allocation live at batch start), ONE batch in flight: every batch "
                                                                 "is resolved before the next one starts"),
            "causal_feed": dict(block(feed, 2), workload="variant whose FREEs name allocations at least 2 batches old (Churn(min_age=2)), TWO batches in flight"),
            "replay_value": n_alloc1 / (ms_r_dev / a.steps / 1e3), "replay_ms_per_step": ms_r_dev / a.steps,
            "replay_e2e_value": n_alloc1 / (max(ms_r_e2e, wall_r * 1e3) / a.steps / 1e3),
            "replay_note": "the original stream, all 16 batches handed over in one isl_place_stream* call: the pipelining ceiling; NOT causally available to a live caller",
        }
        value = per(head, head["dev_ms"])
        variant = ("the original config-4 stream: a FREE may name any allocation live at batch start" if A == 1 else
                   "a FREE of batch b names an allocation placed by batch b - %d or earlier (Churn(min_age))" % A)
        line = base_line(ctx, "c4", value, head["dev_ms"],
                         {"mode": "strict causal: one batch in flight" if A == 1 else "causal feed", "min_age_batches": A, "batches_in_flight": A,
                          "workload_variant": variant,
                          "ops_per_step": n_ops, "alloc_requests_per_step": n_alloc, "free_requests_per_step": n_ops - n_alloc,
                          "ops_counted": "ALLOC decisions (placed or definitively no-capacity); FREEs are resolved inside the same step but not counted",
                          "ops_per_sec_incl_frees": n_ops / (head["dev_ms"] / 1e3),
                          "batches_per_step": nb, "gpus_in_inventory": G, "policy": "first-fit", "parallelism": "segment pipeline with speculative rounds, 1 GPU"},
                         parity, head["launches"], clocks)
        if A == 1:
            e2e_ms, api = head["calls_ms"], ("isl_place_batch once per batch, host buffers in and out, synchronous (the call SURVEY 8d defines the metric on; each call's H2D and D2H "
                                             "inside); CUDA events around the step and the host clock, the larger is reported")
        else:
            e2e_ms, api = head["open_ms"], ("isl_stream_open / isl_stream_submit / isl_stream_wait / isl_stream_close, pinned host buffers; batch b submitted after "
                                            "isl_stream_wait(b - %d); CUDA events around the step and the host clock, the larger is reported" % A)
        line["e2e"] = {"value": per(head, e2e_ms), "unit": UNIT, "h2d_bytes_per_step": 8 * n_ops, "d2h_bytes_per_step": 8 * n_ops,
                       "ms_per_step": e2e_ms, "ops_per_sec_incl_frees": n_ops / (e2e_ms / 1e3), "api": api,
                       "open_stream_value": per(head, head["open_ms"]), "open_stream_ms_per_step": head["open_ms"]}
        line["roofline"] = roofline
        line["cpu_baseline"] = cpu
        line.update(lines_extra)
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, np.concatenate(head["got"]), head["occ"])
        eng.close()
        return line, parity

    # ---- N > 1: partitioned inventory
    from instaslice_b200 import dist as D
    lo, hi = D.partition_bounds(G, world, rank)
    eng.set_partition(lo, hi)
    D.connect_ring(eng, rank, world)          # next rank's token inbox mapped through CUDA IPC (peer store over NVLink)
    D.connect_owner(eng, rank, world)         # rank 0's result array mapped into every other rank; ring size for the causal window
    D.connect_spec(eng, rank, world, G)       # every rank's record memory of the speculative rounds mapped into every other rank
    eng.set_causal_window(A)
    stream_ids = iter(range(1, 1 << 30))
    triples = []          # (start, pipeline enqueued-to-end, all-gather done) events of every device step: the phase table comes from the TIMED steps

    def step_device():
        occ_view.copy_(d_occ0)
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        # every rank runs the segment pipeline over its own GPU range; tokens, PLACED records and the causal-window counter cross
        # ranks inside the running kernels
        eng.place_stream_partitioned(sizes, d_in_all.data_ptr(), d_res.data_ptr(), next(stream_ids))
        e[1].record()
        occ_view.copy_(D.gather_occupancy(occ_view[lo:hi], G, world, rank))   # NCCL all-gather of the occupancy shards (also tells rank 0 every record has landed)
        e[2].record()
        triples.append(e)

    def step_e2e():         # rank 0 is the controller: it owns the host buffers; the request stream reaches the other ranks over NVLink
        occ_view.copy_(d_occ0)
        if rank == 0:
            d_in_all.copy_(h_in_all, non_blocking=True)
        dist.broadcast(d_in_all, src=0)
        eng.place_stream_partitioned(sizes, d_in_all.data_ptr(), d_res.data_ptr(), next(stream_ids))
        occ_view.copy_(D.gather_occupancy(occ_view[lo:hi], G, world, rank))
        if rank == 0:
            h_out_all.copy_(d_res, non_blocking=True)

    if rank == 0:
        sampler.start()
    launches0 = eng.stats()["kernel_launches"]
    ms_dev, _ = ctx.timed(step_device, a.steps, a.warmup)
    st_n = eng.stats()
    launches = st_n["kernel_launches"] - launches0
    sp = torch.tensor([st_n["spec_chunks"], st_n["spec_rounds"], st_n["spec_sims"]], dtype=torch.float64, device="cuda")
    dist.all_reduce(sp, op=dist.ReduceOp.SUM)       # the last stage (last rank) counts chunks and rounds, every rank its simulations
    spec_stats = {"chunks": int(sp[0].item()), "rounds_per_chunk": float(sp[1].item()) / max(1.0, float(sp[0].item())), "simulations_per_chunk": float(sp[2].item()) / max(1.0, float(sp[0].item()))}
    clocks = sampler.stop() if rank == 0 else None
    got_dev = results_of(d_res) if rank == 0 else None
    occ_dev = occ_view.cpu().numpy()
    ms_e2e, wall_e2e = ctx.timed(step_e2e, a.steps, a.warmup)
    got_e2e = results_of(h_out_all) if rank == 0 else None
    timed_triples = triples[a.warmup:a.warmup + a.steps]          # the K timed device steps (the e2e leg does not use step_device)
    ph = torch.tensor([sum(e[0].elapsed_time(e[1]) for e in timed_triples) / a.steps, sum(e[1].elapsed_time(e[2]) for e in timed_triples) / a.steps],
                      dtype=torch.float64, device="cuda")
    dist.all_reduce(ph, op=dist.ReduceOp.MAX)
    line = None
    if rank == 0:
        import oracle
        cpu, ok = cpu_baseline_batches(ch.node_off, ch.rows, occ0, batches, got_dev, occ_dev, 0)
        parity = ok and all(np.array_equal(x, y) for x, y in zip(got_e2e, got_dev))
        ms_pipe = float(ph[0].item())
        alg_bytes = 16 * n_ops + 2 * G * nb
        peak, how = measured_peak()
        achieved = alg_bytes / (ms_pipe / 1e3) / 1e9
        value = n_alloc * a.steps / (ms_dev / 1e3)
        line = base_line(ctx, "c4", value, ms_dev / a.steps,
                         {"mode": ("strict causal: one batch in flight" if A == 1 else "causal feed") + " (device-side window across ranks)", "min_age_batches": A, "batches_in_flight": A,
                          "workload_variant": ("the original config-4 stream: a FREE may name any allocation live at batch start" if A == 1 else
                                               "a FREE of batch b names an allocation placed by batch b - %d or earlier (min_age)" % A),
                          "ops_per_step": n_ops, "alloc_requests_per_step": n_alloc, "free_requests_per_step": n_ops - n_alloc,
                          "ops_counted": "ALLOC decisions (placed or definitively no-capacity); FREEs are resolved inside the same step but not counted",
                          "ops_per_sec_incl_frees": n_ops * a.steps / (ms_dev / 1e3),
                          "batches_per_step": nb, "gpus_in_inventory": G, "policy": "first-fit",
                          "parallelism": "inventory partitioned over %d ranks: ONE sequence of inventory stages over all ranks, speculative rounds with the per-round records "
                                         "peer-stored into the other ranks' record memory + PLACED records peer-stored into rank 0's result array + "
                                         "peer-atomic window counter + NCCL all-gather of the occupancy shards" % world,
                          "speculative_rounds": spec_stats},
                         parity, launches, clocks)
        e2e_ms = max(ms_e2e, 0.0)
        line["e2e"] = {"value": n_alloc * a.steps / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": 8 * n_ops, "d2h_bytes_per_step": 8 * n_ops,
                       "ms_per_step": e2e_ms / a.steps,
                       "api": "rank 0: H2D of the stream + NCCL broadcast to the other ranks, isl_place_stream_partitioned per rank (causal window %d), NCCL all-gather of occupancy, "
                              "D2H of rank 0's result array" % A}
        line["roofline"] = {"bound": "hbm", "kernel": "k_pipeline", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic(),
                            "peak_source": how, "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": ms_pipe, "launches": world,
                            "note": "per-rank k_pipeline incl. its waits for the other ranks' records (max over ranks); a batch is ONE sequential recurrence over the "
                                    "whole inventory, resolved by speculative rounds of all stages of all ranks — more ranks add NVLink latency to every round, not parallel work",
                            "phase_ms_per_step_max_over_ranks": {"pre-pass + pipeline (enqueue to kernel end)": ms_pipe, "occupancy all-gather (NCCL) + copy back": float(ph[1].item()),
                                                                  "result merge": 0.0}}
        line["cpu_baseline"] = cpu
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, np.concatenate(got_dev), occ_dev)
    dist.barrier()
    eng.close()
    return line, parity


# ---- the reference arm ----------------------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the reference's own CPU algorithm.  The Go binary cannot be built here (no go / gccgo, un-vendored deps),
    so this is oracle/ref_faithful.cpp — the structure-for-structure port, one reconcile worker like the reference — on a bounded
    sample of the same workload, counted in the same unit (ALLOC decisions/s)."""
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    import oracle
    from instaslice_b200 import engine as E, tables
    from instaslice_b200 import workloads as W
    oracle.build()
    cfgname = args.config
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    if cfgname == "c5":
        rate, seconds, G = 10000.0, min(float(args.seconds), 2.0), 4096
        n, arrivals, life = c5_trace(W, rate, seconds)
        rows = E.make_profiles(tables.A100_40GB)
        node_off = W.node_offsets(G // 8, 8)
        ff = oracle.Faithful(node_off, rows)
        lat, _, _, sz, wall, _ = c5_replay(C.cast(oracle.lib().orc_f_place_batch, C.c_void_p).value, ff._h, n, arrivals, life, tables.profile_index(tables.A100_40GB, "3g.20gb"))
        s = latency_summary(lat)
        sample = "ref_faithful.cpp through the native open-loop driver, first %.0f s of the trace (%d requests)" % (seconds, n)
        print(json.dumps({"impl": "reference", "metric": "placement_latency_p50_us", "value": s["p50"], "unit": "us", "n_gpus": args.gpus, "steps": 1, "warmup": 0,
                          "ms_per_step": wall * 1e3, "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                          "config": {"workload": WORKLOADS["c5"], "sample": sample}, "latency_us": s,
                          "cpu_baseline": {"value": s["p50"], "unit": "us", "cores": 1, "kind": "port", "sample": sample},
                          "e2e": {"value": s["p50"], "unit": "us", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0
    if cfgname == "c4":
        # the own arm's workload (same min_age), recorded through ref_fast (this arm may execute oracle/)
        ch = W.Churn(min_age=max(1, args.min_age))
        fast = oracle.Fast(ch.node_off, ch.rows)
        fast.load(np.zeros(ch.G, dtype=np.uint8))
        results = []

        def placer(req):
            results.append(fast.place(req))
            return results[-1]
        ch.generate(placer)
        nbp = ch.n_prefill_batches
        prefill = list(zip(ch.batches[:nbp], results[:nbp]))
        prefix = ch.batches[nbp][: args.faithful_ops]
        node_off, rows = ch.node_off, ch.rows
        make_state = lambda: faithful_from_prefill(oracle, node_off, rows, prefill)
        what = "the first %d operations of churn batch 0 (SURVEY 8d prefix) on the pre-filled 65536-GPU inventory, split over the %d timed steps" % (len(prefix), steps)
    else:
        node_off, occ0, rows, req = {"c1": W.config1, "c2": W.config2, "c3": W.config3, "c3bf": W.config3}[cfgname]()
        prefix = req if cfgname in ("c1", "c2") else req[:20000]

        def make_state():
            f = oracle.Faithful(node_off, rows)
            f.load_occupancy_as_dangling(occ0)
            return f
        what = ("the whole job" if len(prefix) == len(req) else "the first %d requests of the job" % len(prefix)) + ", split over the %d timed steps" % steps
    # warm-up on a state of its own (small), then ONE pass over the prefix cut into `steps` consecutive slices on one evolving state
    if warmup:
        w = make_state()
        for _ in range(warmup):
            w.place(prefix[: max(1, min(64, len(prefix)))])
    f = make_state()
    cuts = np.linspace(0, len(prefix), steps + 1).astype(int)
    total, n_alloc = 0.0, 0
    for i in range(steps):
        piece = prefix[cuts[i]:cuts[i + 1]]
        t0 = time.perf_counter()
        f.place(piece)
        total += time.perf_counter() - t0
        n_alloc += int((piece["op"] == E.OP_ALLOC).sum())
    value = n_alloc / total if total > 0 else 0.0
    sample = "ref_faithful.cpp on %s: %d ops = %d ALLOC decisions in %.1f s" % (what, len(prefix), n_alloc, total)
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
                      "ms_per_step": total / steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8",
                      "data": "synthetic", "config": {"workload": WORKLOADS[cfgname], "sample": sample, "min_age_batches": max(1, args.min_age) if cfgname == "c4" else None,
                                                      "ops_counted": "ALLOC decisions (placed or definitively no-capacity)"},
                      "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample,
                                       "note": "single reconcile worker like the reference (controller-runtime default); the Go binary cannot be built in this image; "
                                               "API-server / etcd time is excluded on both arms"},
                      "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
    return 0


def run_own(args):
    ctx = Ctx(args)
    if args.config == "c4":
        line, parity = run_c4(ctx)
    elif args.config == "c5":
        line, parity = run_c5(ctx) if ctx.rank == 0 else (None, True)
    else:
        line, parity = run_single_batch(ctx, args.config)
    if ctx.world > 1:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()
        sys.stdout.flush()
    if ctx.rank == 0 and line is not None:
        sys.stdout.flush()
        if ctx.real_stdout is not None:     # file descriptor 1 stays on stderr to the end (NCCL still logs while the process exits): the JSON line
            os.write(ctx.real_stdout, (json.dumps(line) + "\n").encode())      # goes straight to the real stdout — its only line
        else:
            print(json.dumps(line), flush=True)
    return 0 if parity else 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--config", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--min-age", type=int, default=1, help="c4: a FREE names an allocation at least this many batches old = batches in flight of the causal feed")
    ap.add_argument("--faithful-ops", type=int, default=10000, help="c4: operations of the churn prefix the reference-as-written port is timed on (SURVEY 8d)")
    ap.add_argument("--seconds", type=float, default=10.0, help="c5: length of the replay")
    ap.add_argument("--dump-outputs", metavar="DIR", help="c1-c4: write the results of the last timed step and the final occupancy to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "own" or args.config == "c5"):
        ap.error("--dump-outputs needs --impl own and one of the configs c1-c4")
    args.warmup = max(args.warmup, 3) if args.impl == "own" else args.warmup
    sys.exit(run_reference(args) if args.impl == "reference" else run_own(args))


if __name__ == "__main__":
    main()
