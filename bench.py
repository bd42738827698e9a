#!/usr/bin/env python
"""bench.py -- GCRA decisions/sec on B200 (BASELINE.json metric), one JSON line.

A "step" is one tick: one pass of the hot path over one batch of 2^20 synthetic requests.

  N=1   BASELINE.json configs[1]: 10 M resident keys, Zipf-1.0 request stream (tests/traces.py
        config2), one `now` per tick advancing 1 ms, after a warm pass that inserts every key.
  N>1   configs[4] shape: the key space (10 M keys per GPU) is hash-sharded across the N engines;
        every rank ingests its own 2^20-request slice of the global tick, routes each request to
        the owning shard, decides locally, and routes the results back.  Weak scaling.

value        kernel-only: requests already resident in HBM, K steps back to back on the stream
e2e          the same K ticks through the C-ABI pinned host ring (gcra_ring_*): H2D of every tick's
             requests, kernels, D2H of every tick's results inside the timed region
roofline     K1 (all launches of a tick), algorithmic bytes / CUDA-event time; `traffic` is read from the
             newest committed `ncu --set full` capture under profiles/ (null when there is none)
sweep        K2 on BASELINE configs[2]: 100 M resident keys, expired fractions 0 / 1 / 50 / 100 %
sustained    the resident ticks cycled (their clocks advanced) for >= 0.5 s of device time
parity       the CPU oracle (C++ restatement of the reference; the reference is Rust and cannot be built
             here) replays the SAME trace: at N=1 the whole 10 M-key trace (warm pass + every tick), at
             N>1 a key subset (the hottest keys + sampled cold keys; keys are independent) of the first ticks
cpu_baseline that oracle replay, timed (single thread = the reference's design point)

`--impl reference` times the CPU restatement on all host cores (hash-sharded stores, built ONCE at the
full key count) on the same config instead.

`--dump-outputs DIR` writes the result rows of the last timed tick (at N>1 rank 0's slice; for `--impl reference`
the last tick of the last step) as DIR/<field>.npy, one float64 array per result field.  The trace is seeded, so
the same arguments give the same requests and two builds can be compared output for output.
"""
import argparse
import glob
import json
import os
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # many streams per engine: one hardware queue each
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import traces  # noqa: E402

TICK = 1 << 20
KEYS_PER_GPU = 10_000_000
METRIC = "gcra_decisions_per_sec"
UNIT = "decisions/s"
REF_TICKS_PER_STEP = 2


def measured_peak_gbs():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu=0):
        self.gpu, self.rows, self.proc = gpu, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def build_requests(tc, key_hash_of, trace):
    req = np.empty(len(trace), tc.REQ_DTYPE)
    req["key_hash"] = key_hash_of[trace["key"].astype(np.int64)]
    for f in ("max_burst", "count_per_period", "period", "quantity", "now_ns"):
        req[f] = trace[f]
    return req


def dump_outputs(out_dir, res):
    """Every field a caller of the timed path receives, one tick of RES_DTYPE rows (2^20 rows: 40 MB).  The fields
    are integers; float64 holds them exactly below 2^53, which is checked rather than assumed."""
    os.makedirs(out_dir, exist_ok=True)
    for name in ("allowed", "status", "remaining", "reset_after_ns", "retry_after_ns"):
        col = res[name]
        f = col.astype(np.float64)
        if not np.array_equal(f.astype(col.dtype), col):
            raise SystemExit("--dump-outputs: %s has a value float64 cannot hold exactly" % name)
        np.save(os.path.join(out_dir, name + ".npy"), f)


def traffic_from_profiles():
    """DRAM bytes (read + write) of the K1 kernels of ONE tick, summed from the newest committed
    `ncu --set full` raw page under profiles/ (written by tools/ncu_k1_summary.py)."""
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_k1_traffic.json")))
    if not files:
        return None, None
    try:
        d = json.load(open(files[-1]))
        return float(d["dram_bytes_per_tick"]), os.path.relpath(files[-1], ROOT)
    except Exception:
        return None, None


# ---------------------------------------------------------------------------------------------------------
# --impl reference
# ---------------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """The CPU restatement of the reference on all host cores: hash-sharded AdaptiveStores built ONCE at the
    full key count of this config (same key universe and tick generator as the GPU arm), every step a fresh
    bounded sample of ticks.  Median over the timed steps."""
    if rank != 0:
        return
    import oracle
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    n_keys = args.keys * max(args.gpus, 1)
    t0 = time.time()
    stores = [oracle.OracleStore(oracle.ADAPTIVE, capacity=max(n_keys // cores, 1000), created_ns=traces.T0)
              for _ in range(cores)]
    for a in range(0, n_keys, 10_000_000):                       # untimed: table population
        ids = np.arange(a, min(a + 10_000_000, n_keys), dtype=np.uint64)
        w = np.zeros(len(ids), traces.REQ_DTYPE)
        w["key"] = ids
        traces.fill_policy(w, (ids % np.uint64(8)).astype(np.int64))
        w["quantity"] = 1
        w["now_ns"] = traces.T0
        oracle.replay_sharded(stores, w)
    build_s = time.time() - t0
    W, K = max(args.warmup, 3), args.steps
    vals = []
    for s in range(W + K):
        tr = traces.config2(n_keys=n_keys, n_ticks=REF_TICKS_PER_STEP, tick_size=TICK, start_tick=s * REF_TICKS_PER_STEP)
        out, sec = oracle.replay_sharded(stores, tr)             # timed: the decision loops only
        if s >= W:
            vals.append(len(tr) / sec)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out[-TICK:])
    value = float(np.median(vals))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(vals), "warmup": W, "ms_per_step": 1e3 * TICK / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": "%dM keys, Zipf-1.0 request stream, ticks of 2^20 requests (tests/traces.py config2)"
                               % (n_keys // 1_000_000),
                   "keys": n_keys, "tick": TICK, "ticks_per_step": REF_TICKS_PER_STEP,
                   "same_config_as_gpu_arm": True, "build_seconds": round(build_s, 1)},
        "spread": {"min": float(min(vals)), "max": float(max(vals)), "steps": len(vals)},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d hash-sharded AdaptiveStore restatements (C++ oracle; the Rust reference cannot be "
                                   "built here), one pinned thread each, built once at %d keys; every step = %d fresh "
                                   "ticks of 2^20 requests, median of %d steps" % (cores, n_keys, REF_TICKS_PER_STEP, len(vals))},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
# K2 block (N=1): BASELINE configs[2]
# ---------------------------------------------------------------------------------------------------------
def sweep_block(tc, peak, device, n_keys=100_000_000):
    """100 M resident keys (one policy, creation clocks staggered over 100 s so that a sweep at a chosen time
    expires a chosen fraction), sweeps at expired fractions 0 / 1 / 50 / 100 %.  Algorithmic bytes: 16 B per
    table slot scanned + 16 B per evicted entry."""
    B = 1 << 20
    st = tc.ManualStore(capacity=n_keys, device=device, created_ns=traces.T0, max_batch=B)
    lim = tc.RateLimiter(st)
    burst, count, period = 100, 1000, 60                 # emission interval 60 ms, tolerance 5.94 s
    dvt = 99 * 60_000_000
    req = np.empty(B, tc.REQ_DTYPE)
    t0 = time.time()
    for a in range(0, n_keys, B):
        ids = np.arange(a, min(a + B, n_keys), dtype=np.uint64)
        r = req[:len(ids)]
        r["key_hash"] = tc.hash_key_ids(ids)
        r["max_burst"], r["count_per_period"], r["period"], r["quantity"] = burst, count, period, 1
        r["now_ns"] = traces.T0 + (ids % np.uint64(100)).astype(np.int64) * 1_000_000_000
        lim.rate_limit_batch(r)
    fill_s = time.time() - t0
    slots = st.stats()["table_slots"]
    out = []
    # an entry created at T0 + j s expires at T0 + j s + dvt
    plan = [("0 %", traces.T0), ("0 % (repeat)", traces.T0 + 1),
            ("1 %", traces.T0 + dvt + 500_000_000), ("50 %", traces.T0 + dvt + 50_500_000_000),
            ("100 % (the rest)", traces.T0 + dvt + 200_000_000_000), ("empty table", traces.T0 + dvt + 300_000_000_000)]
    for label, now in plan:
        before = st.len()
        removed = st.sweep(now)
        ms = st.last_sweep_ms()
        alg = 16.0 * slots + 16.0 * removed
        out.append({"expired": label, "live_before": before, "removed": removed, "ms": ms,
                    "achieved_GBps": alg / ms / 1e6, "frac": alg / ms / 1e6 / peak})
    st.close()
    return {"kernel": "sweep_kernel", "keys": n_keys, "table_slots": slots, "fill_seconds": round(fill_s, 1),
            "algorithmic_bytes": "16 B per slot scanned + 16 B per evicted entry", "peak_GBps": peak, "runs": out}


# ---------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--keys", type=int, default=KEYS_PER_GPU)
    ap.add_argument("--no-cpu", action="store_true", help="skip the oracle replay (no parity, no cpu_baseline)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--sustain-sec", type=float, default=0.5)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed tick's results as DIR/<field>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import throttlecrab_b200 as tc
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_MIN_P2P_NCHANNELS", "8")
        dist.init_process_group("nccl", device_id=dev)

    W, K = max(args.warmup, 3), args.steps
    n_local_keys = args.keys
    n_keys = n_local_keys * world
    peak, peak_kind = measured_peak_gbs()

    # ---------------------------------------------------------------- synthetic workload
    t0 = time.time()
    key_hash_of = tc.hash_key_ids(np.arange(n_keys, dtype=np.uint64))
    store = tc.ManualStore(capacity=n_local_keys, device=local_rank, created_ns=traces.T0,
                           max_batch=TICK if world == 1 else 2 * TICK)
    lim = tc.RateLimiter(store)
    if world == 1:
        # warm pass: every key inserted once (BASELINE configs[1]: keys resident)
        warm = build_requests(tc, key_hash_of, traces.warm_pass(n_keys))
        for a in range(0, n_keys, TICK):
            lim.rate_limit_batch(warm[a:a + TICK])
        del warm
        tr = traces.config2(n_keys=n_keys, n_ticks=W + K, tick_size=TICK)
        ticks = build_requests(tc, key_hash_of, tr)
    else:
        from throttlecrab_b200.sharded import make_sharded
        sh = make_sharded(lim, dist, dev)
        # warm pass through the sharded path: rank r submits keys [r*10M, (r+1)*10M), owners insert them
        stream0 = torch.cuda.Stream(dev)
        torch.cuda.set_stream(stream0)
        wres = torch.empty(TICK * 32, dtype=torch.uint8, device=dev)
        for a in range(0, n_local_keys, TICK):
            ids = np.arange(rank * n_local_keys + a, rank * n_local_keys + min(a + TICK, n_local_keys), dtype=np.uint64)
            w = np.zeros(TICK, traces.REQ_DTYPE)          # padded with copies of the last key (harmless)
            w["key"][:len(ids)] = ids
            w["key"][len(ids):] = ids[-1]
            traces.fill_policy(w, (w["key"] % np.uint64(8)).astype(np.int64))
            w["quantity"] = 1
            w["now_ns"] = traces.T0
            wreq = torch.from_numpy(build_requests(tc, key_hash_of, w).view(np.uint8)).to(dev)
            sh.step(wreq, wres)
        torch.cuda.synchronize()
        # every rank generates ITS slice of each global Zipf tick (same generator as N=1)
        tr = traces.config2_rank_slice(n_keys, TICK, 0, W + K, rank, world)
        ticks = build_requests(tc, key_hash_of, tr)
    gen_s = time.time() - t0

    d_req = torch.from_numpy(ticks.view(np.uint8).reshape(W + K, TICK * 48)).to(dev)
    d_res = torch.empty((W + K, TICK * 32), dtype=torch.uint8, device=dev)
    # an explicit (non-default) stream: handle 0 would mean "the engine's own stream" to the C ABI
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)

    def step(i):
        if world == 1:
            lim.submit_device(TICK, d_req[i].data_ptr(), d_res[i].data_ptr(), stream.cuda_stream)
        else:
            sh.submit(d_req[i], d_res[i])

    def drain():
        if world > 1:
            sh.finish()
        else:
            lim.join(stream.cuda_stream)

    # ---------------------------------------------------------------- kernel-only (value)
    for i in range(W):
        step(i)
    drain()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = store.launch_count()
    stats0 = store.stats()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    step_ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    ev0.record(stream)
    step_ev[0].record(stream)
    for i in range(W, W + K):
        step(i)
        step_ev[i - W + 1].record(stream)
    drain()
    ev1.record(stream)
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    total_ms = ev0.elapsed_time(ev1)
    launches = store.launch_count() - launches0
    stats1 = store.stats()
    step_ms = [step_ev[i].elapsed_time(step_ev[i + 1]) for i in range(K)]
    if dist:
        tmax = torch.tensor([total_ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        total_ms = float(tmax.item())
    value = world * K * TICK / (total_ms * 1e-3)

    res_all = d_res.cpu().numpy().view(tc.RES_DTYPE).reshape(W + K, TICK)      # every tick's results, warm-up included
    res_np = res_all[W:]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res_all[W + K - 1])
    n_allowed = int(res_np["allowed"].sum())
    n_ok = int((res_np["status"] == 0).sum())

    # ---------------------------------------------------------------- sustained: the resident ticks cycled
    sustained = None
    if world == 1 and args.sustain_sec > 0:
        cycles = max(int(np.ceil(args.sustain_sec / ((W + K) * total_ms / K * 1e-3))), 1)
        req_i64 = d_req.view(torch.int64).view(W + K, TICK, 6)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        s0.record(stream)
        for c in range(cycles):
            # the clock of every resident tick moves on by a whole cycle (a device-side add on the same stream)
            req_i64[:, :, 5] += (W + K) * 1_000_000
            for i in range(W + K):
                step(i)
            drain()
        s1.record(stream)
        torch.cuda.synchronize()
        sus_ms = s0.elapsed_time(s1)
        sustained = {"value": cycles * (W + K) * TICK / (sus_ms * 1e-3), "unit": UNIT, "seconds": sus_ms * 1e-3,
                     "ticks": cycles * (W + K),
                     "note": "the %d resident ticks cycled %d times, every cycle's clocks advanced by %d ms on the device "
                             "(the add is inside the timed region)" % (W + K, cycles, W + K)}

    phases = phase_detail = None
    if world == 1:
        # phase split of ONE tick run serially on one stream (library-side CUDA events); the timed region above
        # pipelines consecutive ticks over three streams, so its per-tick time is below this total
        extra = torch.empty(TICK * 32, dtype=torch.uint8, device=dev)
        if os.environ.get("GCRA_DBG"):          # timing experiments only: this serial tick's results are wrong
            store._L.gcra_debug_set(store._h, int(os.environ["GCRA_DBG"]))
        lim.rate_limit_batch_device(TICK, d_req[W].data_ptr(), extra.data_ptr(), stream.cuda_stream)
        torch.cuda.synchronize()
        phases = store.last_kernel_ms()
        try:
            phase_detail = store.last_kernel_ms_detail()
        except Exception:
            phase_detail = None

    # ---------------------------------------------------------------- e2e through the pinned ring
    e2e = None
    if world == 1 and not args.no_e2e:
        store2 = tc.ManualStore(capacity=n_local_keys, device=local_rank, created_ns=traces.T0, max_batch=TICK)
        lim2 = tc.RateLimiter(store2)
        warm = build_requests(tc, key_hash_of, traces.warm_pass(n_keys))
        for a in range(0, n_keys, TICK):
            lim2.rate_limit_batch(warm[a:a + TICK])
        del warm
        KE = min(K, 32)          # every step owns a pinned 80-MiB slot: cap the pinned memory at ~3 GB
        ring = tc.Ring(lim2, slots=W + KE, slot_capacity=TICK)
        for i in range(W + KE):
            ring.req[i][:] = ticks[i * TICK:(i + 1) * TICK]      # requests sit in pinned host memory
        for i in range(W):
            ring.submit(i, TICK)
        for i in range(W):
            ring.wait(i)
        store2.sync()
        t_a = time.perf_counter()
        for i in range(W, W + KE):
            ring.submit(i, TICK)
        for i in range(W, W + KE):
            ring.wait(i)
        t_b = time.perf_counter()
        e2e_val = KE * TICK / (t_b - t_a)
        got = np.concatenate([ring.res[i] for i in range(W, W + KE)])
        same = got.tobytes() == res_np[:KE].reshape(-1).tobytes()
        e2e = {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": TICK * 48, "d2h_bytes_per_step": TICK * 32,
               "api": "gcra_ring_submit/gcra_ring_wait, pinned host ring, 48-byte requests", "steps": KE,
               "matches_kernel_only_results": bool(same)}
        del ring
        # extra: compact 16-byte requests (policy table + per-call now), same ticks, same results
        try:
            store3 = tc.ManualStore(capacity=n_local_keys, device=local_rank, created_ns=traces.T0, max_batch=TICK)
            lim3 = tc.RateLimiter(store3)
            pol = np.zeros(8, tc.POLICY_DTYPE)
            pol["max_burst"], pol["count_per_period"], pol["period"] = traces.POLICIES.T
            lim3.set_policies(pol)
            warm = build_requests(tc, key_hash_of, traces.warm_pass(n_keys))
            for a in range(0, n_keys, TICK):
                lim3.rate_limit_batch(warm[a:a + TICK])
            del warm
            ring16 = tc.Ring(lim3, slots=W + KE, slot_capacity=TICK, compact=True)
            for i in range(W + KE):
                sl = ticks[i * TICK:(i + 1) * TICK]
                r16 = ring16.req[i]
                r16["key_hash"] = sl["key_hash"]
                r16["quantity"] = sl["quantity"]
                pidx = np.zeros(TICK, np.uint32)
                for j, p in enumerate(traces.POLICIES):
                    m = (sl["max_burst"] == p[0]) & (sl["count_per_period"] == p[1]) & (sl["period"] == p[2])
                    pidx[m] = j
                r16["policy"] = pidx
            nows = [int(ticks["now_ns"][i * TICK]) for i in range(W + KE)]
            for i in range(W):
                ring16.submit(i, TICK, nows[i])
            for i in range(W):
                ring16.wait(i)
            store3.sync()
            t_a = time.perf_counter()
            for i in range(W, W + KE):
                ring16.submit(i, TICK, nows[i])
            for i in range(W, W + KE):
                ring16.wait(i)
            t_b = time.perf_counter()
            got16 = np.concatenate([ring16.res[i] for i in range(W, W + KE)])
            e2e["compact_requests"] = {"value": KE * TICK / (t_b - t_a), "unit": UNIT, "h2d_bytes_per_step": TICK * 16,
                                       "d2h_bytes_per_step": TICK * 32,
                                       "matches_kernel_only_results": bool(got16.tobytes() == res_np[:KE].reshape(-1).tobytes())}
            del ring16
            store3.close()
        except Exception as ex:      # the extra must never cost the main line
            e2e["compact_requests"] = {"error": repr(ex)}
        store2.close()

    if world > 1 and not args.no_e2e:
        # e2e at N GPUs: every rank copies its tick slice from pinned host memory, routes, decides,
        # routes back and copies the results to pinned host memory (time continues after the timed ticks)
        tr2 = traces.config2_rank_slice(n_keys, TICK, W + K, K, rank, world)
        h_req = torch.from_numpy(build_requests(tc, key_hash_of, tr2).view(np.uint8).reshape(K, TICK * 48)).pin_memory()
        h_res = torch.empty((K, TICK * 32), dtype=torch.uint8).pin_memory()
        dqs = [torch.empty(TICK * 48, dtype=torch.uint8, device=dev) for _ in range(K)]
        drs = [torch.empty(TICK * 32, dtype=torch.uint8, device=dev) for _ in range(K)]
        s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        sh.finish()
        torch.cuda.synchronize()
        dist.barrier()
        t_a = time.perf_counter()
        copied = 0
        for i in range(K):
            with torch.cuda.stream(s_in):                     # H2D of tick i overlaps earlier ticks
                dqs[i].copy_(h_req[i], non_blocking=True)
            sh.submit(dqs[i], drs[i], ready_stream=s_in.cuda_stream)
            if i >= 1:                                        # tick i-1's results are on their way
                sh.wait_tick(1, s_out)
                with torch.cuda.stream(s_out):
                    h_res[copied].copy_(drs[copied], non_blocking=True)
                copied += 1
        sh.finish()
        s_out.wait_stream(stream)
        with torch.cuda.stream(s_out):
            while copied < K:
                h_res[copied].copy_(drs[copied], non_blocking=True)
                copied += 1
        stream.wait_stream(s_out)
        torch.cuda.synchronize()
        dist.barrier()
        t_b = time.perf_counter()
        tt = torch.tensor([t_b - t_a], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": world * K * TICK / float(tt.item()), "unit": UNIT, "h2d_bytes_per_step": TICK * 48,
               "d2h_bytes_per_step": TICK * 32,
               "api": "per rank: pinned host -> H2D -> sharded submit (partition + route over NVLink, decide, results "
                      "back, unpermute) -> D2H to pinned host, copies on their own streams"}

    clocks = sampler.stop() if rank == 0 else None

    # ---------------------------------------------------------------- oracle: parity + CPU baseline
    cpu = parity = None
    if not args.no_cpu:
        import oracle
        if world == 1:
            # the WHOLE trace -- warm pass and every tick the engine ran (warm-up and timed) -- through ONE reference
            # store, one request at a time; the tick part is the timed single-thread CPU baseline
            sto = oracle.OracleStore(oracle.ADAPTIVE, capacity=n_keys, created_ns=traces.T0)
            sto.replay(traces.warm_pass(n_keys))
            t_a = time.perf_counter()
            want = sto.replay(tr)
            sec = time.perf_counter() - t_a
            got = res_all.reshape(-1)
            a = want.view(np.uint8).reshape(len(want), -1)
            b = got.view(np.uint8).reshape(len(got), -1)
            bad = np.nonzero((a != b).any(axis=1))[0]
            parity = {"checked_rows": int(len(want)), "mismatches": int(len(bad)),
                      "scope": "full trace: %d-key warm pass + all %d ticks (warm-up and timed) vs one oracle store"
                               % (n_keys, W + K)}
            if len(bad):
                i = int(bad[0])
                parity["first_mismatch"] = {"row": i, "oracle": str(want[i]), "engine": str(got[i])}
            cpu = {"value": len(tr) / sec, "unit": UNIT, "cores": 1, "kind": "port",
                   "sample": "C++ restatement of throttlecrab AdaptiveStore + RateLimiter (Rust toolchain unavailable), "
                             "string keys, 1 thread: %d-key warm pass (untimed) + %d Zipf ticks of 2^20 requests timed "
                             "(%.1f s)" % (n_keys, W + K, sec)}
            sto.close()
        else:
            parity = sharded_parity(tc, oracle, dist, rank, world, n_keys, n_local_keys, tr, res_all, W, K)
            # a peer-memory wait that gave up (a rank never delivered a tick) raises a flag in the rank's window
            try:
                gave_up = sh.error() if hasattr(sh, "error") else 0
            except Exception:
                gave_up = -1
            flag = torch.tensor([gave_up], dtype=torch.int32, device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MAX)
            if parity is not None:
                parity["peer_wait_gave_up"] = int(flag.item())

    # ---------------------------------------------------------------- K2 (N=1)
    sweep = None
    if world == 1 and rank == 0 and not args.no_sweep:
        try:
            store.close()
            del d_req, d_res
            torch.cuda.empty_cache()
            sweep = sweep_block(tc, peak, local_rank)
        except Exception as ex:
            sweep = {"error": repr(ex)}

    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return
    alg_bytes = 112.0 * n_allowed + 96.0 * (K * TICK - n_allowed)
    roof = None
    if world == 1:
        t_k1 = total_ms * 1e-3
        ach = alg_bytes / t_k1 / 1e9
        traffic, traffic_src = traffic_from_profiles()
        d_idx = stats1["index_batches"] - stats0["index_batches"]
        roof = {"bound": "hbm",
                "kernel": "K1, all kernels of a tick (index-order pipeline: probe | decide in batch order + resolve | sorted "
                          "residue on three streams; sort pipeline: ingest + radix sort | decide)",
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "peak_kind": peak_kind,
                "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes_per_tick": alg_bytes / K,
                "algorithmic_bytes_per_decision": {"allowed": 112, "denied": 96},
                "ticks_on_index_order_pipeline": d_idx, "ticks_on_sort_pipeline": K - d_idx,
                "residue_fraction": ((stats1["residue_rows"] - stats0["residue_rows"])
                                     / max(stats1["residue_batches"] - stats0["residue_batches"], 1)) / TICK,
                "pipeline_drains": stats1["drains"] - stats0["drains"],
                "serial_tick_phase_ms": {"total": phases[0], "stage1": phases[1], "stage2": phases[2], "stage3": phases[3]},
                "serial_tick_detail_ms": phase_detail}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int64", "data": "synthetic",
        "config": {"workload": ("10M keys, Zipf-1.0 request stream, ticks of 2^20 requests (BASELINE configs[1])"
                                if world == 1 else
                                "%dM keys hash-sharded over %d GPUs, Zipf-1.0 stream, 2^20 requests per GPU per tick "
                                "(BASELINE configs[4] shape)" % (n_keys // 1_000_000, world)),
                   "sharded_pipeline": (None if world == 1 else sh.describe()),
                   "keys": n_keys, "tick": TICK, "request_bytes": 48, "result_bytes": 32,
                   "l2": "no flush: table %.2f GB and a distinct 80 MB tick per step exceed the 126 MB L2"
                         % (stats1["table_slots"] * 32 / 1e9),
                   "allowed_fraction": n_allowed / max(n_ok, 1), "gen_seconds": round(gen_s, 1)},
        "host_enqueue_ms_per_step": {"min": min(step_ms), "median": float(np.median(step_ms)), "max": max(step_ms)},
        "roofline": roof, "sweep": sweep, "sustained": sustained, "parity": parity, "cpu_baseline": cpu, "e2e": e2e,
        "gpu_launches": int(launches), "clocks": clocks,
    }
    print(json.dumps(line), flush=True)
    if dist:
        dist.destroy_process_group()


def sharded_parity(tc, oracle, dist, rank, world, n_keys, n_local_keys, tr, res_all, W, K, n_ticks=4):
    """N>1: keys are independent, so ONE oracle store replaying every request of a key subset -- in global
    order: tick by tick, rank 0's rows before rank 1's -- must reproduce the engine's rows for those keys
    exactly.  Subset: the 4 hottest keys (they span all ranks and test the cross-rank order), 64 keys of middle
    rank, 3000 sampled cold keys; ticks: the first `n_ticks` the engine ran (their history is complete)."""
    P = min(n_ticks, W + K)
    ranks = np.concatenate([np.arange(4), np.arange(1000, 1064),
                            1064 + (traces.stream(9, 0, 3000) % np.uint64(n_keys - 1064))]).astype(np.uint64)
    keys = np.unique(traces.rank_to_key(ranks, n_keys))
    padded = np.array([(r + 1) * n_local_keys - 1 for r in range(world)], np.uint64)   # warm-pass padding keys
    keys = np.setdiff1d(keys, padded)
    rows = tr[:P * TICK]
    mask = np.isin(rows["key"], keys)
    mine = (rows[mask], res_all[:P].reshape(-1)[mask], (np.nonzero(mask)[0] // TICK).astype(np.int32))
    gathered = [None] * world if rank == 0 else None
    dist.gather_object(mine, gathered, dst=0)
    if rank != 0:
        return None
    sto = oracle.OracleStore(oracle.PERIODIC, capacity=len(keys) * 2, created_ns=traces.T0, p0=10**9)
    w = np.zeros(len(keys), traces.REQ_DTYPE)
    w["key"] = keys
    traces.fill_policy(w, (keys % np.uint64(8)).astype(np.int64))
    w["quantity"] = 1
    w["now_ns"] = traces.T0
    sto.replay(w)
    checked = bad = 0
    first = None
    for t in range(P):
        req_t = np.concatenate([g[0][g[2] == t] for g in gathered])        # rank order = global order inside a tick
        got_t = np.concatenate([g[1][g[2] == t] for g in gathered])
        want_t = sto.replay(req_t)
        a = want_t.view(np.uint8).reshape(len(want_t), -1)
        b = got_t.view(np.uint8).reshape(len(got_t), -1)
        m = np.nonzero((a != b).any(axis=1))[0]
        checked += len(req_t)
        bad += len(m)
        if len(m) and first is None:
            i = int(m[0])
            first = {"tick": t, "oracle": str(want_t[i]), "engine": str(got_t[i]), "request": str(req_t[i])}
    sto.close()
    out = {"checked_rows": int(checked), "mismatches": int(bad),
           "scope": "%d keys (4 hottest, 64 of middle rank, sampled cold) over the first %d ticks of all %d ranks, "
                    "in global order, vs one oracle store" % (len(keys), P, world)}
    if first:
        out["first_mismatch"] = first
    return out


if __name__ == "__main__":
    main()
