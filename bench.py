#!/usr/bin/env python
"""bench.py -- requests/sec (+ p50/p99 latency) of the b200 hot path on BASELINE.json configs[1]:
synthetic 1000-tree x depth-6 XGBoost-semantics regressor, 32 float32 features, max_batch=64.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A STEP = one pass of the hot path over one scheduler batch of 64 single-row requests.
  value   device-resident: the batch is already in HBM; one forest kernel launch per step, timed with
          CUDA events on the launching stream, L2 flushed before every timed step
  e2e     the same batch through the C ABI with HOST buffers: b2s_infer_batch (collate into the pinned
          slot, H2D, kernel, result written back to the host) + b2s_event_wait (scatter to the 64
          per-request buffers), wall clock, up to 4 batches in flight
  Every forest leg times exactly K steps, once, after an untimed warm-up in its own step form (>= W steps and
  >= WARMUP_MIN_S); step k reads input set k % 64, so the inputs of the last timed step depend on K alone, and
  --dump-outputs DIR writes what that step of `value` returned.  A small K is a noisy figure (a 20-step region of this
  workload is 0.3 ms).
  plugin  the metric BASELINE.json names, through the reference-facing plugin API
          (B200PreprocessRequest.process under asyncio): closed-loop req/s and open-loop Poisson
          (lambda = 2000 req/s) p50/p99 latency
  roofline / cpu_baseline: see DESIGN.md ("Measurement")
N > 1: one process per GPU, independent replicas (requests are independent: no data-path collective,
weak scaling); NCCL only for the timing barrier / max-over-ranks reduction.
"""
import argparse
import asyncio
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_TREES, DEPTH, N_FEATURES, MAX_BATCH = 1000, 6, 32, 64
WORKLOAD = "xgboost-synth-1000trees-depth6-32feat-f32_maxbatch64"
WORKLOAD_MIN_STEPS = 200     # BERT / ResNet sections: timed steps whatever --steps says (2.6-3 ms each: >= 0.5 s per leg)
# batches in flight in the BERT / ResNet e2e loops = the staging slots of an endpoint stream (BatchPolicy.n_slots default): with 2,
# the ResNet loop ran at 3.38 ms per batch against 2.93 ms on the device (collate + H2D of batch k+2 not hidden); 3: 2.96; 4: 2.74
WORKLOAD_E2E_DEPTH = int(os.environ.get("B2S_BENCH_E2E_DEPTH", "4"))
MIN_TIMED_S, MIN_REPEATS, MAX_LEG_WALL_S = 0.5, 5, 25.0
# a single K-step region timed right after a 50-step warm-up ran the e2e leg 25 % slower than the steady state
# (B200, 1000 W power limit, K = 500)
WARMUP_MIN_S = 0.5


def _config():
    """the `config` object: identical in both arms (the driver compares them)"""
    return dict(workload=WORKLOAD, step="one scheduler batch of 64 single-row requests", max_batch=MAX_BATCH,
                n_trees=N_TREES, depth=DEPTH, n_features=N_FEATURES,
                timing="exactly K timed steps (--steps), one region, after an untimed warm-up",
                l2="GPU arm: flushed (256 MiB memset on the launching stream) before every timed step of `value`")


def _repeat_region(region, min_timed_s=MIN_TIMED_S, min_repeats=MIN_REPEATS, max_wall_s=MAX_LEG_WALL_S):
    """region() -> seconds of TIMED work of one K-step region.  Returns (median, all samples)."""
    samples, total, t0 = [], 0.0, time.perf_counter()
    while len(samples) < min_repeats or total < min_timed_s:
        dt = float(region())
        samples.append(dt)
        total += dt
        if time.perf_counter() - t0 > max_wall_s and len(samples) >= min_repeats:
            break
    return float(np.median(samples)), samples


def _warm_up(run, n):
    """Untimed warm-up of a leg in its own step form: run(n) runs n steps; repeated until WARMUP_MIN_S have passed, so
    that clocks and host caches have settled before the leg's K timed steps, whatever W is."""
    t0 = time.perf_counter()
    run(n)
    while time.perf_counter() - t0 < WARMUP_MIN_S:
        run(n)


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def _traffic_bytes():
    """dram bytes per launch of the dominant kernel from the committed ncu capture, or None."""
    p = os.path.join(ROOT, "profiles", "forest_traffic.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                return json.load(f).get("dram_bytes_per_launch")
        except Exception:  # noqa
            return None
    return None


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown," \
        "clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.proc = None
        self.lines = []
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self, keep_busy=None):
        """`keep_busy()`: re-runs the timed kernel; called while no sample has arrived yet (nvidia-smi can take longer to
        print its first line than the timed region lasts), so that the clocks reported are clocks under this load."""
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        deadline = time.time() + 3.0
        while len(self.lines) < 2 and time.time() < deadline:
            if keep_busy is not None:
                keep_busy()
            else:
                time.sleep(0.05)
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def _dist_setup(n_gpus):
    """One process per GPU (torchrun).  NCCL on the GPU box; B2S_DIST_BACKEND=gloo lets the same code
    path run on CPU (tests/test_multi_rank_cpu.py, world_size 2)."""
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        backend = os.environ.get("B2S_DIST_BACKEND", "nccl")
        if backend == "nccl":
            torch.cuda.set_device(local)
            dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local))
        else:
            dist_mod.init_process_group(backend)
        dist = dist_mod
    return rank, world, local, dist


def _dist_device(dist, local):
    return "cuda:%d" % local if dist.get_backend() == "nccl" else "cpu"


def _barrier_sync(dist, local):
    if dist is not None:
        import torch
        dist.barrier()
        if dist.get_backend() == "nccl":
            torch.cuda.synchronize(local)


def _max_over_ranks(dist, local, x):
    if dist is None:
        return float(x)
    import torch
    t = torch.tensor([float(x)], device=_dist_device(dist, local), dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _sum_over_ranks(dist, local, x):
    if dist is None:
        return float(x)
    import torch
    t = torch.tensor([float(x)], device=_dist_device(dist, local), dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


def _dump_outputs(out_dir, **arrays):
    """--dump-outputs: each array as <out_dir>/<name>.npy (float32 / float64), for output-for-output comparison of
    two builds run with the same arguments"""
    if not out_dir:
        return
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def whole_job_value(world, units_per_rank_per_step, steps, max_seconds):
    """`value` of the contract: units all ranks processed / the slowest rank's time (weak scaling)."""
    return world * units_per_rank_per_step * steps / max_seconds


def _make_model():
    from oracle import oracle as orc
    forest = orc.synth_xgb_forest(n_trees=N_TREES, depth=DEPTH, n_features=N_FEATURES, seed=0)
    return forest


def _cpu_pick_threads(h, X, out, n_procs):
    """The reference arm may use every host thread; an OpenMP team larger than the 64 rows of a batch (or than the
    box's CPU quota) only adds fork/join cost.  Fixed sweep: every candidate team size runs for 0.3 s (after 0.1 s of
    warm-up: the OpenMP pool resizes lazily), the two fastest are re-timed for 1 s each and the winner of THAT decides
    (a 0.15 s picker made the CPU arm swing 3x between boxes in round 1).  Returns (threads, {team size: req/s})."""
    cands = sorted(set(c for c in (1, 2, 4, 8, 16, 32, 64, n_procs) if 1 <= c <= max(1, min(n_procs, MAX_BATCH))))

    def rate(c, seconds):
        t_end = time.perf_counter() + 0.1
        while time.perf_counter() < t_end:
            h.predict_xgb_into(X[0], 0.5, out, c)
        t0, reps = time.perf_counter(), 0
        while time.perf_counter() - t0 < seconds:
            h.predict_xgb_into(X[reps % 256], 0.5, out, c)
            reps += 1
        return reps * MAX_BATCH / (time.perf_counter() - t0)
    sweep = {c: rate(c, 0.3) for c in cands}
    finalists = sorted(sweep, key=sweep.get, reverse=True)[:2]
    final = {c: rate(c, 1.0) for c in finalists}
    best = max(final, key=final.get)
    sweep.update(final)
    return best, sweep


def _cpu_loop(forest, steps, warmup=3):
    """The oracle port (no compiled reference exists: clearml-serving is pure Python and xgboost is not installable) on
    the host cores: one step = one batch of 64 rows, OpenMP over rows with the fastest team size the box offers.
    Returns (region, out, threads, n_procs, sweep): region() times `steps` steps, step k on input set k % 256, and
    leaves the last step's predictions in `out`."""
    from oracle import oracle as orc
    h = orc.ForestHandle(forest)
    n_procs = orc.max_threads()
    rng = np.random.default_rng(1)
    X = rng.standard_normal((256, MAX_BATCH, N_FEATURES)).astype(np.float32)
    out = np.empty(MAX_BATCH, np.float32)
    threads, sweep = _cpu_pick_threads(h, X, out, n_procs)
    for w in range(warmup):
        h.predict_xgb_into(X[w % 256], 0.5, out, threads)

    def region():
        t0 = time.perf_counter()
        for k in range(steps):
            h.predict_xgb_into(X[k % 256], 0.5, out, threads)
        return time.perf_counter() - t0
    return region, out, threads, n_procs, sweep


def _cpu_baseline(forest, seconds):
    """comparison leg, independent of --steps: its 200-step region is repeated (_repeat_region), median region"""
    steps = 200
    region, _out, threads, n_procs, sweep = _cpu_loop(forest, steps)
    med, samples = _repeat_region(region)
    reps = len(samples)
    return dict(value=steps * MAX_BATCH / med, unit="requests/s", cores=int(threads), kind="port",
                sample="median of {} regions of {} batches x {} rows; oracle/forest_oracle.c (restatement of the xgboost "
                       "CPU predictor), OpenMP over rows, team size {} of {} host threads (fixed sweep, finalists re-timed "
                       "for 1 s)".format(reps, steps, MAX_BATCH, threads, n_procs),
                team_sweep_req_s={str(k): round(v) for k, v in sorted(sweep.items())})


def _reference_python_path(seconds):
    """`cpu_baseline_ref` (kind "ref"): the REFERENCE'S OWN code -- ModelRequestProcessor.process_request ->
    _process_request -> SKLearnPreprocessRequest.process -> sklearn predict (model_request_processor.py:253-304,
    1309-1369; preprocess_service.py:459-464) -- imported under stubs from baseline/_ref (or /root/reference), on a
    GradientBoostingRegressor of the configs[1] shape (the xgboost engine itself cannot run: not installable), with
    p50 / p99 per request; and the same for configs[0] (LogisticRegression on iris, batch 1)."""
    from oracle import ref_bench as rb
    from oracle import ref_harness as rh
    if not rh.available():
        return dict(unavailable="reference package not found (baseline/_ref is created by __graft_entry__.build() "
                                "where /root/reference exists)")
    out = dict(kind="ref", cores=1, source=rh.REFERENCE_ROOT,
               path="ModelRequestProcessor.process_request -> SKLearnPreprocessRequest.process (reference code, stubs for "
                    "clearml / vllm imports), JSON-dict bodies, serial closed loop in one process")
    t0 = time.perf_counter()
    gbr = rb.fit_cfg2_gbr()
    out["gbr_fit_s"] = round(time.perf_counter() - t0, 1)
    out["gbr_matches_golden_bitwise"] = rb.golden_check(gbr)
    for name, kind, model in (("cfg2_gbr_1000x6x32", "trees", gbr), ("cfg1_lr_iris", "iris", rb.fit_iris_lr())):
        _ref, proc, url = rb.make_reference_processor(model, kind)
        _X, bodies = rb.bodies_for(kind)
        res, _reply = rb.closed_loop(proc, url, bodies, seconds)
        n_proc = max(1, min(8, (os.cpu_count() or 2) // 2))
        try:
            mp = rb.multi_process(kind, model, n_proc, min(seconds, 3.0))
        except Exception as ex:  # noqa
            mp = dict(error="{}: {}".format(type(ex).__name__, ex))
        out[name] = dict(value=res["req_s"], unit="requests/s", p50_us=res["p50_us"], p99_us=res["p99_us"],
                         completed=res["completed"], sample="{:.1f} s closed loop".format(seconds), multi_process=mp)
    return out, gbr


def _b200_same_models(gbr, device, seconds=2.0):
    """The b200 plugin on the SAME two models the reference path was timed on (fp64 forest of the GBR; the iris
    LogisticRegression, which BASELINE configs[0] calls "plumbing, no GPU" -- here it is the linear kernel), same
    JSON-dict bodies through a user Preprocess class, replies compared with sklearn's own predictions."""
    from clearml_serving_b200 import BasePreprocessRequest, ModelEndpoint, formats
    from clearml_serving_b200.model_request_processor import ModelRequestProcessor
    from oracle import ref_bench as rb
    cls = BasePreprocessRequest.get_engine_cls("b200")
    out = {}
    for name, kind, model, pre in (("cfg2_gbr_1000x6x32", "trees", gbr, rb._TreePreprocess()),
                                   ("cfg1_lr_iris", "iris", rb.fit_iris_lr(), rb._IrisPreprocess())):
        X, bodies = rb.bodies_for(kind)
        want = model.predict(X)
        p = ModelRequestProcessor()
        ep = ModelEndpoint(engine_type="b200", serving_url="same", auxiliary_cfg={"max_batch_size": MAX_BATCH, "b200.device": device})
        eng = cls.__new__(cls)
        BasePreprocessRequest.__init__(eng, model_endpoint=ep, task=None)
        eng._model = formats.pack_sklearn(model)
        eng._b200_setup()
        eng._preprocess = pre
        p._endpoints["same"] = ep
        p._engine_processor_lookup["same"] = eng
        lat, bad = [], [0]

        async def closed(conc, secs):
            stop = time.perf_counter() + secs
            n = [0]

            async def worker(w):
                i = w
                while time.perf_counter() < stop:
                    t = time.perf_counter()
                    r = await p.process_request(base_url="same", version=None, request_body=bodies[i % len(bodies)], serve_type="process")
                    lat.append(time.perf_counter() - t)
                    if r["y"][0] != want[i % len(bodies)]:
                        bad[0] += 1
                    i += conc
                    n[0] += 1
            t0 = time.perf_counter()
            await asyncio.gather(*[worker(w) for w in range(conc)])
            return n[0] / (time.perf_counter() - t0)
        try:
            asyncio.run(closed(8, 0.3))
            lat.clear(); bad[0] = 0
            serial = asyncio.run(closed(1, seconds))           # one request in flight: the latency the reference figure is
            a = np.asarray(lat) * 1e6
            res = dict(serial=dict(value=serial, unit="requests/s", p50_us=float(np.percentile(a, 50)), p99_us=float(np.percentile(a, 99))))
            lat.clear()
            conc = asyncio.run(closed(256, seconds))
            a = np.asarray(lat) * 1e6
            res["concurrency_256"] = dict(value=conc, unit="requests/s", p50_us=float(np.percentile(a, 50)), p99_us=float(np.percentile(a, 99)))
            res["mismatched_vs_sklearn"] = bad[0]
            out[name] = res
        finally:
            p.shutdown()
    return out


def run_reference(args):
    # rank 0 alone runs the CPU arm; the other ranks exit 0 without work (no process group needed)
    if int(os.environ.get("RANK", 0)) != 0:
        return
    forest = _make_model()
    W = max(args.warmup, 3)
    region, out, threads, n_procs, sweep = _cpu_loop(forest, args.steps, warmup=W)
    secs = region()
    _dump_outputs(args.dump_outputs, forest_predictions=out)
    value = args.steps * MAX_BATCH / secs
    line = dict(metric="requests/sec", value=value, unit="requests/s", n_gpus=args.gpus, steps=args.steps,
                warmup=W, ms_per_step=secs / args.steps * 1e3, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f32", data="synthetic", impl="reference",
                config=_config(),
                cpu_baseline=dict(value=value, unit="requests/s", cores=int(threads), kind="port",
                                  sample="one region of {} steps x {} rows; oracle port of the xgboost CPU predictor, "
                                         "OpenMP over rows, team size {} of {} host threads (fixed sweep, finalists re-timed "
                                         "for 1 s)".format(args.steps, MAX_BATCH, threads, n_procs),
                                  team_sweep_req_s={str(k): round(v) for k, v in sorted(sweep.items())}),
                e2e=dict(value=value, unit="requests/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


def _plugin_metrics(forest, device, seconds=2.0, lam=2000.0):
    """requests/s + latency through B200PreprocessRequest.process (the reference-facing plugin API)."""
    from clearml_serving_b200 import BasePreprocessRequest, ModelEndpoint, formats
    packed = formats.pack_forest(forest, "xgb", base=0.5)
    cls = BasePreprocessRequest.get_engine_cls("b200")

    def make_engine(delay_us):
        ep = ModelEndpoint(engine_type="b200", serving_url="bench_xgb",
                           auxiliary_cfg={"max_batch_size": MAX_BATCH, "dynamic_batching.max_queue_delay_microseconds": delay_us,
                                          "b200.device": device})
        e = cls.__new__(cls)
        BasePreprocessRequest.__init__(e, model_endpoint=ep, task=None)
        e._model = packed
        e._b200_setup()
        return e
    eng = make_engine(1000)
    rng = np.random.default_rng(3)
    X = rng.standard_normal((4096, 1, N_FEATURES)).astype(np.float32)
    out = {}

    async def closed_loop(conc):
        stop = time.perf_counter() + seconds
        count = 0

        async def worker(w):
            nonlocal count
            i = w
            while time.perf_counter() < stop:
                await eng.process(X[i % 4096], {}, None)
                i += conc
                count += 1
        t0 = time.perf_counter()
        await asyncio.gather(*[worker(w) for w in range(conc)])
        return count / (time.perf_counter() - t0)

    async def open_loop():
        loop = asyncio.get_running_loop()
        n = int(lam * seconds)
        gaps = np.random.default_rng(2).exponential(1.0 / lam, n)
        lat = []
        pending = []

        async def one(i):
            t = time.perf_counter()
            await eng.process(X[i % 4096], {}, None)
            lat.append(time.perf_counter() - t)
        t_next = loop.time()
        for i in range(n):
            t_next += gaps[i]
            delay = t_next - loop.time()
            if delay > 0:
                await asyncio.sleep(delay)
            pending.append(asyncio.ensure_future(one(i)))
        await asyncio.gather(*pending)
        lat = np.asarray(lat) * 1e6
        return dict(offered_req_s=lam, completed=n, p50_us=float(np.percentile(lat, 50)),
                    p99_us=float(np.percentile(lat, 99)), mean_us=float(lat.mean()))
    try:
        asyncio.run(closed_loop(64))  # warm-up
        out["closed_loop_req_s"] = asyncio.run(closed_loop(256))
        out["closed_loop_concurrency"] = 256
        out["poisson"] = asyncio.run(open_loop())
        st = eng.engine_stats()
        out["mean_batch_rows"] = st["mean_batch_rows"]
        out["policy"] = repr(eng._policy)
    finally:
        eng.unload()
    # the same arrival process with Triton's default queue delay (0: dispatch whatever is queued as soon as a lane is
    # free): the latency floor of the path, without the 1 ms the policy above spends waiting for batch-mates
    eng = make_engine(0)
    try:
        asyncio.run(closed_loop(16))  # warm-up
        out["poisson_no_queue_delay"] = asyncio.run(open_loop())
        out["poisson_no_queue_delay"]["mean_batch_rows"] = eng.engine_stats()["mean_batch_rows"]
    finally:
        eng.unload()
    return out


def rest_load(app, path, bodies, headers, seconds=2.0, concurrency=64, check=None):
    """Level L1 of SURVEY.md 8(d): the FastAPI app behind uvicorn on 127.0.0.1, an aiohttp closed-loop client in the same
    process (no `ab` / `wrk` in the image).  `bodies`: request payloads (bytes) cycled by the workers.  Returns requests/s,
    p50 / p99 latency and the count of non-200 replies; `check(reply bytes, body index)` may assert on every reply."""
    import socket
    import threading

    import aiohttp
    import uvicorn
    sock = socket.socket()
    sock.bind(("127.0.0.1", 0))
    port = sock.getsockname()[1]
    sock.close()
    server = uvicorn.Server(uvicorn.Config(app, host="127.0.0.1", port=port, log_level="error", access_log=False))
    th = threading.Thread(target=server.run, name="b2s-rest-bench", daemon=True)
    th.start()
    t_wait = time.time() + 10.0
    while not server.started and time.time() < t_wait:
        time.sleep(0.01)
    if not server.started:
        raise RuntimeError("uvicorn did not start")
    url = "http://127.0.0.1:{}{}".format(port, path)
    lat, bad, wrong = [], [0], [0]

    async def run():
        async with aiohttp.ClientSession(connector=aiohttp.TCPConnector(limit=concurrency),
                                         timeout=aiohttp.ClientTimeout(total=20)) as session:
            async def one(i):
                t = time.perf_counter()
                async with session.post(url, data=bodies[i % len(bodies)], headers=headers) as r:
                    payload = await r.read()
                    if r.status != 200:
                        bad[0] += 1
                    elif check is not None:
                        try:
                            ok = check(payload, i % len(bodies))
                        except Exception:  # noqa
                            ok = False
                        if ok is False:
                            wrong[0] += 1
                lat.append(time.perf_counter() - t)
            for i in range(min(concurrency, 32)):   # warm-up: connections, first batches
                await one(i)
            lat.clear()
            bad[0] = wrong[0] = 0
            stop = time.perf_counter() + seconds

            async def worker(w):
                i = w
                while time.perf_counter() < stop:
                    await one(i)
                    i += concurrency
            t0 = time.perf_counter()
            await asyncio.gather(*[worker(w) for w in range(concurrency)])
            return time.perf_counter() - t0
    try:
        elapsed = asyncio.run(run())
    finally:
        server.should_exit = True
        th.join(timeout=10)
    a = np.asarray(lat) * 1e6
    return dict(req_s=len(lat) / elapsed, p50_us=float(np.percentile(a, 50)), p99_us=float(np.percentile(a, 99)),
                completed=len(lat), failed=bad[0], mismatched=wrong[0], concurrency=concurrency, server="uvicorn (1 worker) + aiohttp client, same process")


def _rest_metrics(forest, device, seconds=2.0):
    """REST-level requests/s of the configs[1] endpoint: JSON bodies through a user Preprocess class (the reference's route,
    examples/xgboost) and binary tensor frames (clearml_serving_b200/wire.py), both against the real engine."""
    from clearml_serving_b200 import BasePreprocessRequest, ModelEndpoint, formats, wire
    from clearml_serving_b200.main import create_app
    from clearml_serving_b200.model_request_processor import ModelRequestProcessor
    from oracle import oracle as orc   # the checker of the replies
    packed = formats.pack_forest(forest, "xgb", base=0.5)
    cls = BasePreprocessRequest.get_engine_cls("b200")
    rng = np.random.default_rng(5)
    X = rng.standard_normal((512, N_FEATURES)).astype(np.float32)
    want = orc.forest_predict_xgb(forest, X, 0.5)

    class _User(object):   # examples/xgboost/preprocess.py, inline
        def preprocess(self, body, state, collect_custom_statistics_fn=None):
            return np.array([[body.get("x{}".format(i)) for i in range(N_FEATURES)]], dtype=np.float32)

        def postprocess(self, data, state, collect_custom_statistics_fn=None):
            return dict(y=data.tolist())
    out = {}
    for name in ("json", "frames"):
        p = ModelRequestProcessor()
        ep = ModelEndpoint(engine_type="b200", serving_url="bench_xgb",
                           auxiliary_cfg={"max_batch_size": MAX_BATCH, "dynamic_batching.max_queue_delay_microseconds": 1000,
                                          "b200.device": device})
        eng = cls.__new__(cls)
        BasePreprocessRequest.__init__(eng, model_endpoint=ep, task=None)
        eng._model = packed
        eng._b200_setup()
        p._endpoints["bench_xgb"] = ep
        p._engine_processor_lookup["bench_xgb"] = eng
        try:
            if name == "json":
                eng._preprocess = _User()
                bodies = [json.dumps({"x{}".format(j): float(X[i, j]) for j in range(N_FEATURES)}).encode() for i in range(len(X))]
                headers = {"Content-Type": "application/json"}

                def check(payload, i):
                    return bool(np.float32(json.loads(payload)["y"][0]) == want[i])
            else:
                bodies = [wire.encode_tensors([X[i:i + 1]]) for i in range(len(X))]
                headers = {"Content-Type": wire.MEDIA_TYPE}

                def check(payload, i):
                    return bool(wire.decode_tensors(payload)[0][0] == want[i])
            out[name] = rest_load(create_app(p), "/serve/bench_xgb", bodies, headers, seconds=seconds, check=check)
        finally:
            p.shutdown()
    return out


# ------------------------------------------------------------------------------------------------
# second workload (BASELINE.json configs[3]): BERT-base fp16, mixed S in {16,64,128,256}, max_batch=64
# ------------------------------------------------------------------------------------------------
def _bert_flops(lens):
    # BASELINE.md section 3: 169.87e6*S + 36864*S^2 FLOP per sequence (linear part measured, + attention)
    return float(sum(169.87e6 * s + 36864.0 * s * s for s in lens))


def _bert_workload(native, device, steps, warmup, cpu_seconds, dist=None, local=0, world=1):
    import torch
    from transformers import BertConfig, BertForSequenceClassification
    from clearml_serving_b200 import formats
    torch.manual_seed(0)
    model_t = BertForSequenceClassification(BertConfig()).eval()
    pm = formats.pack_bert(model_t)
    model = native.Model(pm.kind, pm.blob, device=device)
    B, SMAX = 64, 256
    stream = native.Stream(model, B, SMAX, WORKLOAD_E2E_DEPTH)
    timer = native.Timer(stream)
    rng = np.random.default_rng(1)
    n_sets = 8
    sets = []
    for k in range(n_sets):
        lens = rng.choice([16, 64, 128, 256], size=B)
        reqs = []
        for n in lens:
            reqs.append([rng.integers(0, 30522, (1, n)).astype(np.int32), np.zeros((1, n), np.int32), np.ones((1, n), np.int32)])
        sets.append((lens, reqs))
    # device-resident copies
    dsets = []
    for lens, reqs in sets:
        off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        bufs = []
        for i in range(3):
            flat = np.concatenate([r[i].reshape(-1) for r in reqs])
            b = native.DeviceBuffer(flat.nbytes, device); b.upload(flat); bufs.append(b)
        doff = native.DeviceBuffer(off.nbytes, device); doff.upload(off)
        dsets.append((bufs, doff))
    d_out = native.DeviceBuffer(B * 2 * 4, device)
    for w in range(max(warmup, 3)):
        bufs, doff = dsets[w % n_sets]
        stream.infer_device(B, [b.ptr for b in bufs], [d_out.ptr], doff.ptr)
    stream.synchronize()
    launches0 = native.launch_count()
    _barrier_sync(dist, local)
    # >= 200 steps whatever --steps says: ~0.55 s of timed device work, and an e2e loop long enough to amortise pipeline fill / drain
    steps = max(steps, WORKLOAD_MIN_STEPS)
    total_ms, flops = 0.0, 0.0
    for k in range(steps):
        bufs, doff = dsets[k % n_sets]
        stream.flush_l2()
        timer.start()
        stream.infer_device(B, [b.ptr for b in bufs], [d_out.ptr], doff.ptr)
        timer.stop()
        total_ms += timer.elapsed_ms()
        flops += _bert_flops(sets[k % n_sets][0])
    launches = native.launch_count() - launches0
    _barrier_sync(dist, local)
    total_ms = _max_over_ranks(dist, local, total_ms)       # every rank runs the same sets: same FLOPs, slowest rank's time
    # e2e through the C ABI with host tensors (64 requests x 3 inputs), 2 batches in flight
    t0 = time.perf_counter()
    inflight = []
    for k in range(steps):
        if len(inflight) == WORKLOAD_E2E_DEPTH:
            item = inflight.pop(0)      # keep the output buffers alive until the scatter has run
            stream.wait(item[0])
        ev, outs, keep = stream.infer_batch(sets[k % n_sets][1])
        inflight.append((ev, outs, keep))
    for it in inflight:
        stream.wait(it[0])
    e2e_s = _max_over_ranks(dist, local, time.perf_counter() - t0)
    # parity guard on one batch (full parity lives in tests/test_gpu_bert.py)
    ev, outs, keep = stream.infer_batch(sets[0][1][:4])
    stream.wait(ev)
    with torch.no_grad():
        ref = np.concatenate([model_t(input_ids=torch.from_numpy(r[0]).long(), token_type_ids=torch.from_numpy(r[1]).long(),
                                      attention_mask=torch.from_numpy(r[2]).long()).logits.numpy() for r in sets[0][1][:4]])
    got = np.concatenate([o[0] for o in outs])
    rel = float(np.abs(got - ref).max() / np.abs(ref).max())
    # CPU arm: the same model in torch fp32 on the host cores, one request at a time (no batching in the reference)
    n_cpu, t_cpu0 = 0, time.perf_counter()
    with torch.no_grad():
        while cpu_seconds > 0 and time.perf_counter() - t_cpu0 < cpu_seconds:
            r = sets[0][1][n_cpu % B]
            model_t(input_ids=torch.from_numpy(r[0]).long(), token_type_ids=torch.from_numpy(r[1]).long(),
                    attention_mask=torch.from_numpy(r[2]).long())
            n_cpu += 1
    cpu_dt = time.perf_counter() - t_cpu0
    peak = 1431.4
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        with open(pk) as f:
            peak = float(json.load(f).get("bf16_tflops_sustained", peak))
    achieved = flops / (total_ms * 1e-3) / 1e12
    res = dict(workload="bert-base-fp16_mixedS16-256_maxbatch64_ragged", metric="sequences/sec", replicas=world,
               value=world * B * steps / (total_ms * 1e-3), ms_per_step=total_ms / steps, steps=steps,
               e2e=dict(value=world * B * steps / e2e_s, unit="sequences/s", ms_per_step=e2e_s / steps * 1e3, in_flight=WORKLOAD_E2E_DEPTH,
                        h2d_bytes_per_step=int(np.mean([sum(l) for l, _ in sets]) * 12), d2h_bytes_per_step=B * 8),
               gpu_launches_per_step=launches / steps, parity_rel_err_vs_torch_cpu_fp32=rel,
               roofline=dict(bound="tensor", achieved=achieved, peak=peak, unit="TFLOP/s", frac=achieved / peak,
                             peak_source="MEASURED_PEAKS.json bf16_tflops_sustained (kernels timed inside a step)",
                             flops_per_step_mean=flops / steps),
               cpu_baseline=dict(value=n_cpu / cpu_dt, unit="sequences/s", cores=int(torch.get_num_threads()), kind="port",
                                 sample="{} single-sequence torch fp32 forwards in {:.1f}s".format(n_cpu, cpu_dt)) if n_cpu else None)
    timer.destroy()
    for bufs, doff in dsets:
        for b in bufs:
            b.free()
        doff.free()
    d_out.free()
    stream.destroy()
    model.free()
    return res


# ------------------------------------------------------------------------------------------------
# third workload (BASELINE.json configs[2]): ResNet-50 fp16, 3x224x224, max_batch=128
# ------------------------------------------------------------------------------------------------
def _resnet_workload(native, device, steps, warmup, cpu_seconds, dist=None, local=0, world=1):
    import torch
    import torchvision
    from clearml_serving_b200 import formats
    torch.manual_seed(0)
    model_t = torchvision.models.resnet50(weights=None).eval()
    with torch.no_grad():   # trained-looking BatchNorm statistics keep activations O(1) (see tests/test_gpu_resnet.py)
        gen = torch.Generator().manual_seed(0)
        for name, m in model_t.named_modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.num_features, generator=gen) * 0.1)
                m.running_var.copy_(torch.rand(m.num_features, generator=gen) + 0.5)
                m.weight.copy_((torch.rand(m.num_features, generator=gen) * 0.5 + 0.75) * (0.3 if name.endswith("bn3") else 1.0))
                m.bias.copy_(torch.randn(m.num_features, generator=gen) * 0.1)
    pm = formats.pack_resnet(model_t)
    model = native.Model(pm.kind, pm.blob, device=device)
    B = 128
    E2E_DEPTH = WORKLOAD_E2E_DEPTH
    stream = native.Stream(model, B, 0, E2E_DEPTH)
    timer = native.Timer(stream)
    rng = np.random.default_rng(1)
    n_sets = 2
    X = [rng.standard_normal((B, 3, 224, 224)).astype(np.float32) for _ in range(n_sets)]
    d_in = []
    for x in X:
        b = native.DeviceBuffer(x.nbytes, device); b.upload(x); d_in.append(b)
    d_out = native.DeviceBuffer(B * 1000 * 4, device)
    for w in range(max(warmup, 3)):
        stream.infer_device(B, [d_in[w % n_sets].ptr], [d_out.ptr])
    stream.synchronize()
    launches0 = native.launch_count()
    _barrier_sync(dist, local)
    steps = max(steps, WORKLOAD_MIN_STEPS)      # ~0.6 s of timed device work whatever --steps says
    total_ms = 0.0
    for k in range(steps):
        stream.flush_l2()
        timer.start()
        stream.infer_device(B, [d_in[k % n_sets].ptr], [d_out.ptr])
        timer.stop()
        total_ms += timer.elapsed_ms()
    launches = native.launch_count() - launches0
    _barrier_sync(dist, local)
    total_ms = _max_over_ranks(dist, local, total_ms)
    got = d_out.download(np.float32, B * 1000).reshape(B, 1000)[:2]
    with torch.no_grad():
        ref = model_t(torch.from_numpy(X[(steps - 1) % n_sets][:2])).numpy()
    rel = float(np.abs(got - ref).max() / np.abs(ref).max())
    # e2e: 128 single-image requests per step through the C ABI (77 MB of fp32 pixels host -> device)
    reqs = [[[X[s][i:i + 1]] for i in range(B)] for s in range(n_sets)]
    e2e_steps = steps       # the 8-batch loop of round 1 spent 12 % of its time filling and draining the 2-deep pipeline
    for k in range(3):   # warm-up: first touch of the pinned slots, collate workers started
        item = stream.infer_batch(reqs[k % n_sets])   # (event, outputs, keep-alive): the scatter writes into `outputs`
        stream.wait(item[0])
    t0 = time.perf_counter()
    inflight = []
    for k in range(e2e_steps):
        if len(inflight) == E2E_DEPTH:
            item = inflight.pop(0)
            stream.wait(item[0])
        inflight.append(stream.infer_batch(reqs[k % n_sets]))
    for item in inflight:
        stream.wait(item[0])
    e2e_s = _max_over_ranks(dist, local, time.perf_counter() - t0)
    # the same requests as uint8 pixels (what an image endpoint receives: examples/pytorch/preprocess.py decodes to uint8
    # before any float conversion; the Triton client's dtype universe includes uint8, preprocess_service.py:271-282):
    # 4x fewer host->device bytes, the cast + normalisation-free stem kernel reads uint8 directly
    e2e_u8 = None
    try:
        pm8 = formats.pack_resnet(model_t, input_dtype="uint8")
        model8 = native.Model(pm8.kind, pm8.blob, device=device)
        stream8 = native.Stream(model8, B, 0, E2E_DEPTH)
        X8 = [rng.integers(0, 256, (B, 3, 224, 224)).astype(np.uint8) for _ in range(n_sets)]
        reqs8 = [[[X8[s][i:i + 1]] for i in range(B)] for s in range(n_sets)]
        for k in range(3):
            item = stream8.infer_batch(reqs8[k % n_sets])
            stream8.wait(item[0])
        t0 = time.perf_counter()
        inflight = []
        for k in range(e2e_steps):
            if len(inflight) == E2E_DEPTH:
                item = inflight.pop(0)
                stream8.wait(item[0])
            inflight.append(stream8.infer_batch(reqs8[k % n_sets]))
        for item in inflight:
            stream8.wait(item[0])
        e2e8_s = _max_over_ranks(dist, local, time.perf_counter() - t0)
        e2e_u8 = dict(value=world * B * e2e_steps / e2e8_s, unit="images/s", ms_per_step=e2e8_s / e2e_steps * 1e3, in_flight=WORKLOAD_E2E_DEPTH,
                      h2d_bytes_per_step=B * 3 * 224 * 224, d2h_bytes_per_step=B * 4000, pixels="uint8")
        stream8.destroy()
        model8.free()
    except Exception as ex:  # noqa
        e2e_u8 = dict(error="{}: {}".format(type(ex).__name__, ex))
        if world > 1:
            _max_over_ranks(dist, local, 0.0)
    n_cpu, t_cpu0 = 0, time.perf_counter()
    with torch.no_grad():
        while cpu_seconds > 0 and time.perf_counter() - t_cpu0 < cpu_seconds:
            model_t(torch.from_numpy(X[0][n_cpu % B:n_cpu % B + 1]))
            n_cpu += 1
    cpu_dt = time.perf_counter() - t_cpu0
    peak = 1431.4
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        with open(pk) as f:
            peak = float(json.load(f).get("bf16_tflops_sustained", peak))
    flops_per_img = 8.178e9   # BASELINE.md section 3 (torch FlopCounterMode, 2*MAC)
    achieved = flops_per_img * B * steps / (total_ms * 1e-3) / 1e12
    e2e_f32 = dict(value=world * B * e2e_steps / e2e_s, unit="images/s", ms_per_step=e2e_s / e2e_steps * 1e3, in_flight=WORKLOAD_E2E_DEPTH,
                   h2d_bytes_per_step=B * 3 * 224 * 224 * 4, d2h_bytes_per_step=B * 4000, pixels="float32")
    res = dict(workload="resnet50-fp16_3x224x224_maxbatch128", metric="images/sec", replicas=world,
               value=world * B * steps / (total_ms * 1e-3), ms_per_step=total_ms / steps, steps=steps,
               # an image endpoint receives uint8 pixels (examples/pytorch/preprocess.py): that is the end-to-end figure; the
               # float32 form (4x the host -> device bytes, host-memcpy bound when several ranks share a host) is kept beside it
               e2e=e2e_u8 if isinstance(e2e_u8, dict) and "value" in e2e_u8 else e2e_f32,
               e2e_float32_pixels=e2e_f32,
               gpu_launches_per_step=launches / steps, parity_rel_err_vs_torch_cpu_fp32=rel,
               roofline=dict(bound="tensor", achieved=achieved, peak=peak, unit="TFLOP/s", frac=achieved / peak,
                             peak_source="MEASURED_PEAKS.json bf16_tflops_sustained", flops_per_image=flops_per_img,
                             note="implicit GEMM (im2col-mode TMA), stem as a 4x4 convolution over the space-to-depth image; layers 1-2 are bound by fp16 activation traffic, not by the tensor pipe (DESIGN.md 5.4)"),
               cpu_baseline=dict(value=n_cpu / cpu_dt, unit="images/s", cores=int(torch.get_num_threads()), kind="port",
                                 sample="{} single-image torch fp32 forwards in {:.1f}s".format(n_cpu, cpu_dt)) if n_cpu else None)
    timer.destroy()
    for b in d_in:
        b.free()
    d_out.free()
    stream.destroy()
    model.free()
    return res


def _llama_serving_leg(eng, spec, batch, prompt_len, gen, seconds=8.0):
    """The OpenAI-route scheduler on the same engine: CONTINUOUS BATCHING over the paged KV cache (llm_service.
    ContinuousBatcher: requests join the running batch at the next iteration, leave when done).  Closed loop at `batch`
    clients (saturation) and an open-loop Poisson stream at 60 % of it: requests/s, time to first token, inter-token
    latency, end-to-end latency.  Same workload shape as the waves above (prompt 512, 128 new tokens, greedy)."""
    import threading
    from clearml_serving_b200 import llm_service as S
    b = S.ContinuousBatcher(eng, max_batch=batch, max_ctx=eng.max_ctx, chunk=4)
    rng = np.random.default_rng(7)
    prompts = [rng.integers(0, spec.vocab_size, prompt_len).astype(np.int32) for _ in range(64)]

    def one(i, rec):
        t0 = time.perf_counter()
        stamps = []

        def on_tokens(toks, finished):
            stamps.append((time.perf_counter(), len(toks)))
        f = b.submit(prompts[i % len(prompts)], gen, on_tokens)
        f.result(timeout=120)
        t1 = time.perf_counter()
        itl = []
        for (ta, _na), (tb, nb) in zip(stamps[:-1], stamps[1:]):
            itl.extend([(tb - ta) / nb] * nb)
        rec.append(dict(ttft=stamps[0][0] - t0, e2e=t1 - t0, itl=itl))

    def summarise(rec, wall):
        tt = np.array([r["ttft"] for r in rec]) * 1e3
        ee = np.array([r["e2e"] for r in rec]) * 1e3
        it = np.array([x for r in rec for x in r["itl"]]) * 1e3
        return dict(completed=len(rec), requests_per_s=len(rec) / wall, gen_tokens_per_s=len(rec) * gen / wall,
                    ttft_ms=dict(mean=float(tt.mean()), p50=float(np.percentile(tt, 50)), p99=float(np.percentile(tt, 99))),
                    itl_ms=dict(mean=float(it.mean()), p50=float(np.percentile(it, 50)), p99=float(np.percentile(it, 99))),
                    e2e_ms=dict(p50=float(np.percentile(ee, 50)), p99=float(np.percentile(ee, 99))))
    try:
        # closed loop: `batch` clients, each sends its next request when the previous one is done
        rec, stop = [], time.perf_counter() + seconds
        def client(k):
            i = k
            while time.perf_counter() < stop:
                one(i, rec)
                i += batch
        t0 = time.perf_counter()
        th = [threading.Thread(target=client, args=(k,)) for k in range(batch)]
        [t.start() for t in th]
        [t.join() for t in th]
        closed = summarise(rec, time.perf_counter() - t0)
        # open loop: Poisson arrivals at 60 % of the closed-loop rate
        lam = 0.6 * closed["requests_per_s"]
        rec2, th2 = [], []
        gaps = np.random.default_rng(2).exponential(1.0 / lam, int(lam * seconds))
        t0 = time.perf_counter()
        t_next = t0
        for i, g in enumerate(gaps):
            t_next += g
            dt = t_next - time.perf_counter()
            if dt > 0:
                time.sleep(dt)
            t = threading.Thread(target=one, args=(i, rec2))
            t.start()
            th2.append(t)
        [t.join() for t in th2]
        poisson = summarise(rec2, time.perf_counter() - t0)
        poisson["offered_requests_per_s"] = lam
        st = dict(b.stats)
        return dict(scheduler="continuous batching, paged KV (64-token pages), decode chunk 4", closed_loop=closed, poisson=poisson,
                    iterations=st["iterations"], joined_running=st["joined_running"], max_rows=st["max_rows"], pages_peak=st["pages_peak"],
                    kv_pages=b.n_pages)
    finally:
        b.close()


def _llama_workload(native, rank, world, local, dist, waves=3):
    """BASELINE.json configs[4]: Llama-3-8B bf16 random-init, prompt 512, 128 new tokens, max_batch 32, greedy.
    One GPU: TP 1.  N >= 2 (torchrun): ranks (2i, 2i+1) form tensor-parallel pairs exchanging partial sums through
    peer memory; pairs are independent replicas.  Device-timed (CUDA events on the model's stream), max over ranks."""
    from clearml_serving_b200 import llm as L
    spec = L.LlamaSpec.llama3_8b()
    batch, prompt_len, gen = 32, 512, 128
    tp = 2 if world >= 2 else 1
    group = None
    if tp == 2:
        if world % 2:
            return dict(error="tensor-parallel pairs need an even number of GPUs")
        for i in range(world // 2):   # every rank creates every pair group, in the same order
            g = dist.new_group(ranks=[2 * i, 2 * i + 1], backend="gloo")
            if rank // 2 == i:
                group = g
    tp_check = None
    if tp == 2:
        # parity of the tensor-parallel layout itself, on record in every N >= 2 run: the pair against the single-GPU run of
        # the same (small) random model -- the bf16 bar of tests/test_gpu_llm.py / scripts/llm_tp_check.py.  FATAL when it fails.
        import importlib.util
        sp = importlib.util.spec_from_file_location("llm_tp_check", os.path.join(ROOT, "scripts", "llm_tp_check.py"))
        chk = importlib.util.module_from_spec(sp)
        sp.loader.exec_module(chk)
        ok, tp_check = chk.check(rank % 2, local, group)
        if not ok:
            raise SystemExit("bench: tensor-parallel pair does not reproduce the single-GPU run: {}".format(tp_check))
    eng = L.LlmEngine(spec, device=local, max_batch=batch, max_ctx=prompt_len + gen + 16, max_tokens=batch * prompt_len,
                      tp_size=tp, tp_rank=rank % 2 if tp == 2 else 0, tp_group=group)
    eng.init_random(seed=0, std=0.02)
    rng = np.random.default_rng(1)
    prompts = [rng.integers(0, spec.vocab_size, prompt_len) for _ in range(batch)]
    m = eng.llm
    launches0 = native.launch_count()
    res, e2e = [], []
    for w in range(waves):
        _barrier_sync(dist, local)
        m.flush_l2()
        m.record(0)
        m.prefill(prompts)
        m.record(1)
        m.decode(gen - 1, use_graph=True)
        m.record(2)
        toks = m.tokens(gen)
        res.append((m.elapsed_ms(0, 1), m.elapsed_ms(1, 2)))
    launches = (native.launch_count() - launches0) // waves
    for w in range(2):   # end to end through the Python engine: host token ids in, host token ids out (wall clock)
        _barrier_sync(dist, local)
        t0 = time.perf_counter()
        out = eng.generate(prompts, gen)
        e2e.append(time.perf_counter() - t0)
    # every path must produce the same greedy tokens: the device-timed waves, the Python engine, and -- for a
    # tensor-parallel pair -- both ranks (each rank samples from the exchanged (value, index) pairs)
    # The decode GEMMs accumulate with red.global.add.f32 (stream-K): fp32 summation order is not fixed, so two runs of the
    # same wave can differ in the last bits of a logit and a near-tie of a RANDOM-INIT model's argmax can flip, after
    # which that sequence continues differently.  What must hold: (a) the first sampled token of (nearly) every
    # sequence agrees between the device-timed wave and LlmEngine.generate, (b) the two ranks of a tensor-parallel pair
    # agree EXACTLY (they sample from the same exchanged (value, index) pairs).  (a) is fatal below 90 %.
    first_equal = float(np.mean(out[:, 0] == toks[:, 0]))
    common = [int(np.argmax(np.append(out[i] != toks[i], True))) for i in range(out.shape[0])]
    agreement = dict(first_token_equal_frac=first_equal, mean_common_prefix_tokens=float(np.mean(common)), identical_sequences=int(
        sum(c == out.shape[1] for c in common)), sequences=int(out.shape[0]))
    if first_equal < 0.9:
        raise SystemExit("bench: LlmEngine.generate disagrees with the device-timed wave on the first token of {:.0%} of the "
                         "sequences (rank {})".format(1 - first_equal, rank))
    digest = int(np.asarray(out, np.int64).sum() % (1 << 31)) * 1000003 % (1 << 31) + int(np.asarray(out[:, ::7], np.int64).sum() % 1000003)
    if tp == 2:
        import torch
        t = torch.tensor([digest, -digest], dtype=torch.int64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
        if int(t[0]) != digest or int(-t[1]) != digest:
            raise SystemExit("bench: the two ranks of the tensor-parallel pair disagree on the generated tokens")
    serving = None
    if tp == 1 and world == 1:
        try:
            serving = _llama_serving_leg(eng, spec, batch, prompt_len, gen)
        except Exception as ex:  # noqa
            serving = dict(error="{}: {}".format(type(ex).__name__, ex))
    pre = _max_over_ranks(dist, local, float(np.median([r[0] for r in res[1:]])))
    dec = _max_over_ranks(dist, local, float(np.median([r[1] for r in res[1:]])))
    e2e_s = _max_over_ranks(dist, local, min(e2e))
    if tp == 2:
        dist.barrier()
    eng.close()
    replicas = world // tp
    step_ms = dec / (gen - 1)
    wbytes = (spec.n_params() - spec.vocab_size * spec.hidden_size) * 2 / tp
    kv_bytes = batch * (prompt_len + gen / 2) * spec.num_hidden_layers * 2 * spec.num_key_value_heads * spec.head_dim * 2 / tp
    pre_flops = batch * prompt_len * spec.flops_per_token() / tp
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa
        pass
    tf_peak = float(peaks.get("bf16_tflops_sustained", 1431.4) or 1431.4)   # kernels timed inside a long step
    hbm_peak, _ = _peaks()
    vllm_ref = None
    vp = os.path.join(ROOT, "profiles", "r02_vllm_tp{}.json".format(tp))
    if os.path.exists(vp):
        try:   # the comparator SURVEY.md 2.1 names: vLLM 0.22 on the same workload, measured on a B200 of this pool by
            with open(vp) as f:   # scripts/vllm_compare.py (a separate process: engine start-up + compilation take minutes)
                vllm_ref = json.load(f)
            vllm_ref["note"] = "measured separately with scripts/vllm_compare.py on a B200 of the same pool (not inside this run)"
        except Exception:  # noqa
            vllm_ref = None
    return dict(
        workload="Llama-3-8B bf16 random-init (on-device deterministic init), prompt 512 + 128 new tokens, 32 sequences per wave, greedy",
        parallelism="tp{} x {} replica(s)".format(tp, replicas), metric="requests/sec",
        kernels=dict(decode_attention="stream form (key blocks dealt to all SMs)" if os.environ.get("B2S_LLM_ATTN_STREAM", "1") != "0"
                     else "one CTA per (sequence, kv head)",
                     tp_decode_allreduce=(None if tp == 1 else {"2": "mailboxes (value = arrival flag)", "-1": "flag + peer read", "0": "arrival counts + peer read",
                                                                "1": "remote reductions"}.get(os.environ.get("B2S_LLM_TP_PUSH", "2"), "mailboxes (value = arrival flag)"))),
        value=replicas * batch / ((pre + dec) * 1e-3), gen_tokens_per_s=replicas * batch * gen / ((pre + dec) * 1e-3),
        prefill_ms=pre, decode_ms=dec, decode_step_ms=step_ms, gpu_launches_per_wave=int(launches),
        e2e=dict(value=replicas * batch / e2e_s, unit="requests/s", path="LlmEngine.generate(host token ids) -> host token ids, wall clock",
                 h2d_bytes_per_step=batch * prompt_len * 4, d2h_bytes_per_step=batch * gen * 4),
        roofline=dict(prefill=dict(bound="tensor", achieved=pre_flops / (pre * 1e-3) / 1e12, peak=tf_peak, unit="TFLOP/s",
                                   frac=pre_flops / (pre * 1e-3) / 1e12 / tf_peak),
                      decode=dict(bound="hbm", achieved=(wbytes + kv_bytes) / (step_ms * 1e-3) / 1e9, peak=hbm_peak, unit="GB/s",
                                  frac=(wbytes + kv_bytes) / (step_ms * 1e-3) / 1e9 / hbm_peak,
                                  algorithmic_bytes_per_step=int(wbytes + kv_bytes))),
        vllm_reference=vllm_ref, serving=serving, tp2_vs_tp1_check=tp_check, wave_vs_generate_agreement=agreement,
        tokens_checked="first tokens: device-timed wave vs LlmEngine.generate (fp32 atomics make later tokens of a random-init model "
                       "run-dependent)" + ("; the two ranks of every pair: exact" if tp == 2 else ""),
        cpu_baseline=None, cpu_baseline_note="the reference has no CPU path for this endpoint (it wraps vLLM)",
        waves_ms=[[round(x, 2) for x in r] for r in res])


def _router_leg(forest, world, seconds=2.0):
    """north_star's router on hardware: ONE process, `router.ReplicaSet` dealing the requests of one endpoint round-robin
    over `world` GPUs (one model copy + stream + batcher per GPU), driven through B200PreprocessRequest.process."""
    from clearml_serving_b200 import BasePreprocessRequest, ModelEndpoint, formats
    packed = formats.pack_forest(forest, "xgb", base=0.5)
    cls = BasePreprocessRequest.get_engine_cls("b200")
    ep = ModelEndpoint(engine_type="b200", serving_url="bench_router",
                       auxiliary_cfg={"max_batch_size": MAX_BATCH, "dynamic_batching.max_queue_delay_microseconds": 200,
                                      "b200.devices": list(range(world))})
    eng = cls.__new__(cls)
    BasePreprocessRequest.__init__(eng, model_endpoint=ep, task=None)
    eng._model = packed
    eng._b200_setup()
    rng = np.random.default_rng(3)
    X = rng.standard_normal((4096, 1, N_FEATURES)).astype(np.float32)
    from oracle import oracle as orc
    want = orc.forest_predict_xgb(forest, X[:, 0, :], 0.5)
    bad = [0]

    async def closed_loop(conc, secs):
        stop = time.perf_counter() + secs
        count = [0]

        async def worker(w):
            i = w
            while time.perf_counter() < stop:
                y = await eng.process(X[i % 4096], {}, None)
                if y[0] != want[i % 4096]:
                    bad[0] += 1
                i += conc
                count[0] += 1
        t0 = time.perf_counter()
        await asyncio.gather(*[worker(w) for w in range(conc)])
        return count[0] / (time.perf_counter() - t0)
    try:
        asyncio.run(closed_loop(64, 0.3))
        bad[0] = 0
        rate = asyncio.run(closed_loop(512, seconds))
        st = eng.engine_stats()
        return dict(req_s=rate, replicas=world, concurrency=512, mismatched=bad[0], per_replica_requests=st.get("per_replica_requests"),
                    mean_batch_rows=st.get("mean_batch_rows"),
                    path="one process: B200PreprocessRequest.process -> router.ReplicaSet.pick() -> per-GPU DynamicBatcher")
    finally:
        eng.unload()


def run_b200(args):
    rank, world, local, dist = _dist_setup(args.gpus)
    device = local
    from clearml_serving_b200 import formats, native
    native.ensure_init(device)
    lib = native.lib()
    forest = _make_model()
    packed = formats.pack_forest(forest, "xgb", base=0.5)
    model = native.Model(packed.kind, packed.blob, device=device)
    stream = native.Stream(model, MAX_BATCH, 0, 4)
    timer = native.Timer(stream)
    K, W = args.steps, max(args.warmup, 3)

    rng = np.random.default_rng(1)
    n_sets = 64
    Xs = rng.standard_normal((n_sets, MAX_BATCH, N_FEATURES)).astype(np.float32)

    # correctness guard: a bench of wrong results is worthless
    from oracle import oracle as orc
    ev, outs, keep = stream.infer_batch([[Xs[0][i:i + 1]] for i in range(MAX_BATCH)])
    stream.wait(ev)
    got = np.concatenate([o[0] for o in outs])
    if not np.array_equal(got, orc.forest_predict_xgb(forest, Xs[0], 0.5)):
        raise SystemExit("bench: GPU results differ from the oracle -- refusing to report numbers")

    # ---------------------------------------------------------------- value: device-resident
    d_in = [native.DeviceBuffer(Xs[0].nbytes, device) for _ in range(n_sets)]
    for b, x in zip(d_in, Xs):
        b.upload(x)
    d_out = native.DeviceBuffer(MAX_BATCH * 4, device)

    # step k of every region reads input set k % n_sets: the last timed step's inputs depend on K alone
    def cold_region(n):
        ms = 0.0
        for k in range(n):
            stream.flush_l2()                      # untimed, same stream: evict model + inputs from the 126 MB L2
            timer.start()
            stream.infer_device(MAX_BATCH, [d_in[k % n_sets].ptr], [d_out.ptr])
            timer.stop()
            ms += timer.elapsed_ms()
        return ms * 1e-3

    def warm_region():   # same launches back to back, model resident in L2 (steady-state serving)
        timer.start()
        for k in range(K):
            stream.infer_device(MAX_BATCH, [d_in[k % n_sets].ptr], [d_out.ptr])
        timer.stop()
        return timer.elapsed_ms() * 1e-3
    _warm_up(cold_region, W)

    clocks = ClockSampler(device)
    launches0 = native.launch_count()
    _barrier_sync(dist, local)
    cold_s = cold_region(K)
    stream.synchronize()
    last_out = d_out.download(np.float32, MAX_BATCH)   # what the last timed step returned
    _barrier_sync(dist, local)
    cold_s = _max_over_ranks(dist, local, cold_s)
    warm_s = _max_over_ranks(dist, local, warm_region())
    kernel_launches = native.launch_count() - launches0

    # ---------------------------------------------------------------- e2e: C ABI with host buffers
    n_req = MAX_BATCH
    tins, touts, bufs = [], [], []
    for s in range(n_sets):
        tin = (native.Tensor * n_req)()
        tout = (native.Tensor * n_req)()
        ob = np.zeros((n_req, 1), np.float32)
        for r in range(n_req):
            row = Xs[s][r:r + 1]
            tin[r].data = row.ctypes.data
            tin[r].dtype = 0
            tin[r].ndim = 2
            tin[r].shape[0], tin[r].shape[1] = 1, N_FEATURES
            tout[r].data = ob[r].ctypes.data
        tins.append(tin); touts.append(tout); bufs.append(ob)
    e2e_k = [0]

    def e2e_run(steps, depth):
        inflight = []
        t0 = time.perf_counter()
        for _ in range(steps):
            if len(inflight) == depth:
                native.check(lib.b2s_event_wait(inflight.pop(0)))
            s = e2e_k[0] % n_sets
            e2e_k[0] += 1
            ev = ctypes.c_uint64(0)
            native.check(lib.b2s_infer_batch(model.handle, stream.handle, n_req, tins[s], touts[s], ctypes.byref(ev)))
            inflight.append(ev.value)
        for ev in inflight:
            native.check(lib.b2s_event_wait(ev))
        return time.perf_counter() - t0

    _warm_up(lambda n: e2e_run(n, 4), max(W, 50))
    _barrier_sync(dist, local)
    e2e_s = _max_over_ranks(dist, local, e2e_run(K, 4))
    _warm_up(lambda n: e2e_run(n, 1), max(W, 50))
    _barrier_sync(dist, local)
    e2e_lat_s = _max_over_ranks(dist, local, e2e_run(K, 1))
    _barrier_sync(dist, local)
    launches = native.launch_count() - launches0

    def busy():   # the timed kernel again (untimed), until nvidia-smi has produced its samples
        for k in range(200):
            stream.infer_device(MAX_BATCH, [d_in[k % n_sets].ptr], [d_out.ptr])
        stream.synchronize()
    clk = clocks.stop(keep_busy=busy)
    last = (e2e_k[0] - 1) % n_sets
    if not np.array_equal(bufs[last][:, 0], orc.forest_predict_xgb(forest, Xs[last], 0.5)):
        raise SystemExit("bench: e2e results differ from the oracle")

    # ---------------------------------------------------------------- plugin-level metric (Python API)
    plugin = None
    if not args.no_plugin:
        try:
            plugin = _plugin_metrics(forest, device)
            if dist is not None:
                plugin["closed_loop_req_s_all_ranks"] = _sum_over_ranks(dist, local, plugin["closed_loop_req_s"])
        except Exception as ex:  # noqa
            plugin = dict(error=str(ex))
            if dist is not None:
                _sum_over_ranks(dist, local, 0.0)
        if local == 0 and isinstance(plugin, dict) and "error" not in plugin:
            try:   # REST level (SURVEY.md 8d L1): front-end bound by construction, reported beside the engine-level figures
                plugin["rest"] = _rest_metrics(forest, device)
            except Exception as ex:  # noqa
                plugin["rest"] = dict(error="{}: {}".format(type(ex).__name__, ex))

    # ---------------------------------------------------------------- the router: one process, `world` GPUs
    router = None
    if not args.no_plugin and rank == 0:
        try:
            router = _router_leg(forest, world)
        except Exception as ex:  # noqa
            router = dict(error="{}: {}".format(type(ex).__name__, ex))
    _barrier_sync(dist, local)

    # configs[3] / configs[2]: every rank runs a full replica (weak scaling, max over ranks)
    bert = None
    if args.bert:
        try:
            bert = _bert_workload(native, device, max(10, min(args.steps, 40)), 3, min(args.cpu_seconds, 8.0) if rank == 0 else 0.0,
                                  dist=dist, local=local, world=world)
        except Exception as ex:  # noqa
            bert = dict(error="{}: {}".format(type(ex).__name__, ex))
            if world > 1:
                raise

    resnet = None
    if args.resnet:
        try:
            resnet = _resnet_workload(native, device, max(5, min(args.steps, 20)), 3, min(args.cpu_seconds, 6.0) if rank == 0 else 0.0,
                                      dist=dist, local=local, world=world)
        except Exception as ex:  # noqa
            resnet = dict(error="{}: {}".format(type(ex).__name__, ex))
            if world > 1:
                raise

    llama = None
    if args.llama:
        try:
            llama = _llama_workload(native, rank, world, local, dist)
        except Exception as ex:  # noqa
            llama = dict(error="{}: {}".format(type(ex).__name__, ex))
            if world > 1:
                raise

    if rank == 0:
        _dump_outputs(args.dump_outputs, forest_predictions=last_out)
        peak, peak_src = _peaks()
        algo = model.algo_bytes(MAX_BATCH)
        kernel_s = cold_s / K
        achieved = algo / kernel_s / 1e9
        cpu = _cpu_baseline(forest, args.cpu_seconds) if world == 1 else None
        cpu_ref, same = None, None
        if world == 1 and not args.no_ref_path:
            try:
                r = _reference_python_path(min(args.cpu_seconds, 5.0))
                if isinstance(r, tuple):
                    cpu_ref, gbr = r
                    same = _b200_same_models(gbr, device)
                else:
                    cpu_ref = r
            except Exception as ex:  # noqa
                cpu_ref = dict(error="{}: {}".format(type(ex).__name__, ex))
        value = whole_job_value(world, MAX_BATCH, K, cold_s)
        cfg = _config()
        line = dict(
            metric="requests/sec", value=value, unit="requests/s", n_gpus=world, steps=K, warmup=W,
            ms_per_step=cold_s / K * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None,
            dtype="f32", data="synthetic", config=cfg,
            timed_region_s=dict(value=cold_s, e2e=e2e_s),
            notes=dict(l2="flushed (256 MiB memset on the launching stream) before every timed step; value_l2_warm is the "
                          "back-to-back figure", parallelism="replicas x{} (independent requests, no collective)".format(world)),
            value_l2_warm=world * MAX_BATCH * K / warm_s, ms_per_step_l2_warm=warm_s / K * 1e3,
            e2e=dict(value=world * MAX_BATCH * K / e2e_s, unit="requests/s", h2d_bytes_per_step=MAX_BATCH * N_FEATURES * 4,
                     d2h_bytes_per_step=MAX_BATCH * 4, ms_per_step=e2e_s / K * 1e3, in_flight=4,
                     ms_per_step_serial=e2e_lat_s / K * 1e3,
                     path="b2s_infer_batch(64 host tensors) + b2s_event_wait, wall clock"),
            gpu_launches=int(launches), gpu_launches_value_leg=int(kernel_launches),
            roofline=dict(bound="hbm", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak,
                          traffic=_traffic_bytes(), algorithmic_bytes_per_launch=algo, peak_source=peak_src,
                          kernel="forest_wide_kernel<f32>", note="latency-bound at 64 rows: launch + 1000-add fp32 chain (bit-exactness "
                                                             "forces the sequential sum); see DESIGN.md 5.1"),
            cpu_baseline=cpu, cpu_baseline_ref=cpu_ref, b200_same_models=same, clocks=clk, plugin=plugin, router=router,
            workloads=dict(bert_base=bert, resnet50=resnet, llama3_8b=llama))
        print(json.dumps(line))
    timer.destroy()
    for b in d_in:
        b.free()
    d_out.free()
    stream.destroy()
    model.free()
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-plugin", action="store_true")
    ap.add_argument("--no-ref-path", action="store_true", help="skip the reference-code CPU leg (cpu_baseline_ref)")
    ap.add_argument("--no-bert", dest="bert", action="store_false", help="skip the BERT-base (configs[3]) section")
    ap.add_argument("--no-resnet", dest="resnet", action="store_false", help="skip the ResNet-50 (configs[2]) section")
    ap.add_argument("--no-llama", dest="llama", action="store_false", help="skip the Llama-3-8B (configs[4]) section")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the predictions of the last timed step of `value` (64 rows, float32) to "
                         "DIR/forest_predictions.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
