#!/usr/bin/env python
"""bench.py -- sustained inferences/sec against a local CUDA-shared-memory server, and the
input-pack GB/s of the kernels behind it.

Workload (BASELINE.json configs[1], "C2"): perf_analyzer --shared-memory=cuda, densenet_onnx, one
FP32[3,224,224] input (602,112 B) per request, 1000 x FP32 output (4,000 B), concurrency 64, one
load-generation instance per GPU.  A *step* = one closed-loop round of the 64 slots = 64 completed
requests against the stand-in server (client_b200.testing.native_server: its own process per GPU,
opens the client's CUDA-IPC handles, runs the model as one batched kernel).  Client and server
share the GPU through a private CUDA MPS daemon when the box has one (stated in `config.mps`).

  value     the native generator (include/tb200_loadgen.h, `python -m client_b200.perf.loopback`):
            every request's input regenerated on the device inside its IPC region (Philox4x32-10 ->
            FP32), every response validated on the device; K timed steps (count window), repeated
            to >= 0.1 s, median repetition; all ranks start together, value = sum of requests /
            max time.
  e2e       the same metric through the tritonclient-compatible API, P free-running processes each a
            blocking client (client_b200/perf/host_loop.py): InferenceServerClient.infer ->
            check_shared_memory_region (validated on the device, verdict D2H) +
            fill_shared_memory_region (descriptor H2D, the next request's tensor generated inside the
            region), one stream wait per request.  e2e.host_tensors
            is the reference's loop line for line on the drop-in modules (numpy tensor ->
            set_shared_memory_region H2D -> infer -> get_contents_as_numpy D2H).
  --impl reference   the host-tensor loop on the restated reference code (oracle/ref_client.py: cuda-python
            cudaMemcpyAsync + sync per request, stdlib HTTP), same server, same process count.
  fill_once both arms again with regions filled once and requests only naming them (what
            perf_analyzer itself does, SURVEY.md section 10).
  roofline  the fill kernel (the dominant kernel of a step): 38,535,168 algorithmic bytes per launch /
            CUDA-event time of back-to-back launches over rotating region sets (> L2), against
            MEASURED_PEAKS.json hbm_gbs.
  generator_capacity   the device side of a step alone (fill || validate as graph replays, no server).
  cpu_baseline  the C oracle (oracle/tb200_oracle.c) doing the per-request generation + body marshal
            on one host core.

Multi-GPU: replicas only (SURVEY.md 8e) -- one server + one generator per GPU, each pinned to its
GPU's share of the local NUMA node's cores (client_b200/perf/topology.py); torch.distributed carries
the barrier, the max over ranks and the sums.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SLOTS = 64                    # concurrency
SETS = 4                      # rotating region sets (> L2)
IN_SHAPE = (3, 224, 224)
IN_BYTES = 3 * 224 * 224 * 4  # 602,112
OUT_ELEMS = 1000
OUT_BYTES = OUT_ELEMS * 4
FILL_JOB_BYTES, CHECK_JOB_BYTES, CHECK_RESULT_BYTES = 64, 48, 32  # tb200_fill_job / tb200_check_job / tb200_check_result (include/tb200.h)
SEED = 20260921
WORKLOAD = "C2 densenet_onnx FP32[3,224,224] --shared-memory=cuda concurrency=64"


def profiled_traffic(label):
    """dram read + write bytes per launch of a kernel from the committed ncu summary
    (profiles/r0N_<label>_full.txt, written by scripts/summarize_profiles.py; newest round first);
    the first kernel block of the file.  None if absent."""
    unit = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for tag in ("r02", "r01"):
        path = os.path.join(ROOT, "profiles", "%s_%s_full.txt" % (tag, label))
        try:
            total, seen = 0.0, 0
            for line in open(path):
                parts = line.split()
                if len(parts) == 3 and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and seen < 2:
                    total += float(parts[1].replace(",", "")) * unit.get(parts[2], 1)
                    seen += 1
            if seen == 2:
                return int(total)
        except OSError:
            continue
    return None


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed regions run."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device, period=0.2):
        self.period = period
        self.samples = []
        self._stop = threading.Event()
        self._thread = None
        self._device = device

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self._device), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
            except Exception:
                pass
            self._stop.wait(self.period)

    def start(self):
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=10)
        sm = sorted(int(float(s[0])) for s in self.samples if s[0].replace(".", "").isdigit())
        mx = [int(float(s[1])) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i in range(4) if s[3 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples)}


def run_b200(args):
    from client_b200 import _native
    from client_b200._native import CheckJob
    from client_b200.device import DeviceBuffer, DeviceOps, HostBuffer, make_fill_job, results_array
    import client_b200.utils.cuda_shared_memory as cudashm

    from client_b200.perf.replicas import Replicas

    rep = Replicas()
    world, rank, local = rep.world, rep.rank, rep.local_rank
    stream0 = rep.stream_base(SLOTS)  # disjoint Philox streams per replica
    ctx = _native.Context(local)
    ops = DeviceOps(ctx)
    steps, warmup = args.steps, max(args.warmup, 3)

    # --- regions: per set one input region (64 slots back to back) and one output region
    in_regions = [cudashm.create_shared_memory_region("bench_in_%d" % s, SLOTS * IN_BYTES, local) for s in range(SETS)]
    out_regions = [cudashm.create_shared_memory_region("bench_out_%d" % s, SLOTS * OUT_BYTES, local) for s in range(SETS)]
    # mock server responses: logits written once (the server is not in this loop)
    ops.fill([make_fill_job(r._base_addr, SLOTS * OUT_BYTES, "FP32", stream_id=900 + i, low=-8.0, high=8.0)
              for i, r in enumerate(out_regions)], seed=SEED)
    results = HostBuffer(SETS * SLOTS * 32)
    fill_jobs, check_jobs = [], []
    for s in range(SETS):
        fill_jobs.append((_native.FillJob * SLOTS)(*[
            make_fill_job(in_regions[s]._base_addr + k * IN_BYTES, IN_BYTES, "FP32", stream_id=stream0 + k) for k in range(SLOTS)]))
        check_jobs.append((CheckJob * SLOTS)(*[
            CheckJob(a=out_regions[s]._base_addr + k * OUT_BYTES, nbytes=OUT_BYTES, kind=_native.CHECK_TOP1) for k in range(SLOTS)]))
    ops.sync()

    # --- value: CUDA graphs of GRAPH_STEPS steps; a step = fill(64 slots, epoch advanced in-kernel)
    #     on the main branch || validate(64 outputs) on a parallel branch, rotating over the sets
    def capture(step_sets):
        ops.graph_begin()
        for s in step_sets:
            ops.fork()
            ops.check(check_jobs[s], results.device_ptr + s * SLOTS * 32)   # side branch
            ops.select(False)
            ops.fill_epoch(fill_jobs[s], seed=SEED, bump=SLOTS)             # main branch
            ops.join()
        return ops.graph_end()

    GRAPH_STEPS = 16
    ops.epoch_set(0)
    graph_many = capture([i % SETS for i in range(GRAPH_STEPS)])
    graphs_one = [capture([s]) for s in range(SETS)]

    def run_steps(n):
        for _ in range(n // GRAPH_STEPS):
            graph_many.launch()
        for i in range(n % GRAPH_STEPS):
            graphs_one[i % SETS].launch()

    sampler = ClockSampler(local, period=0.2 if world == 1 else 0.5)
    if rank == 0:  # one nvidia-smi loop per box, not one per rank
        sampler.start()
    timer = _native.Timer(ctx)
    run_steps(max(warmup, GRAPH_STEPS))
    ops.sync()
    rep.barrier()
    # generator capacity (no server): whole graphs only, at least ~100 ms of device time
    cap_steps = max(GRAPH_STEPS, (max(steps, 8000) // GRAPH_STEPS) * GRAPH_STEPS)
    timer.start()
    run_steps(cap_steps)
    timer.stop()
    ops.sync()
    rep.barrier()
    ms_cap = rep.max(timer.elapsed_ms())
    res = results_array(results, SETS * SLOTS)
    assert int(res["mismatches"].sum()) == 0, "non-finite logits reported by the validate kernel"
    cap_value = world * SLOTS * cap_steps / (ms_cap / 1e3)

    # --- roofline of the dominant kernel: fill launches only, back to back inside one graph
    reps = 4
    fill_bytes = SLOTS * IN_BYTES
    peak, peak_src = measured_peak()

    def fill_chain(launch):
        """ms per launch of `reps * SETS` back-to-back fills replayed as one graph, >= 100 ms timed"""
        ops.graph_begin()
        for r in range(reps):
            for s in range(SETS):
                launch(r, s)
        g = ops.graph_end()
        for _ in range(3):
            g.launch()
        ops.sync()
        n = 1000  # 16,000 launches of ~7 us
        timer.start()
        for _ in range(n):
            g.launch()
        timer.stop()
        ops.sync()
        ms = timer.elapsed_ms() / (n * reps * SETS)
        g.close()
        return ms, n * reps * SETS

    # the launch a device pass of the generator issues: stream epoch in the kernel parameters
    fill_ms, fill_launches = fill_chain(lambda r, s: ops.fill(fill_jobs[s], seed=SEED, epoch=(r * SETS + s) * SLOTS))
    achieved = fill_bytes / (fill_ms / 1e3) / 1e9
    # the same kernel reading the device-resident epoch (graph replays that never repeat data)
    fill_dev_ms, _ = fill_chain(lambda r, s: ops.fill_epoch(fill_jobs[s], seed=SEED, bump=SLOTS))
    _native.check(_native.load().tb200_tune(b"fill_pdl", 0))
    fill_serial_ms, _ = fill_chain(lambda r, s: ops.fill(fill_jobs[s], seed=SEED, epoch=(r * SETS + s) * SLOTS))
    _native.check(_native.load().tb200_tune(b"fill_pdl", 1))

    if os.environ.get("TB200_STEP_PARALLEL_MIN_MB"):  # experiment knob (see include/tb200.h)
        _native.check(_native.load().tb200_tune(b"step_parallel_min_mb", int(os.environ["TB200_STEP_PARALLEL_MIN_MB"])))
    # --- e2e: the same step through the public API, job tables H2D + results D2H every step
    e2e_steps = steps
    for i in range(warmup):
        ops.fill(fill_jobs[i % SETS], seed=SEED, epoch=i * SLOTS)
        ops.check(check_jobs[i % SETS], results.device_ptr + (i % SETS) * SLOTS * 32)
    ops.sync()
    rep.barrier()
    # (a) one step per call, waited for before the next one is formed
    t0 = time.perf_counter()
    timer.start()
    bad = 0
    sync_steps = max(10, e2e_steps // 4)
    for i in range(sync_steps):
        s = i % SETS
        ops.step(fill_jobs[s], check_jobs[s], results.device_ptr + s * SLOTS * 32, seed=SEED, epoch=i * SLOTS)
        bad += int(res["mismatches"][s * SLOTS:(s + 1) * SLOTS].sum())
    timer.stop()
    ops.sync()
    sync_ms = rep.max(max(timer.elapsed_ms(), (time.perf_counter() - t0) * 1e3))
    e2e_sync_value = world * SLOTS * sync_steps / (sync_ms / 1e3)
    # (b) the same steps pipelined (step_submit / step_wait, E2E_DEPTH in flight): the host copies
    #     the job tables of step i+1 while the device runs step i; every step's results are still
    #     read by the host inside the timed region, after its own wait
    E2E_DEPTH = 2
    bad_views = [res["mismatches"][s * SLOTS:(s + 1) * SLOTS] for s in range(SETS)]  # the 64 result entries of each set
    result_ptrs = [results.device_ptr + s * SLOTS * 32 for s in range(SETS)]
    rep.barrier()
    t0 = time.perf_counter()
    timer.start()
    inflight = []
    for i in range(e2e_steps):
        s = i % SETS
        inflight.append((ops.step_submit(fill_jobs[s], check_jobs[s], result_ptrs[s], SEED, i * SLOTS), s))
        if len(inflight) > E2E_DEPTH:
            ticket, s0 = inflight.pop(0)
            ops.step_wait(ticket)
            bad += int(bad_views[s0].sum())  # the host reads the step's 64 results
    for ticket, s0 in inflight:
        ops.step_wait(ticket)
        bad += int(bad_views[s0].sum())
    timer.stop()
    ops.sync()
    e2e_wall_ms = (time.perf_counter() - t0) * 1e3
    rep.barrier()
    e2e_ms = rep.max(max(timer.elapsed_ms(), e2e_wall_ms))
    assert bad == 0
    assert SETS > E2E_DEPTH  # steps in flight use different slot sets and result entries
    # what the last of these steps handed its caller: the 64 generated inputs and the 64 verdicts.
    # This loop, not the loopback generator, is dumped because its epochs depend only on the step
    # index; the generator batches requests into device passes as they happen to arrive.
    outputs = None
    if args.dump_outputs and rank == 0:
        s = (e2e_steps - 1) % SETS
        last = res[s * SLOTS:(s + 1) * SLOTS]
        outputs = {"inputs": ops.download(in_regions[s]._base_addr, SLOTS * IN_BYTES, np.float32).reshape((SLOTS,) + IN_SHAPE)}
        outputs.update({"check_" + f: last[f].astype(np.float64) for f in ("mismatches", "sum", "xor32", "argmax", "max_value")})
    api_value = world * SLOTS * e2e_steps / (e2e_ms / 1e3)
    h2d_step = SLOTS * 64 + (SLOTS + 1) * 4 + SLOTS * 48
    d2h_step = SLOTS * 32

    # --- e2e with host tensors: 64 uint8 HWC images (pinned) -> H2D -> cast+scale+CHW pack into the slots
    img_steps = max(5, min(steps, 2000))
    images = HostBuffer(SLOTS * 224 * 224 * 3)
    images.array(np.uint8)[:] = np.random.default_rng(1).integers(0, 256, SLOTS * 224 * 224 * 3, dtype=np.uint8)
    staging = DeviceBuffer(local, SLOTS * 224 * 224 * 3)
    for i in range(3):
        ops.h2d(staging.ptr, images.host_ptr, images.nbytes)
        ops.pack_image(in_regions[i % SETS]._base_addr, "FP32", "NCHW", staging.ptr, SLOTS, 224, 224, 3, "INCEPTION")
    ops.sync()
    t0 = time.perf_counter()
    for i in range(img_steps):
        s = i % SETS
        ops.h2d(staging.ptr, images.host_ptr, images.nbytes)
        ops.pack_image(in_regions[s]._base_addr, "FP32", "NCHW", staging.ptr, SLOTS, 224, 224, 3, "INCEPTION")
        ops.check(check_jobs[s], results.device_ptr + s * SLOTS * 32)
        ops.sync()
    img_ms = (time.perf_counter() - t0) * 1e3
    img_value = world * SLOTS * img_steps / (rep.max(img_ms) / 1e3)

    # --- pack kernel alone (device-resident uint8 sources, one per set so that neither the
    #     sources nor the destinations of consecutive launches are L2 hits), R+W roofline
    pack_src = [DeviceBuffer(local, SLOTS * 224 * 224 * 3) for _ in range(SETS)]
    ops.fill([make_fill_job(b.ptr, SLOTS * 224 * 224 * 3, "UINT8", stream_id=stream0 + 7200 + i) for i, b in enumerate(pack_src)], seed=SEED)
    ops.graph_begin()
    for s in range(SETS):
        ops.pack_image(in_regions[s]._base_addr, "FP32", "NCHW", pack_src[s].ptr, SLOTS, 224, 224, 3, "INCEPTION")
    gpack = ops.graph_end()
    for _ in range(3):
        gpack.launch()
    ops.sync()
    timer.start()
    for _ in range(50):
        gpack.launch()
    timer.stop()
    ops.sync()
    pack_ms = timer.elapsed_ms() / (50 * SETS)
    pack_bytes = SLOTS * (224 * 224 * 3) * (1 + 4)
    # --- C3 extras (BASELINE configs[2]): one FP16[128,3,224,224] request = 38,535,168 B
    c3_fill = [[make_fill_job(in_regions[s]._base_addr, SLOTS * IN_BYTES, "FP16", stream_id=stream0 + 7000 + s)] for s in range(SETS)]
    # the same chain as the headline roofline: 16,000 back-to-back launches, stream epoch in the parameters
    c3_fill_ms, _ = fill_chain(lambda r, s: ops.fill(c3_fill[s], seed=SEED, epoch=r * SETS + s))
    c3_src = [DeviceBuffer(local, 128 * 224 * 224 * 3) for _ in range(SETS)]
    ops.fill([make_fill_job(b.ptr, 128 * 224 * 224 * 3, "UINT8", stream_id=stream0 + 7100 + i) for i, b in enumerate(c3_src)], seed=SEED)
    ops.graph_begin()
    for s in range(SETS):
        ops.pack_image(in_regions[s]._base_addr, "FP16", "NCHW", c3_src[s].ptr, 128, 224, 224, 3, "INCEPTION")
    gc3p = ops.graph_end()
    for _ in range(3):
        gc3p.launch()
    ops.sync()
    timer.start()
    for _ in range(50):
        gc3p.launch()
    timer.stop()
    ops.sync()
    c3_pack_ms = timer.elapsed_ms() / (50 * SETS)
    c3_pack_bytes = 128 * 224 * 224 * 3 * (1 + 2)
    # --- real-image front end: 64 decoded 375x500 RGB photos -> Image.resize(224,224,BILINEAR) ->
    # FP32 CHW INCEPTION, one launch per set (image_client.preprocess after the decode)
    RS_H, RS_W = 375, 500
    rs_src = [DeviceBuffer(local, SLOTS * RS_H * RS_W * 3) for _ in range(SETS)]
    ops.fill([make_fill_job(b.ptr, SLOTS * RS_H * RS_W * 3, "UINT8", stream_id=stream0 + 7200 + i) for i, b in enumerate(rs_src)], seed=SEED)
    ops.graph_begin()
    for s in range(SETS):
        ops.resize_pack_image(in_regions[s]._base_addr, "FP32", "NCHW", rs_src[s].ptr, SLOTS, RS_H, RS_W, 3, 224, 224, "INCEPTION")
    grs = ops.graph_end()
    for _ in range(3):
        grs.launch()
    ops.sync()
    timer.start()
    for _ in range(20):
        grs.launch()
    timer.stop()
    ops.sync()
    rs_ms = timer.elapsed_ms() / (20 * SETS)
    rs_bytes = SLOTS * (RS_H * RS_W * 3 + IN_BYTES)
    # --- request-body compression on the device (HTTP Content-Encoding gzip of a generated body)
    import zlib

    dfl = []
    dfl_src = in_regions[0]._base_addr
    dfl_n = SLOTS * IN_BYTES
    dfl_cap = int(_native.load().tb200_deflate_bound(dfl_n))
    dfl_dst = DeviceBuffer(local, dfl_cap)
    for label, job in (("token ids INT64 [0,30522)", make_fill_job(dfl_src, dfl_n, "INT64", stream_id=stream0 + 7300, low=0, high=30522)),
                       ("zero data", make_fill_job(dfl_src, dfl_n, "FP32", mode="zero")),
                       ("FP32 unit interval (incompressible: stored)", make_fill_job(dfl_src, dfl_n, "FP32", stream_id=stream0 + 7301))):
        ops.fill([job], seed=SEED)
        ops.sync()
        for _ in range(2):
            ops.deflate_async(dfl_dst.ptr, dfl_cap, dfl_src, dfl_n, results.device_ptr + 3072, "gzip")
        ops.sync()
        timer.start()
        for _ in range(5):
            ops.deflate_async(dfl_dst.ptr, dfl_cap, dfl_src, dfl_n, results.device_ptr + 3072, "gzip")
        timer.stop()
        ops.sync()
        d_ms = timer.elapsed_ms() / 5
        out_bytes = int(results.array(np.uint64, 1, offset=3072)[0])
        sample = ops.download(dfl_src, 4 << 20).tobytes()  # host zlib on a 4 MB sample of the same data
        t0 = time.perf_counter()
        zl = zlib.compress(sample, 6)
        z_s = time.perf_counter() - t0
        dfl.append({"data": label, "in_bytes": dfl_n, "out_bytes": out_bytes, "ratio": round(out_bytes / dfl_n, 4), "ms": round(d_ms, 4),
                    "in_gbps": round(dfl_n / (d_ms / 1e3) / 1e9, 1), "host_zlib6_mbps": round(len(sample) / z_s / 1e6, 1),
                    "host_zlib6_ratio": round(len(zl) / len(sample), 4)})

    # ------------------------------------------------------------------------------------------
    # the north-star metric: sustained inferences/sec against the stand-in server (one per GPU)
    # ------------------------------------------------------------------------------------------
    ops.sync()
    nproc, host_cores = host_process_count(world)
    nproc_rank = max(1, nproc // world)
    lb, lb_error = {}, None
    import shutil

    want_mps = shutil.which("nvidia-cuda-mps-control") is not None and not args.no_mps
    box = None
    try:  # this rank's GPU: its own MPS daemon, its server
        box = LoopbackBox([local], use_mps=want_mps, grpc=(world == 1)).__enter__()
    except Exception as ex:
        lb_error = "%s: %s" % (type(ex).__name__, ex)
    have_mps = rep.sum(1.0 if (box is not None and box.mps) else 0.0) >= world  # every rank got its daemon
    rep.barrier()
    # every entry takes `sync`, the ranks' rendezvous between "my instance is warm" and "time now"
    plan = [("warm", lambda sync: box.generator(local, 50, 5, min_seconds=0.05, sync=sync)),
            ("value", lambda sync: box.generator(local, steps, warmup, sync=sync)),
            ("once", lambda sync: box.generator(local, steps, warmup, mode="once", sync=sync)),
            ("warm_host", lambda sync: host_loops(box, "b200", min(nproc_rank, 4), 0.5, "per-request", sync=sync)),
            ("e2e", lambda sync: host_loops(box, "b200", nproc_rank, HOST_LOOP_SECONDS, "device", sync=sync)),
            ("e2e_host", lambda sync: host_loops(box, "b200", nproc_rank, HOST_LOOP_SECONDS, "per-request", sync=sync)),
            ("e2e_once", lambda sync: host_loops(box, "b200", nproc_rank, HOST_LOOP_SECONDS, "once", sync=sync))]
    # every rank walks the same list and meets the others at exactly two barriers per entry, whatever happened
    walked, walk_error = rep.walk(plan, enabled=box is not None and lb_error is None)
    lb.update(walked)
    lb_error = lb_error or walk_error
    if box is not None and lb_error is None and world == 1 and not args.no_loopback:
        extras = {}
        for key, conc, extra in (("c1", 1, ()), ("c256", 256, ()), ("c64_one_pass_at_a_time", 64, ("--device-pipeline", "1")),
                                 ("c1_lookahead8", 1, ("--lookahead", "8")), ("c256_lookahead8", 256, ("--lookahead", "8"))):
            try:
                g = box.generator(local, 400 if conc >= 64 else 4000, 10, concurrency=conc, extra=extra, min_seconds=0.5)
                extras[key] = {k: (round(v, 1) if isinstance(v, float) else v) for k, v in g.items()
                               if k in ("concurrency", "infer_per_s", "p50_us", "p99_us", "failed", "nonfinite", "slots_per_device_pass", "pipeline_depth")}
            except Exception as ex:
                extras[key] = {"error": "%s: %s" % (type(ex).__name__, ex)}
        if box.grpc_urls.get(local):
            try:
                extras["grpc"] = _grpc_loopback_levels(box.grpc_urls[local], box.envs[local])
            except Exception as ex:
                extras["grpc"] = {"error": "%s: %s" % (type(ex).__name__, ex)}
        lb["levels"] = extras
    if box is not None:
        box.__exit__(None, None, None)
    rep.barrier()
    time_sliced = None
    if world == 1 and have_mps and not args.no_loopback and lb_error is None:
        try:  # the same run without MPS: client and server are time-sliced CUDA contexts
            with LoopbackBox([local], use_mps=False) as box:
                box.generator(local, 50, 5, min_seconds=0.05)
                g = box.generator(local, min(steps, 2000), warmup, extra=("--device-window-us", "150"), min_seconds=0.5)
                time_sliced = {"infer_per_s": round(g["infer_per_s"], 1), "p50_us": round(g["p50_us"], 1), "device_window_us": 150,
                               "slots_per_device_pass": round(g["slots_per_device_pass"], 1)}
        except Exception as ex:
            time_sliced = {"error": "%s: %s" % (type(ex).__name__, ex)}
    clocks = sampler.stop()

    any_error = rep.sum(0.0 if lb_error is None else 1.0) > 0
    if any_error and lb_error is None:
        lb_error = "another rank's loopback run failed"

    def total(key, field):
        return rep.sum(lb[key][field])

    if lb_error is None:
        v = lb["value"]
        seconds = rep.max(v["seconds"])
        value = rep.sum(v["count"]) / seconds
        gpu_launches = int(rep.sum(v["gpu_launches"]))
        once_value = rep.sum(lb["once"]["count"]) / rep.max(lb["once"]["seconds"])
        e2e_value = total("e2e", "count") / HOST_LOOP_SECONDS
        e2e_once_value = total("e2e_once", "count") / HOST_LOOP_SECONDS
        e2e_host_value = total("e2e_host", "count") / HOST_LOOP_SECONDS
        ms_step = seconds * 1e3 / (v["count"] / SLOTS)
    else:  # no server could be had: the device side alone, flagged
        value, gpu_launches, once_value, e2e_value, e2e_once_value, e2e_host_value = 0.0, 0, 0.0, 0.0, 0.0, 0.0
        ms_step = None
        v = {}

    line = {
        "metric": "inferences/sec", "value": round(value, 1), "unit": "infer/s",
        "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": round(ms_step, 6) if ms_step else None, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": common_config(have_mps, world),
        "what": "sustained inferences/sec of the native generator against the stand-in server: every request's FP32[3,224,224] input regenerated "
                "on the device inside its CUDA-IPC region, every response validated on the device; %d timed steps of %d requests per repetition, "
                "median of %s repetitions" % (steps, SLOTS, v.get("repetitions")),
        "p50_us": round(v.get("p50_us", 0.0), 1), "p99_us": round(v.get("p99_us", 0.0), 1),
        "failed": int(total("value", "failed")) if lb_error is None else None, "nonfinite": int(total("value", "nonfinite")) if lb_error is None else None,
        "slots_per_device_pass": round(v.get("slots_per_device_pass", 0.0), 1), "pipeline_depth": v.get("pipeline_depth"),
        "pinned_cpus_per_generator": v.get("cpus"), "host_cores": host_cores,
        "input_pack_gbps": round(value * IN_BYTES / 1e9, 1),
        "l2": "inputs of the kernel timings rotate over %d region sets = %d MB > 126 MB L2" % (SETS, SETS * SLOTS * IN_BYTES // 1000000),
        "e2e": {"value": round(e2e_value, 1), "unit": "infer/s", "h2d_bytes_per_step": SLOTS * (FILL_JOB_BYTES + CHECK_JOB_BYTES), "d2h_bytes_per_step": SLOTS * CHECK_RESULT_BYTES,
                "processes": nproc_rank * world, "failed_clients": int(total("e2e", "failed_workers")) if lb_error is None else None,
                "seconds": HOST_LOOP_SECONDS, "p50_us": lb.get("e2e", {}).get("p50_us"),
                "what": "tritonclient-compatible API, one blocking client per process (client_b200/perf/host_loop.py, mode 'device'): per request "
                        "http.InferenceServerClient.infer naming the regions -> cuda_shared_memory.check_shared_memory_region (validate on the device, "
                        "32-byte verdict D2H) + cuda_shared_memory.fill_shared_memory_region (job descriptor H2D, Philox fill of the next request's "
                        "tensor inside the region), one stream wait for both; free-running processes, same server.  The tensors never exist on the host: that is the path "
                        "this library replaces (reference: numpy -> set_shared_memory_region -> get_contents_as_numpy, timed by --impl reference)",
                "host_tensors": {"value": round(e2e_host_value, 1), "h2d_bytes_per_step": SLOTS * IN_BYTES, "d2h_bytes_per_step": SLOTS * OUT_BYTES,
                                 "p50_us": lb.get("e2e_host", {}).get("p50_us"),
                                 "what": "the reference arm's loop line for line on the drop-in modules: numpy Generator.random FP32[3,224,224] -> "
                                         "set_shared_memory_region (H2D) -> infer -> get_contents_as_numpy (D2H); bound by the host's random numbers "
                                         "and PCIe exactly as the reference is"}},
        "fill_once": {"value": round(once_value, 1), "e2e": round(e2e_once_value, 1), "p50_us": lb.get("once", {}).get("p50_us"),
                      "what": "regions filled once, every request only names them (perf_analyzer's own behaviour): native generator / drop-in API loop"},
        "gpu_launches": gpu_launches,
        "roofline": {"bound": "issue (FMA-heavy pipe: 18 IMAD.WIDE per 16 B), then HBM write", "kernel": "fill_uniform_kernel (Philox4x32-10 -> FP32, 64 slots per launch)",
                     "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                     "traffic": profiled_traffic("fill_uniform_kernel"),
                     "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum per launch of a steady-state launch (rotating sets, no cache control), profiles/r02_fill_uniform_kernel_full.txt",
                     "algorithmic_bytes_per_launch": fill_bytes, "ms_per_launch": round(fill_ms, 6),
                     "peak_source": peak_src, "timing": "CUDA events on the launching stream around %d back-to-back launches (graph replays of 16, stream epoch in the kernel parameters -- the launch a device pass issues)" % fill_launches,
                     "device_epoch_graph": {"ms_per_launch": round(fill_dev_ms, 6), "frac": round(fill_bytes / (fill_dev_ms / 1e3) / 1e9 / peak, 4)},
                     "launches_serialised": {"ms_per_launch": round(fill_serial_ms, 6), "frac": round(fill_bytes / (fill_serial_ms / 1e3) / 1e9 / peak, 4),
                                             "what": "the same chain without programmatic dependent launch (tb200_tune fill_pdl=0)"}},
        "generator_capacity": {"value": round(cap_value, 1), "unit": "infer/s", "steps": cap_steps, "ms_per_step": round(ms_cap / cap_steps, 6),
                               "what": "the device side of a step alone, no server: fill(64 slots) || validate(64 outputs) as CUDA-graph replays of 16 steps",
                               "api_pipelined": {"value": round(api_value, 1), "steps": e2e_steps, "h2d_bytes_per_step": h2d_step, "d2h_bytes_per_step": d2h_step,
                                                 "what": "DeviceOps.step_submit()/step_wait(), 2 steps in flight: job tables H2D, results D2H, host reads every step's 64 results"},
                               "api_sync_per_step": {"value": round(e2e_sync_value, 1), "steps": sync_steps}},
        "e2e_host_images": {"value": round(img_value, 1), "unit": "infer/s", "h2d_bytes_per_step": SLOTS * 224 * 224 * 3,
                            "d2h_bytes_per_step": d2h_step, "steps": img_steps,
                            "what": "no server: 64 uint8 HWC host images (pinned) -> H2D -> INCEPTION cast + CHW pack into the IPC slots -> validate"},
        "roofline_pack": {"bound": "hbm", "kernel": "pack_image_chw_tma_kernel (uint8 HWC -> FP32 CHW, INCEPTION)",
                          "achieved": round(pack_bytes / (pack_ms / 1e3) / 1e9, 1), "peak": peak, "unit": "GB/s",
                          "frac": round(pack_bytes / (pack_ms / 1e3) / 1e9 / peak, 4),
                          "traffic": profiled_traffic("pack_image_kernel"),
                          "algorithmic_bytes_per_launch": pack_bytes, "ms_per_launch": round(pack_ms, 6)},
        "resize_pack": {"kernel": "resize_pack_kernel (64 x uint8 375x500x3 -> Pillow BILINEAR 224x224 -> FP32 CHW INCEPTION)",
                        "ms_per_launch": round(rs_ms, 6), "images_per_s": round(SLOTS / (rs_ms / 1e3), 1),
                        "achieved_gbps": round(rs_bytes / (rs_ms / 1e3) / 1e9, 1), "algorithmic_bytes_per_launch": rs_bytes,
                        "frac": round(rs_bytes / (rs_ms / 1e3) / 1e9 / peak, 4)},
        "deflate": {"kernel": "deflate_chunk_kernel + finalize + gather (gzip container, 8 KiB chunks)", "cases": dfl},
        "c3_resnet50_b128_fp16": {
            "fill": {"achieved_gbps": round(SLOTS * IN_BYTES / (c3_fill_ms / 1e3) / 1e9, 1), "ms_per_request": round(c3_fill_ms, 6),
                     "frac": round(SLOTS * IN_BYTES / (c3_fill_ms / 1e3) / 1e9 / peak, 4), "algorithmic_bytes": SLOTS * IN_BYTES},
            "pack_u8_hwc_to_fp16_chw": {"achieved_gbps": round(c3_pack_bytes / (c3_pack_ms / 1e3) / 1e9, 1), "ms_per_request": round(c3_pack_ms, 6),
                                         "frac": round(c3_pack_bytes / (c3_pack_ms / 1e3) / 1e9 / peak, 4), "algorithmic_bytes": c3_pack_bytes},
        },
        "clocks": clocks,
    }
    if lb_error is not None:
        line["loopback_error"] = lb_error
    if "levels" in lb:
        line["loopback_levels"] = lb["levels"]
    if time_sliced is not None:
        line["time_sliced_no_mps"] = time_sliced
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_port()
    if rank == 0 and world == 1:
        try:
            line["wire_c4_c5"] = wire_extra(ops, ctx, local)
        except Exception as ex:
            line["wire_c4_c5"] = {"error": "%s: %s" % (type(ex).__name__, ex)}
    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    if rank == 0:
        print(json.dumps(line), flush=True)
    rep.close()


def wire_extra(ops, ctx, device, seconds=1.0):
    """BASELINE configs[3] / [4] (C4 BERT-large seq384, C5 Llama prompt; quoted on gRPC, no shared
    memory): the tensors go over the wire, so the fill kernel writes them into pinned, device-mapped
    staging laid out as the tail of the ModelInferRequest (raw_input_contents tag + length + tensor
    per input).  (1) the fill launch for 256 slots, timed with CUDA events (its stores cross PCIe /
    C2C to host memory, so the HBM roofline does not apply: GB/s reported as is); (2) the native load
    generator over its gRPC transport against the canned-response gRPC stub, inputs regenerated for
    every request."""
    from client_b200 import _native
    from client_b200.perf.loadgen import SlotSet, TensorSpec
    from client_b200.perf.native import GrpcStubServer, NativeLoadGenerator, grpc_wire_prefixes

    cases = {
        "c4_bert_large_seq384": ([TensorSpec("input_ids", "INT64", [1, 384]), TensorSpec("attention_mask", "INT64", [1, 384])],
                                 [TensorSpec("logits", "FP32", [1, 2])], {"input_ids": (0, 30522), "attention_mask": (0, 2)}),
        "c5_llama3_prompt4096": ([TensorSpec("input_ids", "INT32", [1, 4096])], [TensorSpec("logits", "FP32", [1, 16])],
                                 {"input_ids": (0, 128256)}),
    }
    out = {"transport": "unary gRPC over the generator's own HTTP/2 framing (csrc/h2.h), canned-response gRPC stub (no model)", "concurrency": 256}
    stub = GrpcStubServer(b"\x0a\x01m")
    timer = _native.Timer(ctx)
    try:
        for key, (ins, outs, ranges) in cases.items():
            ss = SlotSet(ins, outs, 256, "none", device, "random", SEED, ranges, name_prefix="bench_" + key, wire_prefixes=grpc_wire_prefixes(ins))
            jobs = ss._fill_jobs(list(range(256)))
            arr = (_native.FillJob * len(jobs))(*jobs)
            for _ in range(3):
                ops.fill(arr, seed=SEED)
            ops.sync()
            timer.start()
            for i in range(50):
                ops.fill(arr, seed=SEED, epoch=i)
            timer.stop()
            ops.sync()
            fill_us = timer.elapsed_ms() / 50 * 1e3
            gen = NativeLoadGenerator(stub.url, "m", "", ss, 256, regenerate=True, validate=False, protocol="grpc")
            gen.start()
            try:
                gen.window(0.3)
                w = gen.window(seconds)
            finally:
                gen.stop()
            out[key] = {"request_input_bytes": ss.in_bytes, "fill_256_slots_us": round(fill_us, 2),
                        "fill_pinned_gbps": round(256 * ss.in_bytes / (fill_us / 1e6) / 1e9, 2),
                        "fill_requests_per_s": round(256 / (fill_us / 1e6)),
                        "generator_infer_per_s": round(w["throughput"]), "p50_us": round(w["p50_us"], 1), "failed": w["failed"],
                        "slots_per_pass": round(w["device_slots"] / max(1, w["device_batches"]), 1)}
            ss.close()
    finally:
        stub.stop()
    # C5 as quoted: prompts on one ModelStreamInfer stream per connection, 16 token responses each
    from client_b200.perf.native import stream_token_responses

    resp, fin = stream_token_responses()
    sstub = GrpcStubServer(resp, final_response=fin, responses_per_request=16)
    try:
        ins, _, ranges = cases["c5_llama3_prompt4096"]
        ss = SlotSet(ins, [], 64, "none", device, "random", SEED, ranges, name_prefix="bench_c5_stream", wire_prefixes=grpc_wire_prefixes(ins))
        gen = NativeLoadGenerator(sstub.url, "llama3_8b", "", ss, 64, regenerate=True, validate=False, protocol="grpc-stream")
        gen.start()
        try:
            gen.window(0.3)
            w = gen.window(seconds)
        finally:
            gen.stop()
        ss.close()
        out["c5_llama3_stream"] = {"concurrency": 64, "tokens_per_request": 16, "infer_per_s": round(w["throughput"]),
                                   "tokens_per_s": round(w["responses_per_s"]), "ttft_p50_us": round(w["ttft_p50_us"], 1),
                                   "ttft_p99_us": round(w["ttft_p99_us"], 1), "p50_us": round(w["p50_us"], 1), "failed": w["failed"]}
    finally:
        sstub.stop()
    return out


SERVER_DESC = "client_b200.testing.native_server (own process per GPU, opens the CUDA-IPC handles, batched model kernel)"


def common_config(mps, world):
    """The config block both arms print (identical keys and values for the same box)."""
    return {"workload": WORKLOAD, "concurrency": SLOTS, "request_input_bytes": IN_BYTES, "request_output_bytes": OUT_BYTES,
            "server": SERVER_DESC, "mps": bool(mps), "instances": world}


class LoopbackBox:
    """The serving side of a loopback run: per device one private CUDA MPS daemon (when the box has the binary)
    and one native server process, pinned to its GPU's server cores.

    One daemon PER GPU, each started with CUDA_VISIBLE_DEVICES = that GPU: an MPS server takes 48 clients in
    all, not per device -- one shared daemon on an 8-GPU box refuses most of 8 x (server + generator + API
    clients) with "device(s) busy or unavailable".  The processes of GPU d therefore run with
    the daemon's only device, ordinal 0 (`ordinal[d]`; TB200_PIN_GPU names the board index for the CPU pinning,
    client_b200/perf/topology.physical_index); without MPS they see every GPU and use ordinal d."""

    # per launch (torchrun ranks share MASTER_PORT): a daemon of an earlier run that is still shutting
    # down cannot be mistaken for ours
    _TAG = os.environ.get("MASTER_PORT", "") + "_" + str(os.getppid() if os.environ.get("RANK") else os.getpid())

    def __init__(self, devices, use_mps=True, manage_mps=True, grpc=False, pin=True):
        import shutil

        self.devices, self.grpc, self.pin = list(devices), grpc, pin
        self.mps = self.manage_mps = use_mps and manage_mps and shutil.which("nvidia-cuda-mps-control") is not None
        self.servers, self.urls, self.grpc_urls, self.envs, self.ordinal = {}, {}, {}, {}, {}
        self._daemons = []
        for d in self.devices:
            self._plain_env(d)

    def _plain_env(self, d):
        self.envs[d], self.ordinal[d] = dict(os.environ), d

    def _mps_env(self, d):
        visible = [x.strip() for x in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if x.strip()]
        phys = visible[d] if d < len(visible) else str(d)
        tag = "%s_g%d" % (self._TAG, d)
        board = phys if phys.isdigit() else str(d)  # UUID entries: the position in the list is the best guess for the pinning
        return dict(os.environ, CUDA_VISIBLE_DEVICES=phys, TB200_PIN_GPU=board, CUDA_MPS_PIPE_DIRECTORY="/tmp/tb200_mps_pipe_" + tag,
                    CUDA_MPS_LOG_DIRECTORY="/tmp/tb200_mps_log_" + tag)

    def _start_mps(self, d):
        env = self._mps_env(d)
        for key in ("CUDA_MPS_PIPE_DIRECTORY", "CUDA_MPS_LOG_DIRECTORY"):
            os.makedirs(env[key], exist_ok=True)
        subprocess.run(["nvidia-cuda-mps-control", "-d"], env=env, timeout=30, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        self._daemons.append(env)
        # a client's CUDA_VISIBLE_DEVICES counts in the devices its MPS daemon exposes -- the one GPU, ordinal 0;
        # which GPU that is on the board (for the CPU pinning) travels in TB200_PIN_GPU
        self.envs[d], self.ordinal[d] = dict(env, CUDA_VISIBLE_DEVICES="0"), 0

    def _stop_mps(self):
        for env in self._daemons:
            try:
                subprocess.run(["nvidia-cuda-mps-control"], input="quit\n", env=env, text=True, timeout=30, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            except Exception:
                pass
        self._daemons = []

    def _start_server(self, dev):
        import select
        import socket

        with socket.socket() as sk:
            sk.bind(("127.0.0.1", 0))
            port = sk.getsockname()[1]
        cmd = [sys.executable, "-m", "client_b200.testing.native_server", "--port", str(port), "--device", str(self.ordinal[dev])]
        if self.grpc:
            cmd += ["--grpc-port", "0"]
        if self.pin:
            cmd += ["--pin-cpus"]
        srv = subprocess.Popen(cmd, cwd=ROOT, env=self.envs[dev], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        ready, _, _ = select.select([srv.stdout], [], [], 90.0)  # a server that never comes up must not hang the bench
        hello = srv.stdout.readline() if ready else "timeout waiting for the server"
        if "listening" not in hello:
            srv.terminate()
            try:
                rest, _ = srv.communicate(timeout=10)  # the rest of what it said (a traceback, usually)
            except Exception:
                srv.kill()
                rest = ""
            raise RuntimeError("native server for device %d did not start: %s" % (dev, " | ".join((hello + (rest or "")).strip().splitlines()[-4:])[:600]))
        self.servers[dev] = srv
        self.urls[dev] = "127.0.0.1:%d" % port
        if "grpc=" in hello:
            self.grpc_urls[dev] = hello.split("grpc=")[1].strip()

    def __enter__(self):
        try:
            if self.manage_mps:
                try:
                    for d in self.devices:
                        self._start_mps(d)
                    time.sleep(1.0)
                except Exception:  # no daemon to be had: time-sliced contexts
                    self._stop_mps()
                    self.mps = self.manage_mps = False
                    for d in self.devices:
                        self._plain_env(d)
            for dev in self.devices:
                try:
                    self._start_server(dev)
                except RuntimeError:
                    if not self.mps:
                        raise
                    time.sleep(5.0)  # a daemon of an earlier run may still hold the GPU while it shuts down: once more
                    self._start_server(dev)
        except Exception:
            self.__exit__(None, None, None)
            raise
        return self

    def __exit__(self, *exc):
        for srv in self.servers.values():
            srv.terminate()
        for srv in self.servers.values():
            try:
                srv.wait(10)
            except Exception:
                srv.kill()
        self.servers = {}
        self._stop_mps()
        return False

    def generator(self, dev, steps, warmup, mode="per-request", concurrency=SLOTS, extra=(), min_seconds=0.1, timeout=120, sync=None):
        """One `python -m client_b200.perf.loopback` child against this box's server for `dev`.  `sync`: called
        once when the child is warm (or has failed); the child starts timing when it returns -- with one
        rank per GPU that is the barrier that makes every instance time the same interval."""
        import tempfile

        cmd = [sys.executable, "-m", "client_b200.perf.loopback", "-u", self.urls[dev], "--device", str(self.ordinal[dev]), "--concurrency", str(concurrency),
               "--steps", str(steps), "--warmup", str(warmup), "--input-data-mode", mode, "--min-seconds", str(min_seconds),
               "--seed", str(SEED), "--json"] + (["--pin-cpus"] if self.pin else []) + list(extra)
        if sync is None:
            r = subprocess.run(cmd, cwd=ROOT, env=self.envs[dev], capture_output=True, text=True, timeout=timeout)
            stdout, stderr = r.stdout, r.stderr
        else:
            with tempfile.TemporaryDirectory(prefix="tb200_sync_") as sync_dir:
                child = subprocess.Popen(cmd + ["--sync-dir", sync_dir], cwd=ROOT, env=self.envs[dev], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
                try:
                    t_end = time.perf_counter() + timeout
                    while not os.path.exists(os.path.join(sync_dir, "ready")) and child.poll() is None and time.perf_counter() < t_end:
                        time.sleep(0.002)
                finally:
                    sync()
                with open(os.path.join(sync_dir, "go"), "w"):
                    pass
                try:
                    stdout, stderr = child.communicate(timeout=timeout)
                except subprocess.TimeoutExpired:
                    child.kill()
                    stdout, stderr = child.communicate()
        for line in stdout.splitlines():
            if line.startswith("{"):
                return json.loads(line)
        raise RuntimeError("generator child failed: " + (stdout + stderr)[-400:])


def _host_loop_worker(impl, url, device, tag, seconds, data_mode, ready, go, q):
    try:
        if impl == "reference":
            from oracle import ref_client as mod
        else:
            from client_b200.perf import host_loop as mod
        n, lat = mod.run_loop(url, device, tag, seconds, data_mode, ready=ready, go=go)
        q.put((n, lat[:: max(1, len(lat) // 2000)], None))
    except Exception as ex:  # the parent must not hang on the barrier
        try:
            ready.abort()
        except Exception:
            pass
        q.put((0, [], "%s: %s" % (type(ex).__name__, ex)))


def host_loops(box, impl, nproc, seconds, data_mode, sync=None):
    """`nproc` free-running client processes (round-robin over the box's servers) for `seconds`
    of wall time; impl "b200" = the drop-in modules, "reference" = the restated reference code.
    `sync`: called once when this rank's clients are ready, before they are released (the ranks' barrier)."""
    import multiprocessing as mp

    ctx = mp.get_context("spawn")
    ready, go, q = ctx.Barrier(nproc + 1), ctx.Event(), ctx.Queue()
    devs = box.devices
    procs = []
    keys = ("CUDA_VISIBLE_DEVICES", "TB200_PIN_GPU", "CUDA_MPS_PIPE_DIRECTORY", "CUDA_MPS_LOG_DIRECTORY")
    saved = {k: os.environ.get(k) for k in keys}
    try:
        for i in range(nproc):
            dev = devs[i % len(devs)]
            for k in keys:  # a spawned child inherits this process's environment: its GPU's daemon, its GPU as ordinal 0
                if k in box.envs[dev]:
                    os.environ[k] = box.envs[dev][k]
                else:
                    os.environ.pop(k, None)
            p = ctx.Process(target=_host_loop_worker,
                            args=(impl, box.urls[dev], box.ordinal[dev], "%s%d_%d" % (impl[0], os.getpid(), i), seconds, data_mode, ready, go, q))
            p.start()
            procs.append(p)
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    try:
        ready.wait(timeout=240)  # every client has its CUDA context, regions and connection
    except Exception:
        pass
    if sync is not None:
        sync()
    t0 = time.perf_counter()
    go.set()
    parts = [q.get(timeout=seconds + 240) for _ in procs]
    dt = time.perf_counter() - t0
    for p in procs:
        p.join(30)
    errors = [e for _, _, e in parts if e]
    total = sum(n for n, _, _ in parts)
    lat = np.concatenate([np.asarray(l, dtype=np.float64) for _, l, _ in parts if len(l)]) / 1e3 if total else np.zeros(1)
    return {"infer_per_s": round(total / seconds, 1), "count": int(total), "seconds": seconds, "wall_seconds": round(dt, 3), "processes": nproc,
            "p50_us": round(float(np.percentile(lat, 50)), 1), "p99_us": round(float(np.percentile(lat, 99)), 1),
            "failed_workers": len(errors), **({"errors": errors[:2]} if errors else {})}


def host_process_count(world):
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    return max(1, min(32 * world, cores // 2)), cores


HOST_LOOP_SECONDS = 2.5

def _grpc_loopback_levels(grpc_url, env=None):
    """BASELINE configs[3] / [4] against the native server's gRPC port: the CLI's native engine
    (tensors generated by the fill kernel into the message tails; C5 on ModelStreamInfer streams
    with 16 token responses per prompt)."""
    out = {}
    for key, argv in (("c4_bert_large_grpc", ["-m", "bert_large"]),
                      ("c5_llama3_stream", ["-m", "llama3_8b", "--streaming", "--shape", "input_ids:1,4096", "--request-parameter", "max_tokens:16:int"])):
        r = subprocess.run([sys.executable, "-m", "client_b200.perf", "-u", grpc_url, "-i", "grpc", "--shared-memory", "none", "--engine", "native",
                            "--concurrency-range", "1:256:16x", "-p", "600", "-r", "4", "--json"] + argv,
                           cwd=ROOT, env=env, capture_output=True, text=True, timeout=240)
        rows = []
        for line in r.stdout.splitlines():
            if line.startswith("{"):
                w = json.loads(line)
                row = {"concurrency": w["concurrency"], "infer_per_s": round(w["throughput"], 1), "p50_us": round(w["p50_us"], 1),
                       "p99_us": round(w["p99_us"], 1), "failed": int(w["failed"])}
                if "ttft_p50_us" in w:
                    row.update(ttft_p50_us=round(w["ttft_p50_us"], 1), tokens_per_s=round(w["responses_per_s"], 1))
                rows.append(row)
        out[key] = rows if rows else {"error": (r.stdout + r.stderr)[-300:]}
    return out


def cpu_baseline_port(seconds=8.0):
    """The C oracle on one host core doing the per-request work of the step: Philox fill
    of one FP32[3,224,224] tensor + tobytes + body join (two memcpys)."""
    from oracle import cref

    lib = cref.lib()
    tensor = np.zeros(IN_BYTES, np.uint8)
    scratch = np.zeros(IN_BYTES, np.uint8)
    header = b'{"inputs":[{"name":"data_0","shape":[3,224,224],"datatype":"FP32","parameters":{"binary_data_size":602112}}]}'
    body = np.zeros(IN_BYTES + len(header), np.uint8)
    hbuf = np.frombuffer(header, np.uint8)
    done = 0
    t0 = time.perf_counter()
    while True:
        for _ in range(64):
            lib.oracle_fill(tensor.ctypes.data, IN_BYTES, cref.DT["FP32"], 0, SEED, done, 0.0, 0.0, 0, 0)
            lib.oracle_marshal_http(body.ctypes.data, hbuf.ctypes.data, len(header), scratch.ctypes.data, tensor.ctypes.data, IN_BYTES)
            done += 1
        if time.perf_counter() - t0 > seconds:
            break
    dt = time.perf_counter() - t0
    return {"value": round(done / dt, 1), "unit": "infer/s", "cores": 1, "kind": "port",
            "sample": "%d requests in %.1f s: oracle_fill FP32[3,224,224] + tobytes + JSON/body join, 1 thread" % (done, dt)}


def run_reference(args):
    """--impl reference: the reference client's own CPU path for C2 (numpy tensor ->
    set_shared_memory_region with a real H2D -> infer -> get_contents_as_numpy), restated in
    oracle/ref_client.py, as free-running worker processes against the same stand-in server(s);
    rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = max(1, args.gpus)
    steps, warmup = args.steps, max(args.warmup, 3)
    nproc, cores = host_process_count(world)
    with LoopbackBox(range(world), grpc=False) as box:
        host_loops(box, "reference", min(nproc, 4), 0.5, "per-request")  # warm-up: contexts, page cache, server
        per_request = host_loops(box, "reference", nproc, HOST_LOOP_SECONDS, "per-request")
        once = host_loops(box, "reference", nproc, HOST_LOOP_SECONDS, "once")
        mps = box.mps
    value = per_request["infer_per_s"]
    sample = ("%d free-running processes x %.1f s: numpy Generator.random FP32[3,224,224] -> cudaMemcpyAsync H2D + sync (set_shared_memory_region) -> "
              "HTTP infer naming the regions -> whole-region D2H + sync (get_contents_as_numpy); oracle/ref_client.py + oracle/wire.py" % (nproc, HOST_LOOP_SECONDS))
    line = {
        "impl": "reference", "metric": "inferences/sec", "value": value, "unit": "infer/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": round(SLOTS / value * 1e3, 4) if value else None,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": common_config(mps, world),
        "cpu_baseline": {"value": value, "unit": "infer/s", "cores": nproc, "kind": "port", "sample": sample, "host_cores": cores},
        "e2e": {"value": value, "unit": "infer/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "p50_us": per_request["p50_us"], "p99_us": per_request["p99_us"],
        "fill_once": {"value": once["infer_per_s"], "p50_us": once["p50_us"], "processes": nproc,
                      "what": "regions filled once, every request only names them (no per-request host tensor work)"},
        "input_pack_gbps": round(value * IN_BYTES / 1e9, 3),
        "timing": "wall clock: completed requests of all processes / the fixed run time (free-running, no per-step barrier)",
    }
    line["failed_clients"] = per_request.get("failed_workers", 0)
    if per_request.get("errors"):
        line["errors"] = per_request["errors"]
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20000,
                    help="timed steps of each repetition of the headline generator and of the DeviceOps step_submit/step_wait "
                         "loop (the one --dump-outputs writes).  Sections that need a longer or shorter window derive "
                         "their own count from it, each reported in the JSON line: the generator-capacity graphs run at "
                         "least 8000 steps, the synchronous API loop a quarter of --steps but at least 10, the host-image "
                         "loop 5 to 2000, the time-sliced run at most 2000")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-loopback", action="store_true", help="skip the extra loopback levels (other concurrencies, gRPC configs, the run without MPS)")
    ap.add_argument("--no-mps", action="store_true", help="do not start a CUDA MPS daemon: client and server time-slice the GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed DeviceOps step returned to DIR (rank 0 only): inputs.npy, the 64 "
                         "FP32[3,224,224] tensors the fill kernel generated for that step; check_<field>.npy, the validate "
                         "kernel's 64 results (float64) over the response logits, which are written once at setup and so "
                         "are the same for every step and every --steps")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
