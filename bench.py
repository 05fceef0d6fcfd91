#!/usr/bin/env python
"""bench.py -- Mpix/s of dense DIS flow on synthetic 1024x436 pairs (op-point 2).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (all pyramid levels: patch inverse search,
densification, variational refinement == the reference's "O.Flow Run-Time"
region, oflow.cpp:113-114,355-360) over B pairs per GPU (default 64 = the batch
of BASELINE configs[3]; one pair alone leaves 147 of 148 SMs idle, see
batch_sweep in the output).  Pixels are counted at the ORIGINAL image size, once
per pair (SURVEY.md section 8d).

  value : device-timed, padded pyramids already resident in HBM; the K steps are dealt round-robin
          to 8-10 lanes (context + stream) so that consecutive steps overlap
  e2e   : same metric through the C-ABI with pinned HOST buffers; every step copies its input and its
          result.  Three legs (e2e.legs): "pyramids" = the strict OFClass contract (all four padded
          float arrays of every level in, flow of level sc_l out; oflow.h:84-86) -- this is e2e.value,
          the region the reference arm times; "finest" = un-padded finest-level images in (rest of the
          pyramid derived on the device inside the timed region); "cli" = 8-bit frames in,
          full-resolution flow out (what run_OF_INT does between imread and SaveFlowFile).  The
          pyramids/finest results are checked bit for bit against the resident path
  sharded : BASELINE configs[3] as written -- 64 pairs TOTAL owned by rank 0, scattered over the ranks'
          GPUs with NCCL, gathered back (strong scaling; of_dis_b200/sharding.py)
  fast_mode : the opt-in red-black refinement (not bit-identical; throughput, delta to the exact flow, EPE of both)
  big_configs : BASELINE configs[2] and [4] (1920x1080 RGB, 2880x1988 stereo) on one GPU, per kernel class
  single_lane / batch_sweep : one lane, L2 flushed before every step (latency of 64, 8, 1 pairs)
  roofline     : dominant kernel (lexicographic SOR), algorithmic bytes / CUDA-event time, plus the
                 issue-slot utilisation of the whole overlapped step
  cpu_baseline : the reference CPU build (oracle/_ref) or the C port on this box's cores

Under torchrun every rank owns B pairs (weak scaling, no data-path collective;
frames are independent -- DESIGN.md section 6); time = max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

H_ORG, W_ORG = 436, 1024
OP_POINT = 2
MAX_DISTINCT = 16
FRAMES_U8 = []  # the 8-bit frames of the pairs make_pairs() returned last ([2][h][w] each)


def make_pairs(n, seed0):
    from of_dis_b200 import params, preprocess, synth

    del FRAMES_U8[:]
    prm = params.operating_point(OP_POINT, W_ORG)
    pyrs = []
    for s in range(min(n, MAX_DISTINCT)):
        i0, i1, _ = synth.synthetic_pair(H_ORG, W_ORG, 1, seed=seed0 + s)
        pyrs.append(preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s))
        FRAMES_U8.append(np.stack([i0, i1]))
    while len(pyrs) < n:  # large batches cycle through the distinct pairs (generation costs 0.3 s each)
        FRAMES_U8.append(FRAMES_U8[len(pyrs) % MAX_DISTINCT])
        pyrs.append(pyrs[len(pyrs) % MAX_DISTINCT])
    return prm, pyrs


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ts, ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                if t0 - 0.05 <= ts <= t1 + 0.2:
                    sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _ref_kind(prm):
    from oracle import port_driver, ref_driver

    if ref_driver.ref_available(prm.flavour()):
        return "reference", ref_driver
    port_driver.build()
    return "port", port_driver


def _native_pass_seconds(pyrs, prm, nrep, threads):
    """One call = nrep passes over pyrs on a native std::thread pool (oracle/ref_wrapper.cpp:
    ofdis_ref_run_many); no Python inside the timed region."""
    from oracle import ref_driver

    return ref_driver.ref_run_many(pyrs, prm, nrep, threads)[0]


def _python_pool_mpix(fn, prm, pyrs, seconds, threads):
    """Round-1 harness kept for comparison: one ctypes call per pair from a Python thread pool."""
    from concurrent.futures import ThreadPoolExecutor

    fn(pyrs[0], prm)  # warm
    done = 0
    work = [pyrs[i % len(pyrs)] for i in range(max(len(pyrs), threads))]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        while time.perf_counter() - t0 < seconds:
            list(ex.map(lambda p: fn(p, prm), work))
            done += len(work)
    return done * H_ORG * W_ORG / (time.perf_counter() - t0) / 1e6, done


def cpu_reference(prm, pyrs, frames_u8, seconds, threads):
    """Frame-parallel reference CPU build on `threads` host threads (OFClass instances share no mutable
    state, SURVEY 8b).  Returns the cpu_baseline object: OFClass region on 1 and on all threads (native
    pool), the scaling factor, the CLI-level leg (pyramid + OFClass + upsampling) and, for comparison,
    the round-1 Python-thread harness."""
    kind, drv = _ref_kind(prm)
    pix = H_ORG * W_ORG
    if kind != "reference":  # no compiled reference here: the C port through the Python pool
        val, done = _python_pool_mpix(drv.port_run, prm, pyrs, seconds, threads)
        return {"value": val, "unit": "Mpix/s", "cores": threads, "kind": kind,
                "sample": "%d pairs, frame-parallel Python pool over %d threads" % (done, threads)}
    work = [pyrs[i % len(pyrs)] for i in range(max(len(pyrs), threads))]
    _native_pass_seconds(work[:threads], prm, 1, threads)  # warm
    # one thread: a few pairs
    t1 = _native_pass_seconds(work[:4], prm, 1, 1)
    one = 4 * pix / t1 / 1e6
    # all threads, as the --impl reference arm measures it: one pass over the batch per step, a few steps
    steps = [_native_pass_seconds(work, prm, 1, threads) for _ in range(5)]
    many = len(work) * pix / (sum(steps[1:]) / len(steps[1:])) / 1e6
    # ... and sustained: passes back to back for about half of `seconds` (all-core clocks settle: on the
    # pool's hosts the sustained rate is about half of the burst rate above)
    nrep = max(2, int(seconds * 0.5 / max(min(steps), 1e-3)))
    tn = _native_pass_seconds(work, prm, nrep, threads)
    out = {"value": many, "unit": "Mpix/s", "cores": threads, "kind": kind,
           "sample": "%d pairs per step (OFClass ctor region), native std::thread pool over %d threads, 4 steps of one "
                     "pass each -- the scheme of bench.py --impl reference" % (len(work), threads),
           "one_thread": one, "thread_scaling": many / one,
           "sustained": {"value": nrep * len(work) * pix / tn / 1e6, "unit": "Mpix/s",
                         "sample": "%d passes back to back (%.1f s)" % (nrep, tn)}}
    if frames_u8 is not None:
        from oracle import ref_driver

        fr = frames_u8[np.arange(len(work)) % len(frames_u8)]
        ref_driver.ref_run_many_u8(fr[:threads], prm, 1, threads)
        reps = 4  # worker threads reuse their pyramid buffers from the second pair on
        tc = ref_driver.ref_run_many_u8(fr, prm, reps, threads)[0]
        out["cli"] = {"value": reps * len(work) * pix / tc / 1e6, "unit": "Mpix/s",
                      "sample": "8-bit frames -> pyramids -> OFClass -> full-resolution flow (run_dense.cpp:130-178,"
                                "391-414 restated without OpenCV), %d x %d pairs on %d threads" % (reps, len(work), threads)}
    pv, pdone = _python_pool_mpix(drv.ref_run, prm, pyrs, min(seconds * 0.3, 4.0), threads)
    out["python_pool"] = {"value": pv, "note": "round-1 harness: one ctypes call per pair from a Python ThreadPoolExecutor"}
    return out


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # one step = the arm's batch, enlarged to one pair per hardware thread when the batch is smaller
    # (the reference is single-threaded per pair; frame parallelism is the only way it uses the host)
    npairs = max(args.batch * world, cores)
    threads = cores
    prm, pyrs0 = make_pairs(min(npairs, args.batch * world), 0)
    pyrs = [pyrs0[i % len(pyrs0)] for i in range(npairs)]
    kind, drv = _ref_kind(prm)
    times = []
    if kind == "reference":
        for s in range(args.warmup + args.steps):
            t = _native_pass_seconds(pyrs, prm, 1, threads)
            if s >= args.warmup:
                times.append(t)
        how = "native std::thread pool"
    else:
        from concurrent.futures import ThreadPoolExecutor

        with ThreadPoolExecutor(max_workers=threads) as ex:
            for s in range(args.warmup + args.steps):
                t0 = time.perf_counter()
                list(ex.map(lambda p: drv.port_run(p, prm), pyrs))
                if s >= args.warmup:
                    times.append(time.perf_counter() - t0)
        how = "Python thread pool"
    ms = 1e3 * sum(times) / len(times)
    val = npairs * H_ORG * W_ORG / (ms * 1e-3) / 1e6
    line = {
        "impl": "reference", "metric": "Mpix/s dense flow (1024x436, op-point 2)", "value": val, "unit": "Mpix/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": val, "unit": "Mpix/s", "cores": threads, "kind": kind,
                         "sample": "%d pairs per step, frame-parallel over %d threads (%s; host has %d cores), "
                                   "timer = OFClass ctor region" % (npairs, threads, how, cores)},
        "e2e": {"value": val, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_config(args, world):
    return {"workload": "%d x (1024x436 gray pair, op-point 2: P=8 ov=0.4 levels 5..3, 12 GN iters, TV 3 SOR sweeps) "
                        "per GPU per step (BASELINE configs[3]'s batch of 64 pairs of configs[1] geometry; "
                        "single-pair and 8-pair latencies in batch_sweep)" % args.batch,
            "pairs_per_gpu": args.batch, "pairs_total": args.batch * world, "parallelism": "frames x%d" % world,
            "lanes": "%d contexts/streams per GPU, consecutive steps overlap" % max(1, args.lanes),
            "l2": "two alternating working sets of ~2 MB per pair exceed the 126 MB L2 at the default batch; "
                  "single_lane and batch_sweep numbers are taken with L2 flushed (256 MiB write) before every step"}


def measure_sharded(args, prm, rank, world, local, stream, barrier, maxrank):
    """BASELINE configs[3] as written (strong scaling): 64 pairs TOTAL in rank 0's pinned memory ->
    H2D on rank 0 -> NCCL scatter -> engine on every rank's block -> NCCL gather -> D2H on rank 0, all
    inside the timed region (CUDA events on the stream, max over ranks)."""
    import torch

    from of_dis_b200 import sharding

    n_total = 64
    out = {"pairs_total": n_total, "scaling": "strong", "ranks": world}
    dev = torch.device("cuda", local)
    for io in ("ofclass", "cli"):
        eng = sharding.ShardedEngine(prm, n_total, W_ORG, H_ORG, io, dev, stream)
        host_in = host_out = None
        if rank == 0:
            if io == "cli":
                arr = np.stack([FRAMES_U8[i % len(FRAMES_U8)].reshape(-1) for i in range(n_total)])
            else:
                from of_dis_b200 import preprocess

                rows = []
                for i in range(min(n_total, MAX_DISTINCT)):
                    a, b = FRAMES_U8[i % len(FRAMES_U8)]
                    p = preprocess.PairPyramids(a, b, prm.sc_f, prm.p_samp_s)
                    P_ = p.imgpadding
                    rows.append(np.stack([p.i0[prm.sc_l][P_:-P_, P_:-P_], p.i1[prm.sc_l][P_:-P_, P_:-P_]]).reshape(-1))
                arr = np.stack([rows[i % len(rows)] for i in range(n_total)])
            host_in = torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
            host_out = torch.empty((n_total, eng.out_elems), dtype=torch.float32).pin_memory()
        for _ in range(args.warmup):
            eng.step(host_in, host_out)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(args.steps):
            eng.step(host_in, host_out)
        ev1.record(stream)
        torch.cuda.synchronize()
        ms = maxrank(ev0.elapsed_time(ev1) / args.steps)
        barrier()
        out[io] = {"ms_per_step": ms, "value": n_total * H_ORG * W_ORG / (ms * 1e-3) / 1e6, "unit": "Mpix/s",
                   "h2d_bytes_per_step": int(n_total * eng.in_elems * (1 if io == "cli" else 4)),
                   "d2h_bytes_per_step": int(n_total * eng.out_elems * 4), "pairs_per_rank": eng.m,
                   "launches_per_step": None}
        eng.close()
    out["note"] = ("one stream per rank, steps back to back (no overlap between steps): rank 0's PCIe link carries all "
                   "inputs and all flows; 'ofclass' = finest-level float images in / level flow out, 'cli' = 8-bit frames "
                   "in / full-resolution flow out")
    return out


def dump_flows(out_dir, ctx, B, li, prm, limit=64 << 20):
    """What a caller of the resident path receives from `ctx`'s last run: the flow of level sc_l of every pair, as
    DIR/flow.npy; the first pairs only when all of them would exceed `limit` bytes."""
    n = min(B, limit // (li["h"] * li["w"] * prm.nop * 4))
    flow = np.empty((n, li["h"], li["w"], prm.nop), np.float32)
    ctx.get_flow_batch(0, n, flow)
    ctx.sync()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "flow.npy"), flow)


def measure_big_configs():
    """BASELINE configs[2] and configs[4] on this GPU (tools/big_configs.py): step time, per kernel
    class and per level; the SOR of configs[4]'s level 1 at 8 pairs is the launch SURVEY 8(d) names."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import big_configs

        rows = []
        for name, c in big_configs.CFGS.items():
            for b in (1, 8):
                rows.append(big_configs.measure(name, c, b, {}))
        return rows
    except Exception as e:  # must not lose the headline numbers
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=64, help="pairs per GPU per step")
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--lanes", type=int, default=0,
                    help="contexts/streams whose steps overlap; 0 = 8, or the divisor of --steps in 6..12 closest to 8 "
                         "(every lane then runs the same number of steps and the drain is shortest)")
    ap.add_argument("--e2e-upload", choices=("finest", "images", "pyramids", "cli"), default="pyramids",
                    help="which leg becomes e2e.value: pyramids = all four padded arrays of every level as OFClass takes "
                         "them (default: the region the reference arm times), finest = un-padded I0,I1 of the finest used "
                         "level, images = padded I0,I1 of every level, cli = 8-bit frames in / full-resolution flow out")
    ap.add_argument("--no-extras", action="store_true", help="skip the sharded and big_configs legs")
    ap.add_argument("--opt", action="append", default=[], metavar="NAME=VALUE",
                    help="ofdis_set_option on every context (launch-geometry experiments; results are bit-identical)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the flows the last one computed as DIR/flow.npy (float32, "
                         "[pair][h][w][nop] at level sc_l; rank 0's pairs, the first ones only beyond 64 MB)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path")
    args.warmup = max(args.warmup, 3)
    if args.lanes <= 0:
        divs = [d for d in range(6, 13) if args.steps % d == 0]
        args.lanes = min(divs, key=lambda d: (abs(d - 8), -d)) if divs else 8
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    from of_dis_b200 import api, numa

    torch.cuda.set_device(local)
    # pinned staging buffers must live on the GPU's own socket (of_dis_b200/numa.py)
    numa_node, prev_affinity = numa.bind_to_gpu_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    B = args.batch
    prm, pyrs = make_pairs(B, 1000 * rank)
    # a non-default torch stream: the context enqueues on it and torch.cuda.Event times it
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    opts = dict((o.split("=")[0], int(o.split("=")[1])) for o in args.opt)
    if opts:  # every context created below gets the options
        _Context = api.Context

        def _ctx_with_opts(*a, **k):
            c = _Context(*a, **k)
            for name, val in opts.items():
                c.set_option(name, val)
            return c

        api.Context = _ctx_with_opts
    ctx = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, B, device=local,
                      stream=stream.cuda_stream)
    ff = ctx.packed_frame_floats
    host_in = torch.empty((B, ff), dtype=torch.float32).pin_memory()
    for f, p in enumerate(pyrs):
        ctx.pack_frame(p, host_in[f].numpy())
    li = ctx.level_info(prm.sc_l)
    flow_floats = li["w"] * li["h"] * prm.nop
    host_out = torch.empty((B, flow_floats), dtype=torch.float32).pin_memory()
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, steps):
        evs = []
        for _ in range(steps):
            flush.fill_(1.0)  # L2 flush, outside the timed interval
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            step_fn()
            b.record(stream)
            evs.append((a, b))
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs) / steps  # ms per step

    def maxrank(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # NL lanes (context + stream each): step i runs on lane i % NL, so consecutive steps overlap on the
    # device -- copies of one step under the kernels of the others, and the latency-bound refinement
    # kernels of several batches side by side (one batch of 64 pairs occupies 64 of 148 SMs there).
    NL = max(1, args.lanes)
    lanes = [(ctx, stream, host_out)]  # + the cli leg's full-resolution host buffer, appended below
    for _ in range(NL - 1):
        st_l = torch.cuda.Stream()
        lanes.append((api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, B, device=local,
                                  stream=st_l.cuda_stream), st_l,
                      torch.empty((B, flow_floats), dtype=torch.float32).pin_memory()))
    for c in [l[0] for l in lanes]:
        c.upload_packed(0, B, host_in.data_ptr())
        c.set_graph_mode(True)

    def pipelined(step_fn, steps):
        """K steps dealt round-robin to the lanes; device time from one event pair spanning all streams."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for l in lanes[1:]:
            l[1].wait_event(ev0)
        for i in range(steps):
            step_fn(i)
        for l in lanes[1:]:
            stream.wait_stream(l[1])
        ev1.record(stream)
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / steps

    # ---- device-resident throughput -----------------------------------------
    def resident_step(i):
        lanes[i % NL][0].run(B)

    for i in range(NL * args.warmup):
        resident_step(i)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.25)
    l0 = sum(l[0].launch_count for l in lanes)
    t0 = time.time()
    ms_res = maxrank(pipelined(resident_step, args.steps))
    launches = (sum(l[0].launch_count for l in lanes) - l0) // args.steps
    if args.dump_outputs and rank == 0:
        dump_flows(args.dump_outputs, lanes[(args.steps - 1) % NL][0], B, li, prm)
    barrier()
    # The K timed steps above last a few milliseconds.  The same loop over >= 0.5 s: clocks and thermals under a
    # sustained load (the clock sampler runs through both), reported beside `value`, never instead of it.
    n_sus = max(args.steps, int(0.5e3 / max(ms_res, 1e-3)))
    ms_sus = maxrank(pipelined(resident_step, n_sus))
    sustained = {"steps": n_sus, "ms_per_step": ms_sus, "value": None, "seconds": n_sus * ms_sus * 1e-3}
    barrier()
    # one lane alone, L2 flushed before every step (latency of one batch)
    ms_res_single = maxrank(timed(lambda: ctx.run(B), args.steps))

    # ---- end to end with host buffers -----------------------------------------
    # Every step copies its own inputs from pinned host memory and its flows back.  No L2 flush is
    # possible inside an overlapped region; the two alternating working sets (2 x ~2 MB per pair)
    # exceed L2 at the default batch.
    # Default e2e payload: the un-padded I0,I1 of the finest level the run uses; coarser levels (2x2
    # box means), Sobel gradients and border paddings are derived on the device inside the timed
    # region (ofdis_upload_finest_level).  --e2e-upload pyramids ships all four padded arrays of
    # every level exactly as OFClass's constructor takes them.
    n_img = ctx.packed_images_frame_floats
    n_fin = ctx.finest_level_frame_floats
    host_img = torch.empty((B, n_img), dtype=torch.float32).pin_memory()
    host_img.copy_(host_in[:, :n_img])
    host_fin = torch.empty((B, n_fin), dtype=torch.float32).pin_memory()
    P_ = pyrs[0].imgpadding
    for f, p in enumerate(pyrs):
        fin = np.stack([p.i0[prm.sc_l][P_:-P_, P_:-P_], p.i1[prm.sc_l][P_:-P_, P_:-P_]])
        host_fin[f].numpy()[:] = fin.reshape(-1)
    host_u8 = torch.from_numpy(np.ascontiguousarray(np.stack(FRAMES_U8[:B]))).pin_memory()  # [B][2][h][w]
    full_floats = H_ORG * W_ORG * prm.nop
    for i in range(NL):  # full-resolution output buffers of the cli leg, one per lane
        lanes[i] = lanes[i] + (torch.empty((B, full_floats), dtype=torch.float32).pin_memory(),)
    payloads = {
        "finest": (n_fin * 4, flow_floats * 4, "un-padded I0,I1 of level %d in; levels %d..%d, I0x,I0y and paddings derived on "
                   "the device inside the timed region; flow of level %d out" % (prm.sc_l, prm.sc_l + 1, prm.sc_f, prm.sc_l)),
        "images": (n_img * 4, flow_floats * 4, "padded I0,I1 of levels %d..%d in; I0x,I0y derived on the device inside the "
                   "timed region; flow of level %d out" % (prm.sc_l, prm.sc_f, prm.sc_l)),
        "pyramids": (ff * 4, flow_floats * 4, "padded I0,I0x,I0y,I1 of levels %d..%d in (what OFClass takes, oflow.h:84-86); "
                     "flow of level %d out" % (prm.sc_l, prm.sc_f, prm.sc_l)),
        "cli": (2 * H_ORG * W_ORG, full_floats * 4, "8-bit frames in (pyramid, gradients, paddings on the device); "
                "full-resolution flow out (x%d upsampling and crop on the device): run_dense.cpp:130-178,391-414" % (1 << prm.sc_l)),
    }

    def upload(c, mode, b=B):
        if mode == "finest":
            c.upload_finest_level(0, b, host_fin.data_ptr())
        elif mode == "images":
            c.upload_packed_images(0, b, host_img.data_ptr())
        elif mode == "cli":
            c.upload_frames_u8(0, b, host_u8.data_ptr(), W_ORG, H_ORG)
        else:
            c.upload_packed(0, b, host_in.data_ptr())

    def download(c, mode, ho, hfull, b=B):
        if mode == "cli":
            c.get_flow_fullres(0, b, hfull.data_ptr(), W_ORG, H_ORG)
        else:
            c.get_flow_batch(0, b, ho.data_ptr())

    # the e2e path must produce the flows of the resident path (same pairs), bit for bit
    resident_flow = torch.empty((B, flow_floats), dtype=torch.float32)
    ctx.upload_packed(0, B, host_in.data_ptr())
    ctx.run(B)
    ctx.get_flow_batch(0, B, resident_flow.data_ptr())
    ctx.sync()
    from of_dis_b200 import preprocess as _pp

    def measure_e2e(mode):
        def e2e_step(i):
            c, _, ho, hfull = lanes[i % NL]
            upload(c, mode)
            c.run(B)
            download(c, mode, ho, hfull)

        # Warm-up: W steps per lane, continued until 0.4 s of copies have run -- an idle PCIe link takes
        # ~0.2 s of traffic to leave its low-power state (tools/e2e_probe.py: first pass 30 GB/s, then 54).
        n_warm, w_start = 0, time.perf_counter()
        while n_warm < NL * args.warmup or time.perf_counter() - w_start < 0.4:
            e2e_step(n_warm)
            n_warm += 1
            if n_warm % NL == 0:
                torch.cuda.synchronize()
        barrier()
        e2e_step(0)
        torch.cuda.synchronize()
        if mode == "cli":
            exp = _pp.postprocess(resident_flow[0].numpy().reshape(li["h"], li["w"], prm.nop), prm.sc_l, pyrs[0].padw,
                                  pyrs[0].padh, W_ORG, H_ORG)
            same = bool(np.array_equal(lanes[0][3][0].numpy().view(np.uint32), np.ascontiguousarray(exp).reshape(-1).view(np.uint32)))
        else:
            same = bool(torch.equal(resident_flow.view(torch.int32), host_out.view(torch.int32)))
        barrier()
        w0 = time.perf_counter()
        ms = maxrank(pipelined(e2e_step, args.steps))
        wall = (time.perf_counter() - w0) / args.steps * 1e3
        barrier()
        h2d, d2h, what = payloads[mode]
        return {"value": B * world * H_ORG * W_ORG / (ms * 1e-3) / 1e6, "ms_per_step": ms, "wall_ms_per_step": wall,
                "h2d_bytes_per_step": int(B * h2d), "d2h_bytes_per_step": int(B * d2h), "payload": what,
                "result_checked_bitwise": same, "warmup_steps": n_warm}

    mode = args.e2e_upload
    legs = {m: measure_e2e(m) for m in dict.fromkeys([mode, "pyramids", "finest", "cli"])}
    t1 = time.time()
    clocks = sampler.stop(t0, t1)

    # serial variant: one lane, H2D -> run -> D2H back to back, L2 flushed between steps
    def e2e_serial():
        upload(ctx, mode)
        ctx.run(B)
        download(ctx, mode, host_out, lanes[0][3])

    for _ in range(args.warmup):
        e2e_serial()
    ms_e2e_serial = maxrank(timed(e2e_serial, args.steps))
    for c in [l[0] for l in lanes[1:]]:
        c.close()

    # ---- BASELINE configs[3] as written: 64 pairs in total, scattered from rank 0 over NCCL ----
    sharded = None
    if not args.no_extras:
        sharded = measure_sharded(args, prm, rank, world, local, stream, barrier, maxrank)

    if rank != 0:
        ctx.close()
        if world > 1:
            dist.destroy_process_group()
        return

    pix = B * world * H_ORG * W_ORG
    value = pix / (ms_res * 1e-3) / 1e6

    # ---- roofline of the dominant kernel (SOR), measured live with CUDA events ----
    ctx.set_graph_mode(False)
    roof = None
    try:
        prof = ctx.profile_kernels(B, steps=max(3, min(args.steps, 10)))
        peak, how = peaks()
        sor = prof["sor"]
        alg = 0
        for lv in range(prm.sc_l, prm.sc_f + 1):
            g = ctx.level_info(lv)
            alg += prm.tv_innerit * (lv + 1) * 44 * g["w"] * g["h"] * B  # bytes, SURVEY 8(d)
        ach = alg / (sor["ms_per_step"] * 1e-3) / 1e9
        traffic, issue = None, None
        tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp))
            traffic = tj.get("sor_dram_bytes_per_launch")
            # what actually bounds the overlapped step: warp-instruction issue.  ncu counts the warp
            # instructions of one step (profiles/r2_launches_step_b64.csv); an SM issues at most
            # 4 per cycle.  Utilisation = instructions / (step time x SMs x 4 x SM clock).
            wi = tj.get("warp_instructions_per_step")
            if wi and B == 64 and clocks.get("sm_mhz"):
                sms = torch.cuda.get_device_properties(local).multi_processor_count
                issue = {"warp_instructions_per_step": wi, "sms": sms, "sm_mhz": clocks["sm_mhz"],
                         "issue_slot_utilisation": wi / (ms_res * 1e-3 * sms * 4 * clocks["sm_mhz"] * 1e6),
                         "ipc_per_sm": wi / (ms_res * 1e-3 * sms * clocks["sm_mhz"] * 1e6)}
        # the other exact SOR kernel (ofdis_set_option "sor_lane" 1: flag-synchronised warps, no CTA barrier) on the same
        # batch, one stream: the engine picks it by itself for launches of up to 16 frames (batch_sweep below)
        lane_alt = None
        try:
            cl = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, B, device=local, stream=stream.cuda_stream)
            cl.set_option("sor_lane", 1)
            cl.upload_packed(0, B, host_in.data_ptr())
            cl.run(B)
            pl_ = cl.profile_kernels(B, steps=max(3, min(args.steps, 10)))
            cl.close()
            lane_alt = {"kernel": "sor_lane_kernel (same sweeps; warps of 32 rows x two-pixel blocks, shuffles + flag-synchronised "
                                  "shared-memory rings instead of a CTA barrier per super-step)",
                        "kernel_ms_per_step": pl_["sor"]["ms_per_step"], "achieved": alg / (pl_["sor"]["ms_per_step"] * 1e-3) / 1e9,
                        "frac": alg / (pl_["sor"]["ms_per_step"] * 1e-3) / 1e9 / peak,
                        "note": "faster per launch, but 200 KB of shared memory per CTA at the 56-row level: with ten streams "
                                "overlapping it costs 6 % of `value` (profiles/), so batches above 16 frames keep sor_wave_kernel"}
        except Exception as e:
            lane_alt = {"error": str(e)}
        roof = {"bound": "hbm", "kernel": "sor_wave_kernel (lexicographic SOR wavefront, all sweeps fused, one CTA per frame at this level size)", "achieved": ach,
                "sor_lane_kernel": lane_alt,
                "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic, "traffic_note": "ncu dram bytes per SOR launch with caches flushed before every replay (1.04x the "
                "algorithmic bytes); 0.32e6 with --cache-control none, i.e. behind assemble_kernel in the level loop "
                "(profiles/roofline_traffic.json)", "issue": issue, "peak_source": how,
                "algorithmic_bytes_per_step": alg, "kernel_ms_per_step": sor["ms_per_step"],
                "launches_per_step": sor["launches_per_step"],
                "share_of_step": {k: v["ms_per_step"] for k, v in prof.items()}}
    except Exception as e:  # profiling hook missing must not lose the headline numbers
        roof = {"bound": "hbm", "achieved": None, "peak": peaks()[0], "unit": "GB/s", "frac": None, "traffic": None,
                "error": str(e)}

    # ---- latency-bound small batches (configs[1] = one pair; configs[3]'s per-GPU shard = 8) ----
    sweep = {}
    if world == 1:
        for b in (1, 8):
            if b >= B:
                continue
            c2 = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, b, device=local,
                             stream=stream.cuda_stream)
            c2.upload_packed(0, b, host_in.data_ptr())
            c2.set_graph_mode(True)
            for _ in range(3):
                c2.run(b)
            ms = timed(lambda: c2.run(b), 10)

            def e2e_b():
                upload(c2, mode, b)
                c2.run(b)
                download(c2, mode, host_out, lanes[0][3], b)

            for _ in range(3):  # the first upload allocates the context's staging buffer
                e2e_b()
            ms2 = timed(e2e_b, 10)
            sweep[str(b)] = {"ms_per_step": ms, "value": b * H_ORG * W_ORG / (ms * 1e-3) / 1e6,
                             "e2e_ms_per_step": ms2, "e2e_value": b * H_ORG * W_ORG / (ms2 * 1e-3) / 1e6,
                             "sor_kernel": "sor_lane_kernel (engine default for launches of up to 16 frames)"}
            c2.close()
            c4 = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, b, device=local,
                             stream=stream.cuda_stream)
            c4.set_option("sor_lane", 0)  # A/B: the block wavefront (round 1/2 kernel) at the same batch
            c4.upload_packed(0, b, host_in.data_ptr())
            c4.set_graph_mode(True)
            for _ in range(3):
                c4.run(b)
            sweep[str(b)]["sor_wave_kernel_ms_per_step"] = timed(lambda: c4.run(b), 10)
            c4.close()
            if not args.no_extras:  # the same latency with the opt-in red-black refinement (see fast_mode)
                c3 = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, b, device=local,
                                 stream=stream.cuda_stream)
                c3.set_option("sor_fast", 1)
                c3.upload_packed(0, b, host_in.data_ptr())
                c3.set_graph_mode(True)
                for _ in range(3):
                    c3.run(b)
                sweep[str(b)]["fast_mode_ms_per_step"] = timed(lambda: c3.run(b), 10)
                c3.close()

    # ---- opt-in red-black refinement (ofdis_set_option "sor_fast"; NOT the reference's iterate) ----
    fast = None
    if world == 1 and not args.no_extras:
        try:
            from of_dis_b200 import synth as _synth
            fl = []
            for l in lanes:
                c = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, B, device=local, stream=l[1].cuda_stream)
                c.set_option("sor_fast", 1)
                c.upload_packed(0, B, host_in.data_ptr())
                c.set_graph_mode(True)
                fl.append(c)
            for i in range(NL * args.warmup):
                fl[i % NL].run(B)
            barrier()
            ms_fast = pipelined(lambda i: fl[i % NL].run(B), args.steps)
            ms_fast_single = timed(lambda: fl[0].run(B), args.steps)
            # the red-black solver against the same HBM roofline as the exact one: algorithmic bytes of the SOR
            # (SURVEY 8d: 44 bytes per pixel and solve) / event time of its launches in an eager pass
            fl[0].set_graph_mode(False)
            pf = fl[0].profile_kernels(B, steps=max(3, min(args.steps, 10)))
            fl[0].set_graph_mode(True)
            alg_f = sum(prm.tv_innerit * (lv + 1) * 44 * ctx.level_info(lv)["w"] * ctx.level_info(lv)["h"] * B
                        for lv in range(prm.sc_l, prm.sc_f + 1))
            ach_f = alg_f / (pf["sor"]["ms_per_step"] * 1e-3) / 1e9
            fast_flow = torch.empty((B, flow_floats), dtype=torch.float32)
            fl[0].get_flow_batch(0, B, fast_flow.data_ptr())
            fl[0].sync()
            gu, gv = _synth.synthetic_flow(H_ORG, W_ORG, 6.0, False)
            gt = np.stack([gu, gv], -1).astype(np.float32)
            n_chk = min(B, MAX_DISTINCT)
            epe = {"exact": [], "fast": []}
            dlt = []
            for f in range(n_chk):
                full = {}
                for key, src in (("exact", resident_flow), ("fast", fast_flow)):
                    full[key] = _pp.postprocess(src[f].numpy().reshape(li["h"], li["w"], prm.nop), prm.sc_l, pyrs[0].padw,
                                                pyrs[0].padh, W_ORG, H_ORG)
                    epe[key].append(float(np.sqrt(((full[key] - gt) ** 2).sum(-1)).mean()))
                dlt.append(float(np.abs(full["exact"] - full["fast"]).mean()))
            for c in fl:
                c.close()
            fast = {"value": pix / (ms_fast * 1e-3) / 1e6, "ms_per_step": ms_fast, "unit": "Mpix/s",
                    "single_lane_ms_per_step": ms_fast_single,
                    "sor_roofline": {"kernel": "sor_redblack_kernel (all sweeps of a solve in one launch, 32x32 tiles + halo in shared memory)",
                                     "kernel_ms_per_step": pf["sor"]["ms_per_step"], "launches_per_step": pf["sor"]["launches_per_step"],
                                     "achieved": ach_f, "unit": "GB/s", "frac": ach_f / peaks()[0],
                                     "note": "same algorithmic bytes as roofline.achieved; not the reference's iterate"},
                    "mean_abs_delta_px": float(np.mean(dlt)), "epe_exact_px": float(np.mean(epe["exact"])),
                    "epe_fast_px": float(np.mean(epe["fast"])), "pairs_checked": n_chk,
                    "note": "same linear systems, red-black instead of lexicographic sweep order: not bit-identical to the "
                            "reference and excluded from every parity claim and from value/e2e above; deltas at full resolution"}
        except Exception as e:
            fast = {"error": str(e)}

    numa.unbind(prev_affinity)  # the CPU baseline uses every core of the host
    cores = os.cpu_count() or 1
    threads = cores
    frames_u8 = np.ascontiguousarray(np.stack(FRAMES_U8[:min(B, MAX_DISTINCT)]))[..., None]  # [n][2][h][w][1]
    cpu = cpu_reference(prm, pyrs, frames_u8, args.cpu_seconds, threads) if world == 1 else None
    big = None
    if world == 1 and not args.no_extras:
        big = measure_big_configs()
    lead = dict(legs[mode])
    lead.update({"unit": "Mpix/s", "leg": mode, "host_numa_node": numa_node,
                 "flows_equal_resident_path": legs[mode]["result_checked_bitwise"],
                 "mode": "%d lanes (context+stream), step i on lane i %% lanes: copies and kernels of consecutive steps overlap" % NL,
                 "serial_ms_per_step": ms_e2e_serial, "serial_value": pix / (ms_e2e_serial * 1e-3) / 1e6,
                 "legs": legs})
    line = {
        "metric": "Mpix/s dense flow (1024x436, op-point 2)", "value": value, "unit": "Mpix/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_res, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "sustained": dict(sustained, value=pix / (sustained["ms_per_step"] * 1e-3) / 1e6, unit="Mpix/s",
                          note="the `value` loop run for >= 0.5 s (clocks in `clocks` cover it)"),
        "single_lane": {"ms_per_step": ms_res_single, "value": pix / (ms_res_single * 1e-3) / 1e6,
                        "note": "one context, one stream, L2 flushed before every step"},
        "e2e": lead,
        "gpu_launches": int(launches * args.steps), "gpu_launches_per_step": int(launches),
        "clocks": clocks, "roofline": roof, "batch_sweep": sweep, "sharded": sharded, "big_configs": big, "fast_mode": fast,
    }
    if cpu is not None:
        line["cpu_baseline"] = cpu
    print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
