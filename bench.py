#!/usr/bin/env python
"""bench.py - ResNet50 pipeline-partitioned inference throughput on N B200s (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # N = 1
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Queue items are single 224x224x3 images as in the reference (test/test.py:22,47-49).  The engine coalesces
`--coalesce` G in-flight items into one microbatch (one kernel-chain launch per stage, weights streamed once per
group; DEFER(coalesce=G)).  One bench "step" = one pass of the hot path over one such group through the whole
N-stage pipeline; `value` = K x G images / time of K steps.  Stage i lives on GPU i (one process per GPU under
torchrun); the cut list is the reference's for 8 stages (test/test.py:18) and SURVEY.md 8d's for 2 / 4.

Protocol (reference: count results inside a window while the chain stays flooded, test/test.py:25-36):
value  : inputs resident in the first stage's HBM slots; P pre-flood + W warm-up + K timed + T tail microbatches are
         issued back to back under back-pressure only; every stage records a CUDA event behind microbatch W-1 and
         behind microbatch W+K-1 on its own lanes - the device time between them is K steps of a FLOODED pipeline
         (never drained between warm-up and timing; fill and drain are outside the window).  Max over ranks.
e2e    : the same window measured on the host through the public API (DEFER.run_defer + queue.Queue): pinned host
         items, one H2D per item and one D2H per group inside the window; clock starts when result W*G arrives and
         stops when result (W+K)*G arrives while the feeder keeps the input queue full.
parity : the last e2e output of every arm is compared with the CPU oracle (checker only) -> `parity_rel_err`.
roofline / cpu_baseline : see DESIGN.md "Measurement".

--impl reference : the CPU port of the reference path (oracle/torch_cpu.py, all host cores) on the same
         workload - TensorFlow itself is not installable here (SURVEY.md 8c).

--dump-outputs DIR : after the timed pass, write what the last timed microbatch (W+K-1) returned to its caller,
         DIR/probs.npy (float32, G*B x 1000), so that two builds can be compared output for output on the same
         seeded weights and inputs.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import queue
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True     # the tree may be read-only: the bench writes nothing into it

import numpy as np  # noqa: E402


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="resnet50", choices=["resnet50", "resnet152", "vgg16"])
    ap.add_argument("--dtype", default="float32", choices=["float32", "float32_simt", "bfloat16"])
    ap.add_argument("--batch", type=int, default=1, help="samples per queue item (reference: 1)")
    ap.add_argument("--coalesce", type=int, default=0, help="queue items per engine microbatch; 0 = auto")
    ap.add_argument("--depth", type=int, default=0, help="in-flight microbatches (lanes) per stage; 0 = auto")
    ap.add_argument("--conv-backend", type=int, default=0)
    ap.add_argument("--cuts", default="reference", choices=["reference", "balanced"],
                    help="reference: test/test.py:18 list (8) / SURVEY 8d lists (2, 4); balanced: defer_b200.autocut "
                         "on per-op times measured on rank 0's GPU")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--batch1-roofline", action="store_true",
                    help="also time every op on a single-image microbatch (the un-coalesced launch)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the output of the last timed step to DIR/probs.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs:
        if args.impl != "b200":
            ap.error("--dump-outputs applies to --impl b200")
        os.makedirs(args.dump_outputs, exist_ok=True)
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, probs):
    """Write the arrays the timed path returned; a larger output keeps every k-th row so the file stays within
    DUMP_LIMIT_BYTES."""
    probs = np.ascontiguousarray(probs, np.float32)
    stride = -(-probs.nbytes // DUMP_LIMIT_BYTES)
    np.save(Path(out_dir) / "probs.npy", probs[::stride])


# engine defaults (measured on B200, profiles/README.md round 2): G queue items per launch, lanes per stage
DEFAULT_COALESCE = {"resnet50": 32, "resnet152": 16, "vgg16": 8}
DEFAULT_DEPTH = 4


def build_model(name):
    from defer_b200 import applications
    return {"resnet50": applications.ResNet50, "resnet152": applications.ResNet152, "vgg16": applications.VGG16}[name]()


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]),
                "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons, sampled every 50 ms from BEFORE any barrier or timed region until the end
    of the run (the fork/exec never sits inside a timed window); `window(t0, t1)` summarises the samples that arrived
    while the GPU was under load."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu_index, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.terminate)    # an error before stop() must not leave the sampler running
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, windows=()):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()

        def parse(lines):
            sm, smax, reasons = [], [], set()
            for _, ln in lines:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    smax.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            return sm, smax, reasons
        load = [(t, ln) for (t, ln) in self.lines if any(a - 0.05 <= t <= b + 0.1 for a, b in windows)]
        sm, smax, reasons = parse(load if load else self.lines)
        _, smax_all, _ = parse(self.lines)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax_all) if smax_all else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_total": len(self.lines),
                "note": "median over the samples that arrived during the e2e and device-timed passes (50 ms period)"}


# ----------------------------------------------------------------------------------------------- CPU port
def cpu_reference_run(model, n_stages, x, steps, warmup, seconds=None):
    """Times the oracle port of the reference path on the host cores.
    1 stage : test/local_infer.py:16-23 (predict in a loop).  N stages: test/test.py with threads standing in
    for nodes and an in-memory identity hop (the reference hop is a lossless codec)."""
    import torch
    from defer_b200 import applications, dag_util
    from oracle.torch_cpu import TorchCpuModel
    cuts = applications.default_cuts(model, n_stages)
    names = [model.input._keras_history[0].name] + cuts + [model.output._keras_history[0].name]
    parts = [dag_util.construct_model(model, names[i], names[i + 1], part_name=f"part{i+1}") for i in range(n_stages)]
    stages = [TorchCpuModel(p.to_json(), p.get_weights()) for p in parts]
    # torchrun exports OMP_NUM_THREADS=1; the baseline is meant to use the host's cores
    want = int(os.environ.get("DEFER_CPU_THREADS", "0")) or max(1, (os.cpu_count() or 2) // 2)
    if torch.get_num_threads() < want:
        torch.set_num_threads(want)
    cores = torch.get_num_threads()
    if n_stages == 1:
        for _ in range(warmup):
            stages[0].predict(x)
        t0 = time.perf_counter()
        n = 0
        while True:
            stages[0].predict(x)
            n += 1
            el = time.perf_counter() - t0
            if (seconds is not None and el >= seconds) or (seconds is None and (n >= steps or el > 90.0)):
                break
        dt = time.perf_counter() - t0
        return n / dt, dt / n * 1e3, cores, n
    torch.set_num_threads(max(1, cores // n_stages))   # N stage threads share the host cores
    qs = [queue.Queue(8) for _ in range(n_stages + 1)]
    stop = threading.Event()

    def put(q, item):
        while not stop.is_set():
            try:
                q.put(item, timeout=0.1)
                return True
            except queue.Full:
                continue
        return False

    def worker(i):
        while not stop.is_set():
            try:
                item = qs[i].get(timeout=0.1)
            except queue.Empty:
                continue
            if not put(qs[i + 1], stages[i].predict(item)):
                return

    def feeder():
        for _ in range(warmup + steps):
            if not put(qs[0], x):
                return

    ths = [threading.Thread(target=worker, args=(i,)) for i in range(n_stages)] + [threading.Thread(target=feeder)]
    for t in ths:
        t.start()
    for _ in range(warmup):
        qs[-1].get()
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        qs[-1].get()
        done += 1
        if time.perf_counter() - t0 > 90.0:      # bounded sample: stop counting after 90 s
            break
    dt = time.perf_counter() - t0
    stop.set()
    for t in ths:
        t.join()
    return done / dt, dt / done * 1e3, cores, done


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    model = build_model(args.model)
    from defer_b200 import applications
    x = applications.synthetic_input(args.batch)
    steps = min(args.steps, 400)
    val, ms, cores, n = cpu_reference_run(model, args.gpus, x, steps, max(3, min(args.warmup, 10)))
    val *= args.batch
    sample = f"{n} predict calls of {args.model} batch {args.batch}, {args.gpus} stage(s), torch CPU (oneDNN) port"
    line = {"impl": "reference", "metric": "inferences_per_sec", "value": val, "unit": "inferences/s",
            "n_gpus": args.gpus, "steps": n, "warmup": max(3, min(args.warmup, 10)), "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args),
            "cpu_baseline": {"value": val, "unit": "inferences/s", "cores": cores, "kind": "port", "sample": sample,
                             "note": "TensorFlow 1.x reference not installable (SURVEY.md 8c); oracle/torch_cpu.py port; "
                                     "one step = one predict call on one queue item"},
            "e2e": {"value": val, "unit": "inferences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "host_cpus": os.cpu_count()}
    print(json.dumps(line), flush=True)


def workload_config(args):
    """Identical for both arms: names the workload, not the engine (engine knobs are reported under `engine`)."""
    return {"workload": f"{args.model} {args.gpus}-stage pipeline, queue items of batch {args.batch}, 224x224x3 synthetic "
                        f"image, {'fp32 parity' if args.dtype != 'bfloat16' else 'bf16'}",
            "model": args.model, "stages": args.gpus, "batch": args.batch,
            "parallelism": f"pp{args.gpus}",
            "l2": "not flushed between steps: steady-state pipeline re-reads the same weights every microbatch by "
                  "design; the per-kernel roofline numbers are taken with a 256 MB L2 flush between launches"}


# ----------------------------------------------------------------------------------------------- B200 arm
def run_b200(args):
    from defer_b200 import _cabi
    _cabi.load(build_if_missing=False)   # before torch initialises CUDA (sets CUDA_DEVICE_MAX_CONNECTIONS)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()               # long before any barrier / timed region
    import torch
    from defer_b200 import applications, dag_util
    from defer_b200.dispatcher import DEFER
    from defer_b200.node import Node, StageRunner, pinned_empty

    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit(f"--gpus {args.gpus} needs torchrun with --nproc-per-node {args.gpus}")
        args.gpus = world
    n_stages = args.gpus
    G = args.coalesce or DEFAULT_COALESCE[args.model]
    K, W, B = args.steps, max(args.warmup, 3), args.batch
    # Lanes complete in round-robin bursts; the window [completion of W-1, completion of W+K-1] is exactly K steps of
    # steady state only when both marks sit on the same lane, i.e. K % depth == 0: auto depth = largest divisor of K
    # that is <= DEFAULT_DEPTH (an explicit --depth is honoured and reported as aligned or not).
    depth = args.depth or max(d for d in range(1, DEFAULT_DEPTH + 1) if K % d == 0)
    EB = G * B                                  # samples per engine microbatch

    ctx = None
    if world > 1:
        from defer_b200.dist import DistContext
        ctx = DistContext(ring=max(64, 4 * depth * world), out_elems=1000, batch=EB)
    torch.cuda.set_device(local_rank)

    model = build_model(args.model) if rank == 0 else None
    # G distinct-address pinned queue items holding the same synthetic image (the reference test enqueues one image
    # 1000 times, test/test.py:47-49), plus one resident microbatch for the device-timed pass
    x1 = applications.synthetic_input(B)
    items = []
    if rank == 0:
        for _ in range(max(2 * G, 8)):
            a = pinned_empty((B, 224, 224, 3))
            a[...] = x1
            items.append(a)
    x_group = pinned_empty((EB, 224, 224, 3))
    for g in range(G):
        x_group[g * B:(g + 1) * B] = x1

    # ---- build the pipeline through the public pieces (DEFER partition + dispatch)
    defer = DEFER(list(range(n_stages)), dtype=args.dtype, depth=depth, batch=B, coalesce=G, linger_us=200,
                  conv_backend=args.conv_backend, dist=ctx)
    max_inflight = depth * (world if ctx is not None else 1)
    in_q, out_q = queue.Queue(2 * max_inflight * G), queue.Queue(0)
    node_thread = None
    if ctx is not None:
        node = Node(dist_ctx=ctx, device=local_rank)
        node_thread = threading.Thread(target=node.run, name="defer-node", daemon=True)
        node_thread.start()
    t_defer = None
    cut_info = None
    if rank == 0:
        cuts = applications.default_cuts(model, n_stages)
        if args.cuts == "balanced" and n_stages > 1:
            from defer_b200 import autocut
            probe = StageRunner.from_model(model, device=local_rank, dtype=args.dtype, max_batch=EB, depth=1)
            try:
                op_us = [max(1.0, probe.time_op(i, iters=10, flush_l2=False) - 2.0) for i in range(len(probe.plan.ops))]
            finally:
                probe.close()
            cuts, stage_us = autocut.balanced_cuts(model, n_stages, op_costs=op_us)
            cut_info = {"policy": "balanced (defer_b200.autocut, measured per-op us)", "cuts": cuts,
                        "predicted_stage_us": [round(v, 1) for v in stage_us]}
        else:
            cut_info = {"policy": "reference list (test/test.py:18 for 8 stages; SURVEY 8d for 2/4)", "cuts": cuts}
        t_defer = threading.Thread(target=defer.run_defer, args=(model, cuts, in_q, out_q), daemon=True)
        t_defer.start()
        if not defer.wait_ready(600):
            raise SystemExit("pipeline did not come up")
        if defer._error:
            raise defer._error
    if ctx is not None:
        runner = ctx.local_runner()
    else:
        runner = defer.stages[0]
    my_stages = defer.stages if ctx is None else [runner]

    def barrier_sync():
        if ctx is not None:
            ctx.barrier()
        torch.cuda.synchronize()
        for r in my_stages:
            r.sync()

    result = {}
    windows = []
    T = max_inflight + 2                         # tail microbatches: the chain stays flooded past the end of the window
    # =========================================================================== e2e through DEFER + queues
    if not args.no_e2e:
        barrier_sync()
        n_items = (W + K + T) * G
        if rank == 0:
            def feed():
                for i in range(n_items):
                    in_q.put(items[i % len(items)])
            th = threading.Thread(target=feed, daemon=True)
            t_begin = time.perf_counter()
            th.start()
            last = None
            for _ in range(W * G):
                last = out_q.get(timeout=300)
            t0 = time.perf_counter()
            for _ in range(K * G):
                last = out_q.get(timeout=300)
            t1 = time.perf_counter()
            for _ in range(T * G):
                last = out_q.get(timeout=300)
            th.join()
            windows.append((t_begin, time.perf_counter()))
            dt = t1 - t0
            result["e2e"] = {"value": K * G * B / dt, "unit": "inferences/s", "h2d_bytes_per_step": int(x1.nbytes) * G,
                             "d2h_bytes_per_step": int(EB * 1000 * 4), "ms_per_step": dt / K * 1e3,
                             "items_per_step": G,
                             "timing": "host wall clock on the dispatcher rank from the arrival of result W*G to the arrival of "
                                       "result (W+K)*G in the output queue, input queue kept full before, during and after",
                             "api": "DEFER(coalesce=G).run_defer(model, cuts, queue.Queue, queue.Queue); items are single images"}
            result["probs_sum"] = float(np.asarray(last).sum())
            if not args.no_parity:
                # checker only (never timed): the CPU oracle on the same synthetic image
                from oracle.torch_cpu import TorchCpuModel
                ref = TorchCpuModel(model.to_json(), model.get_weights()).predict(np.asarray(x1))
                got = np.asarray(last, np.float32).reshape(ref.shape)
                result["parity_rel_err"] = float(np.max(np.abs(got - ref)) / np.max(np.abs(ref)))
                result["parity"] = {"rel_err": result["parity_rel_err"], "tolerance": 1e-3 if args.dtype != "bfloat16" else 6e-2,
                                    "against": "oracle/torch_cpu.py (CPU restatement), last e2e output of this arm",
                                    "argmax_match": bool(int(np.argmax(got)) == int(np.argmax(ref)))}
        barrier_sync()

    # =========================================================================== device-timed flooded steady state
    # Drive the stages directly (same lanes / graphs), input resident in the first stage's slots.
    seq0 = defer._submitted if rank == 0 else 0
    if ctx is not None:
        seq0 = int(ctx.max_over_ranks(seq0))
    if rank == 0:
        first = my_stages[0]
        for d in range(depth):
            first.submit(seq0 + d, x_group)   # lands in slot (seq0+d) % depth, stays there
        first.sync()
    P = 2 * max_inflight                       # pre-flood: every lane of every stage busy before the window opens
    total = P + W + K + T
    m0, m1 = seq0 + P + W - 1, seq0 + P + W + K - 1
    for r in my_stages:
        r.mark_after(m0, 0)
        r.mark_after(m1, 1)
    barrier_sync()

    def direct_pass(n, start, keep=None):
        """Issue n microbatches back to back, limited only by back-pressure (at most max_inflight in flight).
        One process: returns a copy of microbatch `keep`'s output (None if not asked for)."""
        if ctx is None:
            last_st = my_stages[-1]
            inflight = 0
            out = np.empty(last_st.out_shape, np.float32)
            kept = None
            for s in range(start, start + n):
                if inflight == depth:
                    last_st.result(s - depth, out)
                    if s - depth == keep:
                        kept = out.copy()
                    inflight -= 1
                for r in my_stages:
                    r.step(s)
                inflight += 1
            for s in range(start + n - inflight, start + n):
                last_st.result(s, out)
                if s == keep:
                    kept = out.copy()
            return kept
        # one process per GPU: rank 0 steps stage 0 and publishes `submitted`; node loops follow
        if rank == 0:
            for s in range(start, start + n):
                while s - ctx.done() >= max_inflight:
                    pass
                runner.step(s)
                ctx.mark_submitted(s + 1)
            while ctx.done() < start + n:
                time.sleep(20e-6)
        else:
            while ctx.done() < start + n and not ctx.stop_requested():
                time.sleep(200e-6)

    if ctx is not None and rank == 0:
        # results of the direct pass are published into the ring by the last rank; nobody consumes them, so move the
        # consumer cursor along (the ring guard would otherwise stall the publisher)
        stop_drain = threading.Event()

        def drain():
            while not stop_drain.is_set():
                ctx.hdr[6] = ctx.hdr[2]
                time.sleep(50e-6)
        threading.Thread(target=drain, daemon=True).start()
    tw0 = time.perf_counter()
    last_out = direct_pass(total, seq0, keep=m1 if args.dump_outputs else None)
    tw1 = time.perf_counter()
    windows.append((tw0, tw1))
    if args.dump_outputs and rank == 0:
        if ctx is not None:
            # the last rank published every result into the ring; the T < ring tail rows have not overwritten m1's
            last_out = ctx.results[m1 % ctx.ring].reshape(EB, -1)
        dump_outputs(args.dump_outputs, last_out)
    ms = max(r.mark_elapsed_ms() for r in my_stages)
    barrier_sync()
    if ctx is not None and rank == 0:
        stop_drain.set()
        ctx.hdr[6] = ctx.hdr[2]
    ms = ctx.max_over_ranks(ms) if ctx is not None else ms
    clocks = sampler.stop(windows) if rank == 0 else None
    launches = sum(r.num_kernels() for r in my_stages) * K
    launches = int(ctx.sum_over_ranks(launches)) if ctx is not None else launches

    # =========================================================================== roofline + CPU baseline (N=1 only)
    peaks = load_peaks()
    roofline = None
    stage_table = None
    roofline_b1 = None

    def op_table(r0, iters=10):
        rows = []
        for i in range(len(r0.plan.ops)):
            info = r0.op_info(i)
            info.update({"op": i, "us_cold": r0.time_op(i, iters=iters, flush_l2=True),
                         "us_hot": r0.time_op(i, iters=2 * iters, flush_l2=False)})
            # per-launch roofline time: the slower of algorithmic bytes / HBM peak and algorithmic flops / bf16 peak
            info["t_hbm_us"] = info["alg_bytes"] / (peaks["hbm_gbs"] * 1e3)
            info["t_tc_us"] = info["alg_flops"] / (peaks["bf16_tflops"] * 1e6)
            info["t_roof_us"] = max(info["t_hbm_us"], info["t_tc_us"])
            rows.append(info)
        return rows

    def roofline_of(rows, batch):
        conv = [r for r in rows if any(k in r["kernel"] for k in ("conv_umma", "conv_mega", "conv_stream")) and "stem" not in r["kernel"]]
        if not conv:
            conv = [r for r in rows if r["kernel"].startswith("conv")]
        groups = {}
        for r in conv:
            groups.setdefault(r["kernel"], []).append(r)
        name, grp = max(groups.items(), key=lambda kv: sum(r["us_cold"] for r in kv[1]))   # dominant kernel by time
        by = sum(r["alg_bytes"] for r in grp)
        fl = sum(r["alg_flops"] for r in grp)
        t_cold = sum(r["us_cold"] for r in grp) * 1e-6
        t_hot = sum(r["us_hot"] for r in grp) * 1e-6
        t_all = sum(r["us_hot"] for r in rows) * 1e-6
        hbm_bound = sum(r["t_hbm_us"] for r in grp) >= sum(r["t_tc_us"] for r in grp)
        best = max(grp, key=lambda r: r["t_roof_us"] / r["us_cold"])
        top = max(grp, key=lambda r: r["us_cold"])
        out = {"kernel": name, "launches_per_step": len(grp), "batch": batch,
               "bound": "hbm" if hbm_bound else "tensor",
               "achieved": by / t_cold / 1e9 if hbm_bound else fl / t_cold / 1e12,
               "peak": peaks["hbm_gbs"] if hbm_bound else peaks["bf16_tflops"],
               "unit": "GB/s" if hbm_bound else "TFLOP/s",
               "frac": (by / t_cold / 1e9 / peaks["hbm_gbs"]) if hbm_bound else (fl / t_cold / 1e12 / peaks["bf16_tflops"]),
               "traffic": None,
               "peak_source": peaks["source"] + " (burst: kernel timed alone)",
               "alg_bytes_per_step": by, "alg_flops_per_step": fl,
               "achieved_gbs": by / t_cold / 1e9, "achieved_tflops": fl / t_cold / 1e12,
               "frac_per_launch_roofline": sum(r["t_roof_us"] for r in grp) / (t_cold * 1e6),
               "hot_l2": {"achieved_gbs": by / t_hot / 1e9, "frac_per_launch_roofline": sum(r["t_roof_us"] for r in grp) / (t_hot * 1e6),
                          "note": "same launches back-to-back without L2 flush"},
               "share_of_step": t_hot / t_all if t_all else None,
               "best_launch": {"layers": best["layers"][:2], "us_cold": best["us_cold"], "alg_MB": best["alg_bytes"] / 1e6,
                               "alg_GF": best["alg_flops"] / 1e9, "frac": best["t_roof_us"] / best["us_cold"],
                               "bound": "hbm" if best["t_hbm_us"] >= best["t_tc_us"] else "tensor"},
               "top_launch": {"layers": top["layers"][:2], "us_cold": top["us_cold"], "us_hot": top["us_hot"],
                              "alg_bytes": top["alg_bytes"], "gbs_cold": top["alg_bytes"] / top["us_cold"] / 1e3},
               "method": "CUDA events on the launching stream, 10 launches per op, 256 MB L2 flush between launches; "
                         "frac = algorithmic bytes (or flops) / time / measured peak; frac_per_launch_roofline = "
                         "sum over launches of max(bytes/HBM, flops/bf16 peak) / sum of measured times"}
        return out

    if rank == 0 and not args.no_roofline and ctx is None:
        rows = op_table(my_stages[0])
        roofline = roofline_of(rows, EB)
        # DRAM traffic of the dominant kernel from the committed `ncu --set full` capture (per launch, like `achieved`):
        # well above the algorithmic bytes would mean wasted re-reads
        tpath = ROOT / "profiles" / "ncu_traffic.json"
        if tpath.exists():
            try:
                tr = json.loads(tpath.read_text())
                key = f"{args.model}_{args.dtype}_b{EB}"
                if key in tr:
                    roofline["traffic"] = tr[key]["traffic_bytes_per_launch"]
                    roofline["traffic_note"] = ("dram__bytes_read.sum + dram__bytes_write.sum per launch, mean of the launches in "
                                                + tr[key]["source"] + "; algorithmic bytes per launch (mean over the step) = "
                                                f"{roofline['alg_bytes_per_step'] / roofline['launches_per_step']:.0f}")
            except Exception:   # a malformed side file must not take the bench line down
                pass
        # the same algorithmic bytes over the TIMED REGION (all lanes overlapping): what the pipeline sustains, as
        # opposed to one launch timed alone behind an L2 flush
        try:
            conv_share = roofline["share_of_step"] or 1.0
            step_s = ms / K * 1e-3
            roofline["steady_state"] = {
                "achieved_gbs": roofline["alg_bytes_per_step"] / step_s / 1e9,
                "frac_of_hbm_peak": roofline["alg_bytes_per_step"] / step_s / 1e9 / peaks["hbm_gbs"],
                "achieved_tflops": roofline["alg_flops_per_step"] / step_s / 1e12,
                "note": "algorithmic bytes / flops of the conv launches of one step / ms_per_step of the timed region "
                        f"({depth} lanes in flight, L2 not flushed); conv launches are {conv_share:.2f} of the "
                        "summed per-launch time"}
        except Exception as e:   # an auxiliary figure must never cost the bench line
            roofline["steady_state"] = {"error": repr(e)}
        stage_table = [{"op": r["op"], "kernel": r["kernel"], "layers": r["layers"][:2], "us_cold": round(r["us_cold"], 2),
                        "us_hot": round(r["us_hot"], 2), "alg_MB": round(r["alg_bytes"] / 1e6, 3),
                        "alg_GF": round(r["alg_flops"] / 1e9, 4),
                        "frac_roof_cold": round(r["t_roof_us"] / r["us_cold"], 4)} for r in rows]
        if args.batch1_roofline and EB > 1:
            # the un-coalesced launch (one image per kernel): latency-bound by construction, reported for reference
            one = StageRunner.from_model(model, device=local_rank, dtype=args.dtype, max_batch=1, depth=1)
            try:
                roofline_b1 = roofline_of(op_table(one, iters=5), 1)
            finally:
                one.close()
    cpu_baseline = None
    if rank == 0 and not args.no_cpu and n_stages == 1:
        val, msc, cores, n = cpu_reference_run(model, 1, np.array(x1), 0, 3, seconds=args.cpu_seconds)
        cpu_baseline = {"value": val * B, "unit": "inferences/s", "cores": cores, "kind": "port",
                        "sample": f"{n} predict calls in {args.cpu_seconds:.0f} s of {args.model} batch {B} "
                                  "(oracle/torch_cpu.py, oneDNN, all host threads; test/local_infer.py protocol)",
                        "host_cpus": os.cpu_count()}

    # =========================================================================== shut down + report
    if rank == 0:
        defer.close()
    if ctx is not None:
        ctx.shutdown(node_thread)
    if rank == 0:
        line = {"metric": "inferences_per_sec", "value": K * EB / (ms * 1e-3), "unit": "inferences/s", "n_gpus": n_stages,
                "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": {"float32": "bf16x3->f32", "float32_simt": "f32", "bfloat16": "bf16"}[args.dtype],
                "data": "synthetic", "config": workload_config(args),
                "engine": {"coalesce": G, "images_per_step": EB, "depth": depth, "max_inflight": max_inflight,
                           "window_lane_aligned": K % depth == 0,
                           "preflood_steps": P, "tail_steps": T, "cuts": cut_info,
                           "step": "one pass of the N-stage hot path over one coalesced group of G single-image queue items"},
                "clocks": clocks, "gpu_launches": launches,
                "wall_ms_per_step_incl_fill_drain": (tw1 - tw0) / total * 1e3,
                "timing": "CUDA events per stage behind microbatch W-1 and W+K-1 of a flooded pipeline (never drained "
                          "between warm-up and timing), max over ranks"}
        line.update(result)
        if roofline is not None:
            line["roofline"] = roofline
            line["ops"] = stage_table
        if roofline_b1 is not None:
            line["roofline_batch1_launch"] = roofline_b1
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
