#!/usr/bin/env python
"""bench.py -- headline benchmark: ResNet-50 INT8 images/s through Net<NV,INT8>::prediction().

  python bench.py --gpus 1 --steps K --warmup W            (driver contract; N>1 under torchrun)
  python bench.py --impl reference ...                      (the CPU path timed on the host cores)

A "step" = one prediction() over one batch of synthetic 224x224 images per GPU.  At N=1 the
workload is BASELINE.json configs[1]: ResNet-50 INT8 batch=8 on 1xB200.  Multi-GPU = one full
replica per GPU (batch-sharded requests, weak scaling), model bytes broadcast from rank 0 over
NCCL, no collective in the per-step path.

JSON line keys: see DESIGN.md section "Measurement".  `value` is device-timed with the inputs
resident in HBM and an L2 flush between timed steps; `e2e` goes through the public API with
pinned host buffers (H2D + prediction + D2H every step).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")   # CPU-baseline arm: idle OpenMP threads sleep instead of spinning (see oracle/pyoracle.py)

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# algorithmic work per image (BASELINE.md section 2 / SURVEY.md section 8d)
MODEL_NAMES = {"resnet50": "ResNet-50", "resnet101": "ResNet-101", "vgg16": "VGG16", "mobilenet_v1": "MobileNet-v1"}
GOP_PER_IMAGE = {"resnet50": 7.716, "resnet101": 15.140, "vgg16": 30.94, "mobilenet_v1": 1.137, "tiny_resnet": 0.0}
# conv + fc weight elements (SURVEY.md section 8d), read once per batch at the operand width
WEIGHT_ELEMS = {"resnet50": 25.50e6, "resnet101": 44.5e6, "vgg16": 138.36e6, "mobilenet_v1": 4.2e6, "tiny_resnet": 0.0}
DTYPE_BYTES = {0: 2, 1: 4, 3: 1, 5: 4, 7: 1}   # saber DataType -> element bytes (AK_HALF, AK_FLOAT, AK_INT8, AK_INT32, AK_UINT8)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="resnet50")
    ap.add_argument("--precision", default="int8", choices=["int8", "fp32", "fp16"])
    ap.add_argument("--batch", type=int, default=8, help="images per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-l2-flush", action="store_true")
    ap.add_argument("--worker-threads", type=int, default=6,
                    help="threads (= Nets = streams) of the Worker the pipelined e2e leg serves requests with; 0 skips it")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<output name>.npy (inputs are seeded: two "
                         "builds run with the same arguments can be compared output for output)")
    return ap.parse_args()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """{name: array} -> dirname/<name>.npy in float32 (float64 kept). Past DUMP_LIMIT_BYTES in all, every array is cut to
    the same share of its rows (images), chosen with a fixed seed, so that two runs still write the same rows."""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: a if a.dtype == np.float64 else a.astype(np.float32) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_LIMIT_BYTES:
            rows = max(1, a.shape[0] * DUMP_LIMIT_BYTES // total)
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], rows, replace=False))]
        np.save(os.path.join(dirname, name + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0, period_ms=100):
        self.index = index
        self.period_ms = period_ms
        self.proc = None
        self.lines = []      # (host time, csv line)
        self.window = None   # (t0, t1): only samples inside it are reported when set

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", str(self.period_ms)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if self.window is not None and not (self.window[0] <= ts <= self.window[1]):
                continue
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_oracle_images_per_s(model, precision, batch, budget_s=20.0, steps=None, warmup=0):
    """The CPU path (oracle port of the x86 Saber semantics) on the host cores; bounded sample."""
    from anakin_b200 import modelzoo
    from oracle import model_walker as W
    from oracle import pyoracle as O
    O.build(ref=False)
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use the host's cores
    O.set_threads(min(os.cpu_count() or 1, 64))
    hw = 32 if model == "tiny_resnet" else 224
    g = modelzoo.build(model, batch=1, precision=precision if precision == "int8" else "fp32")
    scales = None
    if precision == "int8":
        scales = {k: float(np.float32(v)) for k, v in modelzoo.load_calibration(model).items()}
    per_img = max(0.05, GOP_PER_IMAGE.get(model, 1.0) / (150.0 if (precision == "int8" and O.vnni_available()) else 25.0))  # expected GOP/s on 8 cores
    auto_steps = steps is None
    if auto_steps:
        n_img = max(1, min(batch, int(budget_s / per_img / 3)))
        steps, warmup = 3, 0
    else:
        n_img = max(1, min(batch, int(120.0 / max(1, steps + warmup) / per_img)))
    x = modelzoo.synthetic_input(n_img, hw)
    # INT8 convs / fc through the AVX-512 VNNI implementation of the oracle's arithmetic where the CPU has it
    # (oracle/oracle_vnni.c: bit-identical to the scalar restatement, ~10x faster)
    vnni = precision == "int8" and O.vnni_available()
    wcache = {}
    avx512 = O.vnni_available()
    run = (lambda: W.run_int8(g, x, scales, fast=True, weight_cache=wcache)) if precision == "int8" else \
        (lambda: W.run_fp32(g, x, fast=avx512, weight_cache=wcache))
    run()      # fills the cache: BN fold, weight quantisation and packing are init-time work (Net::init), not timed
    for _ in range(warmup):
        run()
    if auto_steps:
        # one warm step sizes the sample: about a quarter of the budget, between 3 and 200 steps
        t0 = time.perf_counter()
        run()
        steps = int(min(200, max(3, budget_s / 4.0 / max(time.perf_counter() - t0, 1e-4))))
    out = None
    t0 = time.perf_counter()
    for _ in range(steps):
        out = run()
    dt = time.perf_counter() - t0
    return {"value": n_img * steps / dt, "unit": "images/s", "cores": O.num_threads(), "kind": "port", "outputs": out,
            "sample": "%d step(s) x %d image(s) of %s %s via oracle/model_walker.py (x86-semantics restatement, %s"
                      "OpenMP, not Anakin's MKL/xbyak build)" % (steps, n_img, model, precision,
                                                                  "AVX-512 VNNI convolutions on weights packed once, AVX-512 pooling, " if vnni else
                                                                  ("AVX-512 FMA convolutions on weights packed once, " if avx512 else "")),
            "ms_per_step": dt / steps * 1e3, "images_per_step": n_img}


LOGIT_NODE = {"tiny_resnet": "fc", "resnet50": "fc1000", "resnet101": "fc1000", "vgg16": "fc8", "mobilenet_v1": "fc7"}


def check_parity(net, model, prec, batch, rank):
    """Every rank compares what it just computed with the committed oracle goldens (tests/golden, made by
    tools/make_golden.py from the pinned CPU oracle): image i of rank r is golden image r*batch + i.
    INT8: logits bit-exact and top-1 equal; FP32: reference criterion on the logits and top-1 equal where the
    oracle's margin is clear. A mismatch aborts the benchmark: a fast wrong answer is not a result."""
    path = os.path.join(ROOT, "tests", "golden", "%s_golden.npz" % model)
    if not os.path.exists(path) or prec == "fp16":
        return {"checked_images": 0, "note": "no golden for this model / precision"}
    gold = np.load(path)
    key = "logits_int8" if prec == "int8" else "logits_fp32"
    if key not in gold:
        return {"checked_images": 0, "note": "no %s golden" % key}
    lo = rank * batch
    n = max(0, min(batch, gold[key].shape[0] - lo))
    if n == 0:
        return {"checked_images": 0, "note": "rank beyond the golden set"}
    arr, info = net.read_tensor(LOGIT_NODE[model])
    c = info["dims"][1]
    got = (arr[..., :c] if info["layout"] == 9 else arr).reshape(batch, -1)[:n]
    want = gold[key][lo:lo + n]
    top1 = net.get_output().argmax(1)[:n]
    if prec == "int8":
        ok = bool(np.array_equal(got, want)) and bool((top1 == gold["top1_int8"][lo:lo + n]).all())
        res = {"checked_images": int(n), "int8_logits_bit_exact": ok, "max_abs_diff": float(np.abs(got - want).max())}
    else:
        off = gold["logit_offset"]
        scale = float(np.abs(want + off).max())
        md = float(np.abs(got - want).max())
        srt = np.sort(want, axis=1)
        clear = (srt[:, -1] - srt[:, -2]) > 4 * md
        ok = md <= 2.5e-4 * scale and bool((top1[clear] == gold["top1_fp32"][lo:lo + n][clear]).all())
        res = {"checked_images": int(n), "fp32_logits_within_2.5e-4_of_scale": ok, "max_abs_diff": md, "logit_scale": scale}
    if not ok:
        raise SystemExit("bench.py: rank %d results differ from the oracle goldens: %s" % (rank, res))
    return res


def time_net(model, prec, batch, local_rank, steps, flush):
    """Device-timed ms per prediction() of another (model, batch) on this rank: CUDA-graph replay, L2 flushed."""
    import torch
    from anakin_b200 import anakin_bin, api, modelzoo
    G = api.Graph.from_bytes(anakin_bin.dumps(modelzoo.build(model, batch=batch, precision=prec if prec == "int8" else "fp32")))
    G.ResetBatchSize("input_0", batch)
    G.Optimize()
    net = api.Net(G, prec, device=local_rank)
    net.set_input("input_0", modelzoo.synthetic_input(batch, 224))
    for _ in range(5):
        net.prediction()
    net.sync()
    stream = torch.cuda.ExternalStream(net.stream, device=torch.device("cuda", local_rank))
    ms = 0.0
    with torch.cuda.stream(stream):
        for _ in range(steps):
            if flush is not None:
                flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            net.prediction()
            b.record(stream)
            b.synchronize()
            ms += a.elapsed_time(b)
    return ms / steps


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_oracle_images_per_s(args.model, args.precision, args.batch, steps=args.steps, warmup=args.warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r["outputs"])
    line = {"impl": "reference", "metric": "%s %s images/sec" % (MODEL_NAMES.get(args.model, args.model), args.precision.upper()),
            "value": r["value"], "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8" if args.precision == "int8" else ("f32" if args.precision == "fp32" else "f16"),
            "data": "synthetic",
            "config": {"workload": "%s %s, CPU oracle port, %d image(s)/step" % (args.model, args.precision, r["images_per_step"]),
                       "batch_per_step": r["images_per_step"]},
            "cpu_baseline": {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from anakin_b200 import anakin_bin, api, modelzoo, saber_abi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the product has no CPU path (use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    sab = saber_abi.load()
    model, prec, batch = args.model, args.precision, args.batch
    hw = 32 if model == "tiny_resnet" else 224

    # ---- model bytes: built on rank 0, broadcast to every replica over NCCL (NVLink)
    if rank == 0:
        blob = anakin_bin.dumps(modelzoo.build(model, batch=batch, precision=prec if prec == "int8" else "fp32"))
    else:
        blob = b""
    bcast_ms = 0.0
    if world > 1:
        from anakin_b200 import dist as adist
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        blob = adist.broadcast_bytes(blob, 0, device="cuda")
        torch.cuda.synchronize()
        bcast_ms = (time.perf_counter() - t0) * 1e3
    G = api.Graph.from_bytes(blob)
    G.ResetBatchSize("input_0", batch)
    G.Optimize()
    # replicas: rank 0 folds / quantises / packs the weights; the others only allocate (receive mode) and get the packed
    # arena -- every weight image, bias and scale table, one contiguous device buffer -- by ONE ncclBroadcast over NVLink
    arena_bytes, arena_ms = 0, 0.0
    t_init = time.perf_counter()
    if world > 1 and rank != 0:
        api.weight_arena_set_receive(True)
    net = api.Net(G, prec, device=local_rank)
    if world > 1:
        api.weight_arena_set_receive(False)
        init_ms = (time.perf_counter() - t_init) * 1e3
        arena_bytes, arena_ms = adist.broadcast_weight_arena(local_rank, 0)
    else:
        init_ms = (time.perf_counter() - t_init) * 1e3
    in_name, out_name = net.in_names[0], net.out_names[0]
    stream = torch.cuda.ExternalStream(net.stream, device=torch.device("cuda", local_rank))

    x = modelzoo.synthetic_input(batch, hw, seed=42 + rank * batch)
    x_pinned = torch.from_numpy(x).pin_memory()
    out_info = net.tensor_info(out_name)
    out_pinned = torch.empty(out_info["bytes"] // 4, dtype=torch.float32).pin_memory()
    net.set_input_ptr(in_name, x_pinned.data_ptr(), x_pinned.numel())
    l0 = sab.b200_launch_count()
    net.prediction()   # eager (builds tensor maps)
    net.sync()
    launches_per_step = int(sab.b200_launch_count() - l0)
    net.prediction()   # captures the CUDA graph
    net.sync()
    top1 = net.get_output().argmax(1)
    parity = check_parity(net, model, prec, batch, rank)

    flush = None if args.no_l2_flush else torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-timed steps, inputs resident, L2 flushed between steps (outside the event pairs)
    # (nvidia-smi needs a few hundred ms before its first line: start it before the warm-up so that it is already
    # sampling, every 25 ms, when the timed region begins; only samples inside the load window are reported)
    sampler = ClockSampler(local_rank, period_ms=25)
    if rank == 0:
        sampler.start()
    t_w = time.perf_counter()
    n_warm = 0
    while n_warm < max(3, args.warmup) or (rank == 0 and sampler.proc and not sampler.lines and time.perf_counter() - t_w < 2.0):
        net.prediction()
        n_warm += 1
        if n_warm % 16 == 0:
            net.sync()
    net.sync()
    K = args.steps
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    barrier()
    t_region0 = time.perf_counter()
    with torch.cuda.stream(stream):
        for i in range(K):
            if flush is not None:
                flush.zero_()
            starts[i].record(stream)
            net.prediction()
            stops[i].record(stream)
    barrier()
    t_region1 = time.perf_counter()
    if args.dump_outputs:
        suffix = "_rank%d" % rank if world > 1 else ""
        dump_outputs(args.dump_outputs, {name + suffix: net.get_output(name) for name in net.out_names})
    per_step = np.array([s.elapsed_time(e) for s, e in zip(starts, stops)])
    total_ms = float(per_step.sum())
    clocks_window = "timed region"
    if rank == 0 and sampler.proc and not any(t_region0 <= ts <= t_region1 for ts, _ in sampler.lines):
        # the timed region was shorter than the sampling period: keep the very same load running (untimed) until a
        # few samples have landed, and report those
        clocks_window = "same load continued right after the timed region (region shorter than the 25 ms sampling period)"
        t_c = time.perf_counter()
        with torch.cuda.stream(stream):
            while time.perf_counter() - t_c < 0.25:
                for _ in range(8):
                    if flush is not None:
                        flush.zero_()
                    net.prediction()
                net.sync()
        t_region1 = time.perf_counter()
    sampler.window = (t_region0, t_region1)

    # ---- back-to-back (warm L2) replay, for context
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(K):
            net.prediction()
        e1.record(stream)
    barrier()
    warm_ms = e0.elapsed_time(e1)

    # ---- end to end through the public API: pinned host in, H2D + prediction + D2H every step
    h2d = x_pinned.numel() * 4
    d2h = out_info["bytes"]
    for _ in range(3):
        net.set_input_ptr(in_name, x_pinned.data_ptr(), x_pinned.numel())
        net.prediction()
        net.read_tensor_into(out_name, out_pinned.data_ptr(), d2h)
    barrier()
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(K):
            net.set_input_ptr(in_name, x_pinned.data_ptr(), x_pinned.numel())   # H2D (async, net stream)
            net.prediction()
            net.read_tensor_into(out_name, out_pinned.data_ptr(), d2h)          # D2H + sync: result on host
        e1.record(stream)
    barrier()
    e2e_ms = e0.elapsed_time(e1)

    # ---- the same through Worker<NV,P>::async_prediction (framework/core/worker.h): T threads, each with its own
    # Net and stream, serve a queue of requests; every request still copies its input H2D from pinned memory and
    # its result D2H, but one request's copies overlap another's kernels. Timed on the host clock from the
    # first submit to the last result (the requests complete on the host).
    worker_ms = None
    T = args.worker_threads
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = clocks_window
    # the Worker leg is host-threaded: poll nvidia-smi slowly there (each query takes driver locks)
    sampler2 = ClockSampler(local_rank, period_ms=1000)
    if rank == 0 and T > 0 and not os.environ.get("BENCH_NO_SAMPLER_E2E"):
        sampler2.start()
    tmpdir = tempfile.TemporaryDirectory(prefix="bench_")    # the source tree may be read-only
    if T > 0:
        mpath = os.path.join(tmpdir.name, "model_rank%d.anakin.bin" % rank)
        with open(mpath, "wb") as f:
            f.write(blob)
        W = api.Worker(mpath, prec, threads=T, devices=[local_rank], batch=batch)
        W.wait_ready()
        depth = 2 * T
        xin = [torch.from_numpy(x).pin_memory() for _ in range(depth)]
        xout = [torch.empty(out_info["bytes"] // 4, dtype=torch.float32).pin_memory() for _ in range(depth)]

        def serve(nreq):
            inflight = 0
            for i in range(nreq):
                if inflight == depth:
                    W.async_get_result()
                    inflight -= 1
                j = i % depth
                W.async_prediction_ptr(xin[j].data_ptr(), xin[j].numel(), xout[j].data_ptr(), xout[j].numel())
                inflight += 1
            while inflight:
                W.async_get_result()
                inflight -= 1

        serve(max(6 * T, 100))     # every thread: eager run, graph capture, warm replays; steady clocks
        barrier()
        t0 = time.perf_counter()
        serve(K)
        worker_ms = (time.perf_counter() - t0) * 1e3
        barrier()
        worker_top1 = [int(v) for v in xout[(K - 1) % depth].numpy().reshape(batch, -1)[:, :int(out_info["dims"][1])].argmax(1)[:4]]
        del W
    clocks_e2e = sampler2.stop() if (rank == 0 and sampler2.proc) else None

    # ---- N > 1 extras: BASELINE config C4 (ResNet-101 INT8, GLOBAL batch 32 split over the GPUs: strong scaling),
    # and the in-process flavour of the replicas (one Worker, one thread per GPU) exercised once from rank 0
    c4 = None
    multi_worker = None
    if world > 1 and model == "resnet50" and prec == "int8" and 32 % world == 0:
        per_gpu = 32 // world
        barrier()
        c4_ms = time_net("resnet101", "int8", per_gpu, local_rank, max(10, K // 5), flush)
        t = torch.tensor([c4_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        c4 = {"model": "resnet101", "precision": "int8", "global_batch": 32, "batch_per_gpu": per_gpu,
              "ms_per_step": float(t.item()), "images_per_s": 32.0 / (float(t.item()) / 1e3), "scaling": "strong"}
        barrier()
        if rank == 0:
            W2 = api.Worker(mpath if T > 0 else None, prec, threads=world, devices=list(range(world)), batch=batch) if T > 0 else None
            if W2 is not None:
                W2.wait_ready()
                nreq = 8 * world
                ins = [torch.from_numpy(x).pin_memory() for _ in range(2 * world)]
                outs = [torch.empty(out_info["bytes"] // 4, dtype=torch.float32).pin_memory() for _ in range(2 * world)]
                for phase in range(2):
                    t0 = time.perf_counter()
                    inflight = 0
                    for i in range(nreq):
                        if inflight == 2 * world:
                            W2.async_get_result(); inflight -= 1
                        j = i % (2 * world)
                        W2.async_prediction_ptr(ins[j].data_ptr(), ins[j].numel(), outs[j].data_ptr(), outs[j].numel())
                        inflight += 1
                    while inflight:
                        W2.async_get_result(); inflight -= 1
                    dt = time.perf_counter() - t0
                multi_worker = {"api": "one Worker, %d threads, thread i on GPU i (in-process replicas)" % world,
                                "images_per_s": nreq * batch / dt, "requests": nreq}
                del W2
        barrier()

    # ---- per-op device times (eager, event pair per op) -> roofline of the dominant kernel
    prof = net.profile_ops(5, 20)
    conv_ms = sum(ms for _, op, ms in prof if op.startswith("Conv") or op == "Dense")
    all_ms = sum(ms for _, _, ms in prof)

    if world > 1:
        t = torch.tensor([total_ms, warm_ms, e2e_ms, worker_ms or 0.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, warm_ms, e2e_ms, wm = [float(v) for v in t.cpu()]
        worker_ms = wm if worker_ms is not None else None
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    P = peaks()
    images = K * batch * world
    value = images / (total_ms / 1e3)
    gop_step = GOP_PER_IMAGE.get(model, 0.0) * batch
    conv_launches = sum(1 for _, op, _ in prof if op.startswith("Conv") or op == "Dense")
    # the roofline is computed from the TIMED region: the conv / fc kernels' share of a step (from the per-op profile)
    # applied to the device-timed graph-replay step
    share = conv_ms / all_ms if all_ms else 0.0
    conv_ms_eager = conv_ms
    conv_ms = (total_ms / K) * share
    # tensor roof: kind::i8 runs at twice the bf16 rate; the measured bf16 GEMM peak x2 is the denominator
    mult = 2.0 if prec == "int8" else (1.0 if prec == "fp16" else 0.5)
    peak_tops = P["bf16_tflops"] * mult
    achieved_tops = (gop_step / 1e3) / (conv_ms / 1e3) if conv_ms > 0 else 0.0
    # HBM roof of the same launches: algorithmic bytes (SURVEY 8d) = per conv / fc op its input, residual and
    # output activations at their stored dtype (logical N*C*H*W, no padding), + the weights once per batch
    def act_bytes(node):
        ti = net.tensor_info(node)
        n_, c_, h_, w_ = ti["dims"]
        return n_ * c_ * h_ * w_ * DTYPE_BYTES.get(ti["dtype"], 4)
    alg_bytes = WEIGHT_ELEMS.get(model, 0.0) * (1 if prec == "int8" else (2 if prec == "fp16" else 4))
    for name, op, ins, _ in G.describe():
        if op.startswith("Conv") or op == "Dense":
            alg_bytes += act_bytes(name) + sum(act_bytes(i) for i in ins)
    achieved_gbs = (alg_bytes / 1e9) / (conv_ms / 1e3) if conv_ms > 0 else 0.0
    t_tensor_us = gop_step / peak_tops * 1e3 if peak_tops else 0.0          # GOP / (TOP/s) = ms -> us
    t_hbm_us = alg_bytes / (P["hbm_gbs"] * 1e9) * 1e6
    hbm_bound = t_hbm_us > t_tensor_us
    # e2e: every step = H2D of that step's input from pinned memory + prediction() + D2H of its result.
    # "serial": one Net, one request at a time (the latency view). Headline: the Worker serving a queue of
    # requests with T Nets / streams, so copies and kernels of different requests overlap.
    serial = {"value": images / (e2e_ms / 1e3), "ms_per_step": e2e_ms / K,
              "api": "Net::prediction(), one request at a time, CUDA-event timed"}
    if worker_ms is not None:
        e2e = {"value": images / (worker_ms / 1e3), "unit": "images/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": worker_ms / K,
               "api": "Worker<NV,%s>::async_prediction / async_get_result, %d threads (Nets, streams) per GPU, "
                      "%d requests in flight; host wall clock, first submit -> last result" % (prec.upper(), T, 2 * T),
               "top1_first": worker_top1, "serial": serial}
    else:
        e2e = dict(serial, unit="images/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h)
    # DRAM / L2 bytes per conv launch: from this round's `ncu --set full` capture of this same workload
    # (profiles/r02_conv_traffic.json, written by tools/ncu_traffic.py from the .ncu-rep; a bench run cannot profile itself)
    traffic = None
    traffic_l2 = None
    tpath = os.path.join(ROOT, "profiles", "r02_conv_traffic.json")
    if model == "resnet50" and prec == "int8" and batch == 8 and os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        traffic = tj.get("dram_bytes_per_launch")
        traffic_l2 = tj.get("lts_bytes_per_launch")
    line = {
        "metric": "%s %s images/sec" % (MODEL_NAMES.get(model, model), prec.upper()),
        "value": value, "unit": "images/s", "n_gpus": world, "steps": K, "warmup": max(3, args.warmup),
        "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8" if prec == "int8" else ("f32" if prec == "fp32" else "f16"), "data": "synthetic",
        "config": {"workload": "%s %s batch=%d per GPU, %dxB200, Net<NV,%s>::prediction() (CUDA-graph replay)" %
                               (model, prec.upper(), batch, world, prec.upper()),
                   "batch_per_gpu": batch, "global_batch": batch * world, "input": "fp32 NCHW [N,3,%d,%d]" % (hw, hw),
                   "l2": "flushed (256 MiB memset) between timed steps" if flush is not None else "not flushed",
                   "parallelism": "replica per GPU, batch-sharded; model bytes NCCL-broadcast (%.1f ms), packed weight arena %.1f MB in one "
                                  "ncclBroadcast (%.1f ms; Net init %.0f ms on this rank)" % (bcast_ms, arena_bytes / 1e6, arena_ms, init_ms)},
        "gpu_launches": launches_per_step * K,
        "launches_per_step": launches_per_step,
        "value_warm_l2": images / (warm_ms / 1e3),
        "ms_per_step_p50": float(np.median(per_step)), "ms_per_step_p99": float(np.percentile(per_step, 99)),
        "e2e": e2e,
        "roofline": {"bound": "hbm" if hbm_bound else "tensor",
                     "kernel": "conv_igemm_kernel / conv_slab_kernel (tcgen05 implicit GEMM, %d launches/step)" % conv_launches,
                     "achieved": achieved_gbs if hbm_bound else achieved_tops,
                     "peak": P["hbm_gbs"] if hbm_bound else peak_tops,
                     "unit": "GB/s" if hbm_bound else ("TOP/s" if prec == "int8" else "TFLOP/s"),
                     "frac": (achieved_gbs / P["hbm_gbs"]) if hbm_bound else (achieved_tops / peak_tops if peak_tops else None),
                     "traffic": traffic,
                     "traffic_l2": traffic_l2,
                     "traffic_unit": "DRAM (and L2) bytes per launch, mean over the step's conv launches (this round's cold-cache ncu capture)",
                     "algorithmic_bytes_per_launch": alg_bytes / conv_launches if conv_launches else None,
                     "algorithmic_gop_per_step": gop_step,
                     "lower_bound_us": {"tensor": t_tensor_us, "hbm": t_hbm_us},
                     "tensor": {"achieved": achieved_tops, "peak": peak_tops, "unit": "TOP/s" if prec == "int8" else "TFLOP/s",
                                "frac": achieved_tops / peak_tops if peak_tops else None,
                                "peak_source": "%s bf16 dense x%.1f" % (P["src"], mult)},
                     "hbm": {"achieved": achieved_gbs, "peak": P["hbm_gbs"], "unit": "GB/s",
                             "frac": achieved_gbs / P["hbm_gbs"], "peak_source": "%s device copy" % P["src"]},
                     "kernel_ms_per_step": conv_ms, "kernel_ms_per_step_eager_profile": conv_ms_eager,
                     "all_ops_ms_per_step_eager": all_ms,
                     "kernel_share_of_step": share},
        "clocks": clocks,
        "clocks_e2e": clocks_e2e,
        "top1_first": [int(v) for v in top1[:4]],
        "parity": parity,
        "cuda_graph": net.cuda_graph_active(),
    }
    if c4 is not None:
        line["strong_scaling_c4"] = c4
    if multi_worker is not None:
        line["worker_in_process_multi_gpu"] = multi_worker
    if world == 1 and not args.no_cpu_baseline:
        cb = cpu_oracle_images_per_s(model, prec, batch)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
