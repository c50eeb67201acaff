#!/usr/bin/env python
"""bench.py -- AlexNet product-quantized forward throughput (images/s) on N B200s, the metric of BASELINE.json.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A "step" is one PQ forward pass (23 layers: 8 PQ layers + ReLU/LRN/pool/softmax) over B synthetic 227x227x3 images
per GPU (default B = 256, BASELINE.json configs[2]; `--batch 1024` with --gpus 8 is configs[3]).  Images are
batch-sharded, weights replicated, and for N > 1 the only exchange is one all-gather of the [B,1000] logits
(NCCL over NVLink) inside the step.  One JSON line is printed by rank 0 (see the task contract):
  value     device-resident images/s, whole job (inputs already in HBM), CUDA events, max over ranks
  e2e       the same metric through the host-buffer C-ABI call qcnn_net_forward_h (pinned host in -> host out)
  roofline  dominant kernel: executed tensor flops (decode-at-use GEMM) or algorithmic bytes / CUDA-event time vs the
            measured peaks of MEASURED_PEAKS.json
  cpu_baseline  the reference's own CPU path timed on this box (rank 0, N = 1 only, bounded sample)
`--impl reference` times the reference CPU implementation with all host cores instead (no GPU work at all).
`--dump-outputs DIR` writes what the last timed step returned to its caller (rank 0: probabilities and logits) as
DIR/prob.npy and DIR/logits.npy, float32; the inputs depend only on the arguments, so two builds can be compared.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

IMG_CHW = (3, 227, 227)
IMG_LEN = 3 * 227 * 227
# ENUM_LyrType order (reference include/CaffePara.h:26)
CONV, POOL, FCNT, RELU, LORN, DRPT, SMAX = range(7)
# (layerInd: (kind, S, K, d, dims...)) of the shipped quantized AlexNet (SURVEY.md A.1 / A.3)
ALEXNET_PQ = {0: ("conv", 1, 128, 8, (96, 11, 11), 3 * 121), 4: ("conv", 6, 128, 8, (256, 5, 5), 48 * 25),
              8: ("conv", 32, 128, 8, (384, 3, 3), 256 * 9), 10: ("conv", 24, 128, 8, (384, 3, 3), 192 * 9),
              12: ("conv", 24, 128, 8, (256, 3, 3), 192 * 9), 15: ("fc", 2304, 32, 4, (4096,), 9216),
              18: ("fc", 1024, 32, 4, (4096,), 4096), 21: ("fc", 4096, 16, 1, (1000,), 4096)}
REAL_DIR = os.path.join(ROOT, "oracle", "_ref", "data", "AlexNet", "Bin.Files")
REAL_PFX = "bvlc_alexnet_aCaF"


# ---------------------------------------------------------------------------------------------------------------
# synthetic data
# ---------------------------------------------------------------------------------------------------------------
def lcg_tables(n):
    """A[i], C[i] with s_{i+1..} : s_i = A[i]*s_0 + C[i] (mod 2^32) for the LCG s <- 1664525 s + 1013904223."""
    a, c = np.uint64(1664525), np.uint64(1013904223)
    mask = np.uint64(0xFFFFFFFF)
    A = np.empty(n, np.uint64)
    Cc = np.empty(n, np.uint64)
    A[0], Cc[0] = a, c
    m = 1
    while m < n:
        k = min(m, n - m)
        # step m+i = (step m) after (step i):  A = A[i]*A[m-1]..., composed as affine maps
        A[m:m + k] = (A[:k] * A[m - 1]) & mask
        Cc[m:m + k] = (A[:k] * Cc[m - 1] + Cc[:k]) & mask
        m += k
    return A, Cc


def lcg_images(n, seed0, tables=None):
    """SURVEY.md 8(d): image i has seed seed0+i; x = ((s>>8)&0xFFFF)/65536*256 - 128 after every update."""
    A, Cc = tables if tables is not None else lcg_tables(IMG_LEN)
    out = np.empty((n, IMG_LEN), np.float32)
    mask = np.uint64(0xFFFFFFFF)
    for i in range(n):
        s = (A * np.uint64((seed0 + i) & 0xFFFFFFFF) + Cc) & mask
        out[i] = ((s >> np.uint64(8)) & np.uint64(0xFFFF)).astype(np.float32) / np.float32(65536.0) * np.float32(256.0) \
            - np.float32(128.0)
    return out.reshape((n,) + IMG_CHW)


def write_synthetic_alexnet(writer, dirpath, pfx, seed=1):
    """Random-init parameters of the AlexNet PQ architecture in the reference's .bin/.cbn formats.  `writer` supplies
    write_bin_f32 / write_cbn_u8: the product's own writers on the B200 arm (qcnn_write_bin_f32 / qcnn_write_cbn_u8),
    the oracle's on the reference arm (which must not load the product library).  Codebooks ~ N(0, 1/fan_in)."""
    rng = np.random.RandomState(seed)
    os.makedirs(dirpath, exist_ok=True)
    for l, (kind, S, K, d, odims, fan) in sorted(ALEXNET_PQ.items()):
        nout = odims[0]
        asmt = rng.randint(0, K, size=tuple(odims) + (S,)).astype(np.uint8)
        bias = (rng.randn(nout) * 0.05).astype(np.float32)
        ctrd = (rng.randn(S, K, d) * (1.0 / np.sqrt(fan))).astype(np.float32)
        if l == 21:
            ctrd *= np.float32(0.25)  # keep logits inside expf range: the reference softmax has no max subtraction
        bits = int(np.ceil(np.log2(K)))
        base = os.path.join(dirpath, pfx)
        writer.write_bin_f32("%s.biasVec.%02d.bin" % (base, l + 1), bias)
        writer.write_bin_f32("%s.ctrdLst.%02d.bin" % (base, l + 1), ctrd)
        writer.write_cbn_u8("%s.asmtLst.%02d.cbn" % (base, l + 1), asmt, bits)


class _OracleWriter(object):
    """File writers of the CPU oracle (reference arm only)."""

    @staticmethod
    def write_bin_f32(path, arr):
        from oracle import pyoracle as po
        po.write_bin(path, np.ascontiguousarray(arr, np.float32))

    @staticmethod
    def write_cbn_u8(path, idx0, bits):
        from oracle import pyoracle as po
        po.write_cbn(path, idx0, bits)


def model_files(writer, tmpdir):
    """The reference's shipped AlexNet files when they were staged next to the compiled reference, else synthetic."""
    if os.path.exists(os.path.join(REAL_DIR, REAL_PFX + ".asmtLst.22.cbn")):
        return REAL_DIR, REAL_PFX, "shipped quantized AlexNet (bvlc_alexnet_aCaF)"
    write_synthetic_alexnet(writer, tmpdir, "synth")
    return tmpdir, "synth", "random-init AlexNet PQ architecture"


DUMP_LIMIT = 64 << 20


def dump_outputs(dirpath, arrays):
    """Writes every array as dirpath/<name>.npy in float32.  Above DUMP_LIMIT bytes in all, each keeps the same fixed,
    seeded sample of its rows, so that dumps of two runs with the same arguments line up row for row."""
    os.makedirs(dirpath, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_LIMIT:
            keep = max(1, a.shape[0] * DUMP_LIMIT // total)
            a = a[np.sort(np.random.RandomState(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(dirpath, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler(object):
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(np.max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------------
# CPU reference legs (the only place bench.py touches oracle/)
# ---------------------------------------------------------------------------------------------------------------
def _ref_worker_loop(conn, dirpath, pfx, cpu):
    """One reference worker: pinned to one host thread, owns one CaffeEva object (the reference has no batching and no
    threading of its own: kDataCntInBatch = 1), serves (seed0, count) requests until told to stop."""
    try:
        os.sched_setaffinity(0, {cpu})
    except (AttributeError, OSError):
        pass
    from oracle import pyoracle as po
    if po.have_ref():
        net = po.RefNet(dirpath, pfx)
    else:
        net = ("port", po.alexnet_layers(), po.load_model(dirpath, pfx, po.alexnet_layers()))
    conn.send("ready")
    while True:
        req = conn.recv()
        if req is None:
            break
        seed0, count = req
        imgs = po.lcg_images(count, seed0)
        t0 = time.perf_counter()
        acc = 0.0
        for i in range(count):
            if isinstance(net, tuple):
                p = po.net_forward(net[1], net[2], imgs[i:i + 1])[0]
            else:
                p = net.forward(imgs[i])
            acc += float(p[0])
        conn.send((time.perf_counter() - t0, acc))
    conn.close()


def cpu_reference_single_thread(dirpath, pfx, images, warmup=2):
    """The reference's CalcFeatMap path, ONE pinned thread, batch 1 (it has no batching: kDataCntInBatch = 1)."""
    from oracle import pyoracle as po
    saved = None
    try:
        saved = os.sched_getaffinity(0)
        os.sched_setaffinity(0, {sorted(saved)[-1]})
    except (AttributeError, OSError):
        pass
    kind = "reference" if po.have_ref() else "port"
    imgs = po.lcg_images(min(images, 8), 12345)
    if kind == "reference":
        net = po.RefNet(dirpath, pfx)
        tot, each = net.time_forward(imgs, warmup, images)
        net.close()
        ms = np.asarray(each)
    else:
        layers = po.alexnet_layers()
        params = po.load_model(dirpath, pfx, layers)
        ms = []
        for i in range(warmup + images):
            t0 = time.perf_counter()
            po.net_forward(layers, params, imgs[i % len(imgs):i % len(imgs) + 1])
            if i >= warmup:
                ms.append((time.perf_counter() - t0) * 1e3)
        ms = np.asarray(ms)
    try:
        if saved:
            os.sched_setaffinity(0, saved)
    except (AttributeError, OSError):
        pass
    return kind, float(np.median(ms)), float(ms.min())


def run_reference_arm(args):
    """--impl reference: the reference CPU implementation on all host cores (one process per core, batch 1 each).
    Loads nothing of the product: no libqcnn_b200.so, no torch, no GPU work."""
    import multiprocessing as mp
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import pyoracle as po
    tmp = tempfile.mkdtemp(prefix="qcnn_ref_")
    dirpath, pfx, what = model_files(_OracleWriter, tmp)
    cpus = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))
    cores = len(cpus)
    per_core = 8                       # images per worker per step: ~0.5 s of CPU work per step
    sample = cores * per_core          # images per step
    ctx = mp.get_context("fork")
    workers = []
    for c in cpus:                     # one pinned process per host thread, each with its own network object
        parent, child = ctx.Pipe()
        pr = ctx.Process(target=_ref_worker_loop, args=(child, dirpath, pfx, c), daemon=True)
        pr.start()
        workers.append((pr, parent))
    for _, conn in workers:
        assert conn.recv() == "ready"

    def step(seed):
        # the step's wall time is what a caller of the whole host sees; per-worker compute times are kept for the record
        t0 = time.perf_counter()
        for w, (_, conn) in enumerate(workers):
            conn.send((seed + w * per_core, per_core))
        busy = [conn.recv()[0] for _, conn in workers]
        return time.perf_counter() - t0, float(np.max(busy))
    for w in range(max(1, args.warmup)):
        step(1000 + w * sample)
    res = [step(5000 + k * sample) for k in range(args.steps)]
    times = [r[0] for r in res]
    for pr, conn in workers:
        conn.send(None)
    for pr, conn in workers:
        pr.join(timeout=10)
    total = float(np.sum(times))
    value = sample * args.steps / total
    kind = "reference" if po.have_ref() else "port"
    line = {
        "impl": "reference", "metric": "alexnet_pq_forward_images_per_s", "value": value, "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, what, args.gpus),
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": kind,
                         "sample": "%d images per step (%d per host thread, batch 1 each, one pinned process per thread), "
                                   "%d steps, slowest worker %.2f s of %.2f s/step"
                                   % (sample, per_core, args.steps, float(np.mean([r[1] for r in res])), total / args.steps)},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def workload_config(args, what, world):
    return {"workload": "AlexNet PQ forward (CalcFeatMap_ConvAprx/_FCntAprx path), batch %d per GPU, synthetic "
                        "227x227x3 LCG images" % args.batch,
            "global_batch": args.batch * world, "per_gpu_batch": args.batch, "parallelism": "dp%d" % world,
            "weights": what, "collective": "all_gather(logits [B,1000]) on a side stream, overlapped with the next step" if world > 1 else "none",
            "l2": "inputs (%.0f MB/step) exceed the 126 MB L2; two input sets alternate" % (args.batch * IMG_LEN * 4 / 1e6)}


# ---------------------------------------------------------------------------------------------------------------
# the B200 arm
# ---------------------------------------------------------------------------------------------------------------
def run_b200_arm(args, q):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    if args.gpus > 1 and world == 1:
        raise SystemExit("launch multi-GPU runs with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    B = args.batch

    tmp = tempfile.mkdtemp(prefix="qcnn_bench_r%d_" % rank)
    dirpath, pfx, what = model_files(q, tmp)
    ctx = q.Context(local)
    net = q.Net(ctx, dirpath, pfx, "AlexNet")

    # NUMA placement of the pinned staging buffers: run this rank on the CPUs next to its GPU (NVML's ideal affinity)
    # before anything is pinned -- on a two-socket host a remote pinned buffer copies at ~30 instead of ~55 GB/s
    # (tools/h2d_bw.py), and the end-to-end number is bound by that copy
    numa = "unbound"
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
        numa = "bound to %d GPU-local cpus" % len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001  (no NVML / not permitted: keep the default placement)
        pass

    # two alternating input sets per rank (distinct images per rank), generated on the host, pinned
    tables = lcg_tables(IMG_LEN)
    host_in = [torch.from_numpy(lcg_images(B, 12345 + (rank * 2 + s) * B, tables)).pin_memory() for s in range(2)]
    dev_in = [h.to(dev, non_blocking=False) for h in host_in]
    host_out = torch.empty((B, 1000), dtype=torch.float32).pin_memory()
    prob = torch.empty((B, 1000), dtype=torch.float32, device=dev)
    logits = torch.empty((B, 1000), dtype=torch.float32, device=dev)
    sharding = importlib.import_module("quantized-cnn_b200.sharding")

    # the path's only exchange: all-gather of the [B,1000] logits (NCCL over NVLink), on a side stream so that it overlaps
    # the next step's first layers (every step still includes its own gather: the timed region ends with a device sync)
    gather = sharding.OverlappedGather(B, 1000, world, dev) if world > 1 else None

    def step(i):
        if world > 1:
            net.forward(dev_in[i & 1], prob=prob, logits=gather.rows(i))
            gather.launch(i)
        else:
            net.forward(dev_in[i & 1], prob=prob, logits=logits)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for w in range(max(args.warmup, 3)):
        step(w)
    barrier()
    launches_per_step = net.launch_count()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    in_range = os.environ.get("QCNN_PROFILE_RANGE") == "1"   # ncu --profile-from-start off: launch list of the timed steps only
    if in_range:
        torch.cuda.cudart().cudaProfilerStart()
    e0.record()
    for k in range(args.steps):
        step(k)
    e1.record()
    barrier()
    if in_range:
        torch.cuda.cudart().cudaProfilerStop()
    if args.dump_outputs and rank == 0:
        # what the last step's caller received: this rank's probabilities and the logits (gathered over all ranks)
        last_logits = gather.full[(args.steps - 1) & 1] if world > 1 else logits
        dump_outputs(args.dump_outputs, {"prob": prob.cpu().numpy(), "logits": last_logits.cpu().numpy()})
    ms_total = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
    ms_total = float(ms_total.item())
    value = world * B * args.steps / (ms_total * 1e-3)

    # ---- end-to-end through the host-buffer C-ABI calls (copies inside the timed region, every step) ----
    # headline: uint8 pixels in (what a BMP decodes to; (float)pixel - mean happens on the device), top-5 out (the k-fold
    # arg-max of CaffeEvaWrapper::Proc on the device) -- qcnn_net_forward_u8_h; also the fp32-tensor entry of
    # CaffeEva::ExecForwardPass(img, prob) -- qcnn_net_forward_h -- which moves 4x the bytes up and whole rows down
    def time_host(fn):
        for w in range(3):
            fn(w)
        barrier()
        t0 = time.perf_counter()
        for k in range(args.steps):
            fn(k)
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return world * B * args.steps / float(t.item())
    e2e_f32 = time_host(lambda k: net.forward_host(host_in[k & 1], host_out))
    # pixels: the same LCG stream, one byte per value, constant mean 128 => inputs in [-128, 127] like the fp32 images
    rs = np.random.RandomState(777 + rank)
    host_u8 = [torch.from_numpy(rs.randint(0, 256, size=(B, 227, 227, 3)).astype(np.uint8)).pin_memory() for s_ in range(2)]
    net.set_input_mean(np.full(IMG_CHW, 128.0, np.float32))
    top_i = torch.empty((B, 5), dtype=torch.int32).pin_memory()
    top_p = torch.empty((B, 5), dtype=torch.float32).pin_memory()
    e2e_sync = time_host(lambda k: net.forward_u8_host(host_u8[k & 1], k=5, idx_h=top_i, val_h=top_p))
    # headline: the asynchronous form of the same call with two steps in flight (qcnn_net_submit_u8_h / qcnn_net_wait):
    # step i+1's pixels cross the host link while step i computes.  Every step still copies its own inputs up and its
    # own top-5 down inside the timed region; the region ends after the last ticket has been waited for.
    top_i2 = [top_i, torch.empty((B, 5), dtype=torch.int32).pin_memory()]
    top_p2 = [top_p, torch.empty((B, 5), dtype=torch.float32).pin_memory()]

    def run_async(steps):
        pending = []
        for k in range(steps):
            if len(pending) == 2:
                net.wait(pending.pop(0))
            pending.append(net.submit_u8_host(host_u8[k & 1], k=5, idx_h=top_i2[k & 1], val_h=top_p2[k & 1]))
        for t in pending:
            net.wait(t)
    run_async(4)
    barrier()
    t0 = time.perf_counter()
    run_async(args.steps)
    torch.cuda.synchronize()
    ta = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ta, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / float(ta.item())
    clocks = sampler.stop() if rank == 0 else None

    # ---- per-layer CUDA-event profile (separate pass: events between kernels) -> dominant kernel + roofline ----
    net.set_profiling(True)
    nl = net.layer_count
    acc = np.zeros(nl)
    reps = max(3, min(args.steps, 10))
    net.forward(dev_in[0], prob=prob)   # un-timed: lets any (re-)tuning for this batch size happen outside the profile
    torch.cuda.synchronize()
    for k in range(reps):
        net.forward(dev_in[k & 1], prob=prob)
        torch.cuda.synchronize()
        acc += np.array([net.layer_time_ms(l) for l in range(nl)])
    net.set_profiling(False)
    layer_ms = acc / reps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    names = {0: "conv1", 4: "conv2", 8: "conv3", 10: "conv4", 12: "conv5", 15: "fc6", 18: "fc7", 21: "fc8",
             2: "lrn1+pool1", 6: "lrn2+pool2", 14: "pool5", 22: "softmax"}
    per_layer = {}
    for l in range(nl):
        if layer_ms[l] <= 0:
            continue
        w = net.layer_work(l, B)
        per_layer[names.get(l, "layer%d" % l)] = {
            "ms": round(float(layer_ms[l]), 4), "alg_GBps": round(w["alg_bytes"] / (layer_ms[l] * 1e-3) / 1e9, 2),
            "lookups_per_s": round(w["lookups"] / (layer_ms[l] * 1e-3), 1) if w["lookups"] else 0}
    pq_layers = [l for l in ALEXNET_PQ if layer_ms[l] > 0]
    dom = max(pq_layers, key=lambda l: layer_ms[l])
    wd = net.layer_work(dom, B)
    sm_clk = (clocks or {}).get("sm_mhz") or float(peaks.get("sm_max_mhz", 1965.0))
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(names[dom])
    except (OSError, ValueError, KeyError):
        pass

    # Tensor-core work of a pq_gemm_tc launch, from the plan the library reports: every CTA runs `ksteps` k-steps of
    # three kind::tf32 MMAs (3xTF32) of 128 channels x NT positions x 8 (DESIGN.md 5): executed MACs, padding included.
    import re

    def tc_macs(l):
        # executed MACs of the launch, padding included: per k-step (8 input values) either THREE kind::tf32 MMAs of
        # 128 x NT x 8 (3xTF32 operands) or TWO kind::f16 MMAs of 128 x NT x 16 (bf16x2 operands, the default)
        d = net.pq_layer(l).describe(B)
        m = re.search(r"pq_gemm_tc.*?NT=(\d+).*?grid=(\d+).*?ksteps=(\d+)", d)
        if not m:
            return None
        per_kstep = 2.0 * 16.0 if "bf16x2" in d else 3.0 * 8.0
        return float(m.group(2)) * float(m.group(3)) * per_kstep * 128.0 * float(m.group(1))

    def tc_is_bf(l):
        return "bf16x2" in net.pq_layer(l).describe(B)
    for l in pq_layers:
        tm = tc_macs(l)
        if tm:
            per_layer[names[l]]["tensor_TFLOPs_executed"] = round(2.0 * tm / (layer_ms[l] * 1e-3) / 1e12, 1)
    ach_gbs = wd["alg_bytes"] / (layer_ms[dom] * 1e-3) / 1e9
    dom_macs = tc_macs(dom)
    # SURVEY.md 8(d): the declared roofline of every kernel of this path is HBM -- algorithmic bytes of the launch over
    # its CUDA-event time against the measured copy bandwidth.  That is `frac`.  The batched kernels are NOT bound by HBM
    # (DESIGN.md 5): what limits the dominant launch is in `tensor` (decode-at-use GEMM: executed 3xTF32 flops incl.
    # padding, and the useful dense-equivalent flops, against measured bf16 / 2) or in `gather` (LUT + gather family).
    roofline = {"bound": "hbm", "kernel": ("pq_gemm_tc_kernel (%s)" if dom_macs else "%s") % names[dom],
                "achieved": round(ach_gbs, 2), "peak": hbm_peak, "unit": "GB/s", "frac": round(ach_gbs / hbm_peak, 5),
                "traffic": traffic, "peak_source": peak_src, "alg_bytes_per_launch": wd["alg_bytes"],
                "ms_per_launch": round(float(layer_ms[dom]), 4),
                "definition": "SURVEY.md 8(d) algorithmic bytes per launch / CUDA-event time of that launch / measured HBM peak"}
    if dom_macs:
        # tf32 MMAs run at half the bf16 rate: peak = measured dense bf16 (cuBLAS, MEASURED_PEAKS.json) / 2
        bf16 = float(peaks.get("bf16_tflops", 1650.0))
        peak_tc = bf16 if tc_is_bf(dom) else bf16 / 2.0     # kind::tf32 issues at half the bf16 rate
        ach = 2.0 * dom_macs / (layer_ms[dom] * 1e-3) / 1e12
        dense = {0: 105415200.0, 4: 223948800.0, 8: 149520384.0, 10: 112140288.0, 12: 74760192.0,
                 15: 37748736.0, 18: 16777216.0, 21: 4096000.0}       # dense-equivalent MACs per image (SURVEY.md App. C)
        useful = 2.0 * dense[dom] * B / (layer_ms[dom] * 1e-3) / 1e12
        all_tc = [(tc_macs(l), layer_ms[l]) for l in pq_layers if tc_macs(l)]
        roofline["tensor"] = {
            "executed_TFLOPs": round(ach, 1), "useful_TFLOPs": round(useful, 1), "peak_TFLOPs": round(peak_tc, 1),
            "frac_executed": round(ach / peak_tc, 4), "frac_useful": round(useful / peak_tc, 4),
            "flops_per_launch_executed": 2.0 * dom_macs, "flops_per_launch_useful": 2.0 * dense[dom] * B,
            "operands": "bf16x2 (two kind::f16 MMAs of K = 16 per k-step)" if tc_is_bf(dom) else "3xTF32 (three kind::tf32 MMAs of K = 8 per k-step)",
            "peak_source": ("MEASURED_PEAKS.json bf16_tflops" if "bf16_tflops" in peaks else "fallback 1650") +
                           ("" if tc_is_bf(dom) else " / 2 (kind::tf32 issues at half the bf16 rate)"),
            "all_pq_gemm_launches": {"launches": len(all_tc),
                                     "executed_TFLOPs": round(sum(2.0 * m for m, _ in all_tc) / (sum(t for _, t in all_tc) * 1e-3) / 1e12, 1),
                                     "ms": round(float(sum(t for _, t in all_tc)), 4)},
            "note": "executed = CTAs x k-steps x MMAs per k-step x 2*128*NT*K, padding included; useful = dense-equivalent MACs"}
    else:
        gather_peak = 32.0 * ctx.sm_count * sm_clk * 1e6       # conflict-free 4-byte shared-memory lookups per second
        roofline["gather"] = {"resource": "shared-memory gather (32 lookups/clk/SM)",
                              "achieved_lookups_per_s": wd["lookups"] / (layer_ms[dom] * 1e-3),
                              "peak_lookups_per_s": gather_peak,
                              "frac": round(wd["lookups"] / (layer_ms[dom] * 1e-3) / gather_peak, 4)}

    # ---- batch-1: latency and the HBM-bound FC assignment stream (L2 flushed between launches) ----
    extra = {}
    if rank == 0:
        one = dev_in[0][:1].contiguous()
        p1 = torch.empty((1, 1000), dtype=torch.float32, device=dev)
        for w in range(5):
            net.forward(one, prob=p1)
        torch.cuda.synchronize()
        lat = []
        for k in range(30):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            net.forward(one, prob=p1)
            b.record()
            torch.cuda.synchronize()
            lat.append(a.elapsed_time(b))
        extra["latency_b1_eager_ms"] = round(float(np.median(lat)), 4)
        # same call on a non-default stream: after two eager passes the library replays a captured CUDA graph
        side = torch.cuda.Stream(device=dev)
        lat = []
        with torch.cuda.stream(side):
            for w in range(5):
                net.forward(one, prob=p1)
            side.synchronize()
            for k in range(30):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(side)
                net.forward(one, prob=p1)
                b.record(side)
                side.synchronize()
                lat.append(a.elapsed_time(b))
        extra["latency_b1_ms"] = round(float(np.median(lat)), 4)
        # HBM-bound kernel of the path: the batch-1 FC assignment stream (fc6 -> fc7 -> fc8 as ONE persistent launch,
        # csrc/fc_chain.cu), L2 flushed before every launch so the assignment matrices come from HBM.  Two clocks:
        #   event  CUDA events around the single launch (includes ~2 us of launch / event overhead: calibrated below with
        #          an empty-ish launch measured the same way) -- the number the roofline fraction is quoted on;
        #   span   %globaltimer, first CTA's first instruction -> last CTA's last instruction (no launch overhead).
        flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
        fcs = [net.pq_layer(l) for l in (15, 18, 21)]
        xin = torch.rand((1, 9216), dtype=torch.float32, device=dev)
        stamps = torch.zeros(32 * ctx.sm_count, dtype=torch.int64, device=dev)

        def timed(fn, reps=12, use_stamps=True):
            ev, sp = [], []
            for k in range(reps):
                flush.fill_(k & 0xFF)          # evict the 126 MB L2
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                torch.cuda.synchronize()
                if k >= 2:
                    ev.append(a.elapsed_time(b) * 1e3)
                    if use_stamps:
                        st_ = stamps.cpu().numpy().reshape(-1, 32)
                        sp.append((st_[:, 1].max() - st_[:, 0].min()) / 1e3)
            return float(np.median(ev)), (float(np.median(sp)) if sp else None)

        tiny = torch.zeros(32, dtype=torch.float32, device=dev)
        ov_us, _ = timed(lambda: ctx.relu(tiny), use_stamps=False)
        fc_b1 = {"event_overhead_us": round(ov_us, 2),
                 "note": "L2 flushed (256 MB fill) before every launch; us_event = CUDA events around ONE launch, "
                         "us_span = %globaltimer first-CTA-start to last-CTA-end; frac = alg_bytes / us_event / HBM peak"}

        def rec(name, layers_, relu_, x_):
            us_ev, us_sp = timed(lambda: q.fc_chain_forward(layers_, relu_, x_, stamps=stamps))
            byt = float(sum(L_.work(1)["alg_bytes"] for L_ in layers_))
            fc_b1[name] = {"us_event": round(us_ev, 2), "us_span": round(us_sp, 2), "alg_bytes": byt,
                           "achieved_GBps": round(byt / (us_ev * 1e-6) / 1e9, 1),
                           "frac_of_hbm_peak": round(byt / (us_ev * 1e-6) / 1e9 / hbm_peak, 4),
                           "frac_of_hbm_peak_span": round(byt / (us_sp * 1e-6) / 1e9 / hbm_peak, 4)}
        try:
            rec("fc6+fc7+fc8", fcs, [1, 1, 0], xin)
            rec("fc6", fcs[:1], [1], xin)
            rec("fc7", fcs[1:2], [1], torch.rand((1, 4096), dtype=torch.float32, device=dev))
            rec("fc8", fcs[2:], [0], torch.rand((1, 4096), dtype=torch.float32, device=dev))
            # the same kernel on a layer large enough to amortise its fixed latencies (launch, first bytes, one cross-CTA
            # reduction): 8192 subspaces x 4096 outputs, K = 32, d = 4 -> 33.5 MB of assignments + 4.2 MB of codebook
            rs2 = np.random.RandomState(5)
            big = q.FcLayer(ctx, 32768, (rs2.randn(8192, 32, 4) * 0.01).astype(np.float32),
                            rs2.randint(0, 32, size=(4096, 8192)).astype(np.uint8), np.zeros(4096, np.float32))
            rec("synthetic fc 32768 -> 4096 (S=8192, K=32, d=4)", [big], [0], torch.rand((1, 32768), dtype=torch.float32, device=dev))
            big.close()
        except q.QcnnError as e:          # shapes the fused kernel does not take: say so instead of a number
            fc_b1["error"] = str(e)
        extra["fc_b1"] = fc_b1
        del flush

    # ---- BASELINE.json configs[3]: 8192 images over 8 GPUs = 1024 per GPU (weak scaling: 1024 per GPU at every N) ----
    config4 = None
    if not args.no_config4:
        B4 = 1024
        big = torch.cat([dev_in[i & 1] for i in range(B4 // B)], 0) if B4 >= B and B4 % B == 0 else None
        if big is not None:
            prob4 = torch.empty((B4, 1000), dtype=torch.float32, device=dev)
            logits4 = torch.empty((B4, 1000), dtype=torch.float32, device=dev)

            gather4 = sharding.OverlappedGather(B4, 1000, world, dev) if world > 1 else None

            def step4(i):
                if world > 1:
                    net.forward(big, prob=prob4, logits=gather4.rows(i))
                    gather4.launch(i)
                else:
                    net.forward(big, prob=prob4, logits=logits4)
            for w in range(3):
                step4(w)
            barrier()
            k4 = max(3, min(args.steps, 8))
            a4, b4 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a4.record()
            for k in range(k4):
                step4(k)
            b4.record()
            barrier()
            ms4 = torch.tensor([a4.elapsed_time(b4)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(ms4, op=dist.ReduceOp.MAX)
            ms4 = float(ms4.item())
            config4 = {"workload": "BASELINE.json configs[3] per-GPU shard: batch 1024 per GPU, logits all-gather",
                       "global_batch": B4 * world, "per_gpu_batch": B4, "steps": k4, "ms_per_step": ms4 / k4,
                       "value": world * B4 * k4 / (ms4 * 1e-3), "unit": "images/s", "data": "device-resident, CUDA events, max over ranks"}
            del big, prob4, logits4

    # ---- strict path (tensor_core = 0 on every PQ layer: LUT + gather kernels, fp32 adds) at the same batch ----
    strict = None
    if not args.no_strict:
        for l in ALEXNET_PQ:
            net.pq_layer(l).set_param("tensor_core", 0)
        for w in range(3):
            step(w)
        barrier()
        ks = max(3, min(args.steps, 10))
        a5, b5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a5.record()
        for k in range(ks):
            step(k)
        b5.record()
        barrier()
        ms5 = torch.tensor([a5.elapsed_time(b5)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms5, op=dist.ReduceOp.MAX)
        ms5 = float(ms5.item())
        strict = {"value": world * B * ks / (ms5 * 1e-3), "unit": "images/s", "ms_per_step": ms5 / ks, "steps": ks,
                  "path": "tensor_core = 0 (LUT + gather kernels; tolerance 1e-4, DESIGN.md 2)",
                  "plans": {names[l]: net.pq_layer(l).describe(B).split(" grid")[0][:60] for l in (0, 4, 8, 10, 12)}}
        for l in ALEXNET_PQ:
            net.pq_layer(l).set_param("tensor_core", 2)

    # ---- the reference CPU path, single thread, same box, same run (rank 0, N = 1 only) ----
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        kind, med_ms, best_ms = cpu_reference_single_thread(dirpath, pfx, args.cpu_images)
        cpu_baseline = {"value": 1000.0 / med_ms, "unit": "images/s", "cores": 1, "kind": kind,
                        "sample": "%d images, batch 1, one pinned thread (median %.1f ms/img, best %.1f)"
                                  % (args.cpu_images, med_ms, best_ms),
                        "host_cores_available": os.cpu_count()}

    if rank == 0:
        line = {
            "metric": "alexnet_pq_forward_images_per_s", "value": value, "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, what, world),
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": B * IMG_LEN, "d2h_bytes_per_step": B * 5 * 8,
                    "call": "qcnn_net_submit_u8_h / qcnn_net_wait, two steps in flight: uint8 HWC pixels in, on-device mean "
                            "subtraction, forward, on-device top-5 out",
                    "host_buffers": "pinned, " + numa,
                    "synchronous_call": {"value": e2e_sync, "call": "qcnn_net_forward_u8_h (one step at a time, chunk pipeline inside the call)"},
                    "fp32_entry": {"value": e2e_f32, "call": "qcnn_net_forward_h (fp32 NCHW in, [B,1000] probabilities out)",
                                   "h2d_bytes_per_step": B * IMG_LEN * 4, "d2h_bytes_per_step": B * 1000 * 4}},
            "gpu_launches": launches_per_step * args.steps,
            "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline, "per_layer": per_layer,
            "extra": extra, "impl": "b200", "config4": config4, "value_strict": strict,
        }
        print(json.dumps(line))
    net.close()
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=256, help="images per GPU per step")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-images", type=int, default=100, help="cpu_baseline sample size (images)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config4", action="store_true", help="skip the 1024-per-GPU (configs[3]) timing")
    ap.add_argument("--no-strict", action="store_true", help="skip the strict-path (tensor_core = 0) timing")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        return run_reference_arm(args)
    q = importlib.import_module("quantized-cnn_b200")   # raises if libqcnn_b200.so is missing: no fallback
    return run_b200_arm(args, q)


if __name__ == "__main__":
    sys.exit(main())
