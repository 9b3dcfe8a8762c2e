#!/usr/bin/env python
"""bench.py — images/s of the YOLO-Nano-1.0x detection forward path (backbone + FPN/PAN
neck + heads + decode + NMS) on N B200s, batch-sharded, no collective.

    python bench.py --gpus N --steps K --warmup W            # this build (CUDA engine)
    python bench.py --impl reference --gpus N ...             # CPU restatement of the reference
    python bench.py ... --dump-outputs DIR                    # also save the last timed step's detections

A "step" is one pass of the hot path over one batch of synthetic images.  Workload at
every N = the configuration BASELINE.json's metric is quoted on ("416 bs256"): configs[1]'s model
(416x416, COCO-80, fp32 parity mode, incl. decode + NMS) at 256 images per GPU (`--batch 64` is
configs[1]'s own batch; `--size 608 --batch 256` is configs[2]), tcgen05 3xTF32, reference random-init weights (torch.manual_seed), conf 0.001 / nms 0.5
— with this init EVERY anchor passes the threshold, i.e. worst-case NMS (BASELINE.md §3).
`value` times the device path with inputs resident in HBM; `e2e` times the C-ABI host call on the reference's
real input — uint8 images, data/transforms.py:445-458 — from pinned host memory (H2D + D2H inside the timed
region); `e2e_f32` is the same through the float32 [B,3,S,S] entry.  `parity` checks two images of the timed batch
against the CPU oracle in the same run.  `--strong` splits `--batch` over the ranks (BASELINE configs[2]).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True      # the tree may be read-only; the benchmark writes nothing into it

import numpy as np  # noqa: E402
import torch  # noqa: E402

SIZE, BATCH, CLASSES = 416, 256, 80


def metric_name(a):
    bs = getattr(a, "total_batch", a.batch)
    tag = "bf16" if getattr(a, "mode", "") == "bf16" else "fp32-parity"
    return (f"images/sec YOLO-Nano-1.0x {a.size} bs{bs} {tag} e2e (backbone+neck+head+decode+NMS)")
CONF, NMS_T = 0.001, 0.5


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default: 100 for detect, 30 for train)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--size", type=int, default=SIZE)
    ap.add_argument("--mode", default="3xtf32", choices=["ffma", "3xtf32", "tf32", "bf16"],
                    help="3xtf32 = the fp32 parity mode (default, the headline); bf16 = BASELINE configs[3] throughput mode")
    ap.add_argument("--weights", default="refinit", choices=["refinit", "calibrated"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-profile", default="")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the detections of the last timed step as DIR/<name>.npy (rank 0; see dump_outputs)")
    ap.add_argument("--strong", action="store_true",
                    help="strong scaling: --batch is the TOTAL batch, split evenly over the ranks (configs[2])")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run oracle check of two images")
    ap.add_argument("--no-latency", action="store_true", help="skip the batch-1 drop-in latency measurement")
    ap.add_argument("--workload", default="detect", choices=["detect", "train"],
                    help="train = BASELINE configs[4]: the data-parallel training step (tools/gpu_train_step_bench.py), "
                         "32 images per GPU unless --batch is given")
    a = ap.parse_args()
    if a.steps is None:
        a.steps = 30 if a.workload == "train" else 100
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.workload != "detect" or a.impl != "b200"):
        ap.error("--dump-outputs records the detect workload of --impl b200 only")
    return a


# --------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.samples.append([v.strip() for v in out.strip().split(",")])
            except Exception:  # noqa: BLE001
                pass
            self.stop_flag.wait(0.05)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if len(s) >= 7 and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) >= 7 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples if len(s) >= 7 for n, v in zip(names, s[3:7]) if v == "Active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples)}


def cpu_baseline(sd, seconds: float, size: int):
    """The oracle port of the reference (torch CPU network + NumPy NMS, batch 1 loop — the
    only batch the reference supports) timed on this host's cores on a bounded sample."""
    from oracle import weights as W
    from oracle import yolo_nano_oracle as O
    cores = len(os.sched_getaffinity(0))
    torch.set_num_threads(cores)
    anchors = W.anchors_for(CLASSES)
    x = W.synthetic_input(4, size, seed=11)
    for i in range(2):
        O.detect(sd, x[i:i + 1], size, CLASSES, anchors, CONF, NMS_T, tie="numpy")
    n, t0 = 0, time.perf_counter()
    net_t = 0.0
    while True:
        xi = x[n % 4:n % 4 + 1]
        t1 = time.perf_counter()
        preds = O.network(sd, xi)
        bb, cl = O.decode(preds, size, CLASSES, anchors)
        net_t += time.perf_counter() - t1
        O.postprocess(bb[0].numpy(), cl[0].numpy(), CLASSES, CONF, NMS_T, False, "numpy")
        n += 1
        el = time.perf_counter() - t0
        if (el >= seconds and n >= 3) or n >= 200:
            break
    return {"value": n / el, "unit": "images/s", "cores": cores, "kind": "port",
            "sample": f"{n} images of the bench workload, batch 1 loop, torch {torch.__version__} CPU + NumPy NMS "
                      f"(oracle/yolo_nano_oracle.py), {el:.1f} s",
            "network_ms_per_image": 1e3 * net_t / n, "nms_ms_per_image": 1e3 * (el - net_t) / n}


def traffic_file(a) -> Path:
    """The committed ncu DRAM-traffic capture of this command at this workload (416^2, 256 images only), reduced to
    bytes per launch and kernel family by tools/ncu_traffic_by_kind.py (launches matched to the plan's ops in order)."""
    name = "r02_dram_traffic_by_kind_b256.json" if (a.size == 416 and a.batch == 256 and a.mode == "3xtf32") else "none"
    return ROOT / "profiles" / name


def load_traffic_by_kind(kind: str, p: Path):
    if not p.exists():
        return None
    d = json.loads(p.read_text()).get("per_kind", {}).get(kind)
    return None if d is None else d["dram_bytes_per_launch"]


def parity_check(eng, sd, x_host, x_dev, size, mode="3xtf32"):
    """Two images of the TIMED batch through the CPU oracle (the checker, never the path) in this same run:
    raw head maps in units of the north_star tolerance (1e-3 + 1e-4 |ref|), decoded boxes in pixels, and the
    keep-sets — exact against the oracle's NMS on the engine's own candidates, and against the oracle end to end
    with the differing boxes counted (on reference-init weights they are exact score ties / 1-ulp order flips)."""
    from oracle import weights as W
    from oracle import yolo_nano_oracle as O
    anchors = W.anchors_for(CLASSES)
    ref_raw = O.network(sd, x_host)
    raw = eng.forward_raw(x_dev)
    worst, over, n, worst_abs = 0.0, 0, 0, 0.0
    for got, want in zip(raw, ref_raw):
        err = np.abs(got.cpu().numpy() - want.numpy())
        worst_abs = max(worst_abs, float(err.max()))
        tol = 1e-3 + 1e-4 * np.abs(want.numpy())
        worst = max(worst, float((err / tol).max())); over += int((err > tol).sum()); n += err.size
    bb, cl = O.decode(ref_raw, size, CLASSES, anchors)
    boxes, scores, cls = eng.forward_decode(x_dev)
    ob, os_, oc, on = eng.forward_detect(x_dev)
    res = {"images": int(x_host.shape[0]), "raw_worst_err_in_tol": round(worst, 4), "raw_over_tol": over, "raw_outputs": n,
           "box_err_px": 0.0, "kept": [], "oracle_kept": [], "keepset_exact_on_own_candidates": True,
           "keepset_differ_vs_oracle": 0}
    for i in range(x_host.shape[0]):
        bh, sh, ch = boxes[i].cpu().numpy(), scores[i].cpu().numpy(), cls[i].cpu().numpy().astype(np.int64)
        res["box_err_px"] = max(res["box_err_px"], float(np.abs(bh - bb[i].numpy()).max()) * size)
        _, _, _, idx = O.postprocess_flat(bh, sh, ch, CLASSES, CONF, NMS_T)
        k = int(on[i])
        same = k == len(idx) and np.array_equal(ob[i, :k].cpu().numpy(), bh[idx]) and \
            np.array_equal(oc[i, :k].cpu().numpy().astype(np.int64), ch[idx])
        res["keepset_exact_on_own_candidates"] = bool(res["keepset_exact_on_own_candidates"] and same)
        _, _, _, ridx = O.postprocess(bb[i].numpy(), cl[i].numpy(), CLASSES, CONF, NMS_T)
        res["kept"].append(k); res["oracle_kept"].append(int(len(ridx)))
        res["keepset_differ_vs_oracle"] += int(len(np.setxor1d(idx, ridx)))
    res["box_err_px"] = round(res["box_err_px"], 6)
    res["raw_worst_abs_err"] = round(worst_abs, 6)
    if mode == "bf16":      # throughput mode: its own stated tolerance (tests/test_gpu_forward.py::test_bf16_mode_*)
        res["tolerance"] = "bf16 mode: raw head maps within 2e-2 absolute on reference-init weights; NMS exact on its inputs"
        res["ok"] = bool(worst_abs < 2e-2 and res["keepset_exact_on_own_candidates"])
    else:
        res["tolerance"] = "north_star: raw 1e-3 + 1e-4 |ref|, boxes 1e-3 px, keep-sets exact up to score ties (counted)"
        res["ok"] = bool(over == 0 and res["keepset_exact_on_own_candidates"] and res["box_err_px"] < 1e-3
                         and res["keepset_differ_vs_oracle"] <= 0.05 * sum(res["oracle_kept"]))
    return res


def latency_b1(sd, dev, size, mode):
    """The reference's own timing method (benchmark.py:40-82): batch 1 through the drop-in class, one image at a
    time, device input, host ndarray results (the call syncs like the reference's .to('cpu')), ms per image."""
    import contextlib
    import io
    import yolo_nano_b200 as pkg
    from oracle import weights as W
    out = {}
    for s in sorted({320, size}):
        with contextlib.redirect_stdout(io.StringIO()):
            m = pkg.YOLONano(dev, input_size=s, num_classes=CLASSES, conf_thresh=CONF, nms_thresh=NMS_T,
                             anchor_size=W.anchors_for(CLASSES), gemm_mode=mode)
        m.load_state_dict(sd)
        m = m.to(dev).eval()
        xs = [W.synthetic_input(1, s, seed=20 + i).to(dev) for i in range(4)]
        for i in range(8):
            m(xs[i % 4])
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        n = 50
        for i in range(n):
            m(xs[i % 4])
        out[str(s)] = round(1e3 * (time.perf_counter() - t0) / n, 4)
        del m
    return {"unit": "ms/image", "batch": 1, "call": "YOLONano.forward(x) -> (bboxes, scores, cls_inds) host ndarrays",
            "by_input_size": out}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, out_dev):
    """Writes what forward_detect handed back in the last timed step, so that two builds can be compared on the
    same seeded inputs: `counts` [B] (detections kept per image), and for a fixed sample of the images
    (`images`, ascending) their valid rows one after another: `boxes` [M,4], `scores` [M], `cls` [M].  Rows past
    an image's count are not part of the result and are left out.  The sample is every image if the worst case
    (all N candidates kept) fits DUMP_BYTES, else a seeded choice of as many images as fit; it depends only on
    the batch and the input size.  All arrays float32 (class ids and counts are exact)."""
    boxes, scores, cls, counts = (t.cpu().numpy() for t in out_dev)
    batch, n = scores.shape
    fit = max(1, (DUMP_BYTES - 8 * batch) // (n * 6 * 4))
    images = np.arange(batch) if fit >= batch else np.sort(np.random.default_rng(0).choice(batch, fit, replace=False))
    rows = [np.arange(int(counts[i])) for i in images]
    arrays = {"counts": counts, "images": images,
              "boxes": np.concatenate([boxes[i, r] for i, r in zip(images, rows)]),
              "scores": np.concatenate([scores[i, r] for i, r in zip(images, rows)]),
              "cls": np.concatenate([cls[i, r] for i, r in zip(images, rows)])}
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), v.astype(np.float32))


def bind_to_gpu_numa_node(index: int):
    """Restrict this rank to the CPU cores NVML reports as local to its GPU (before any pinned host
    buffer is allocated: first touch places the pages on that NUMA node).  With 8 ranks pushing
    133 MB per step each, cross-socket input copies halve the host-side bandwidth.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {w * 64 + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus and len(cpus) < len(os.sched_getaffinity(0)):
            os.sched_setaffinity(0, cpus)
            return sorted(cpus)[0], len(cpus)
    except Exception:
        pass
    return None


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------------------------
def run_reference(a, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (oracle port;
    the Python reference cannot travel to the GPU box), all host threads, rank 0 only."""
    if rank != 0:
        return
    from oracle import weights as W
    from oracle import yolo_nano_oracle as O
    cores = len(os.sched_getaffinity(0))
    torch.set_num_threads(cores)
    sd = W.reference_init(CLASSES, seed=3) if a.weights == "refinit" else W.calibrated(CLASSES, seed=2)
    anchors = W.anchors_for(CLASSES)
    per_step = 2                      # bounded sample of the batch
    x = W.synthetic_input(per_step, a.size, seed=11)
    def step():
        O.detect(sd, x, a.size, CLASSES, anchors, CONF, NMS_T, tie="numpy")
    for _ in range(a.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        step()
    dt = time.perf_counter() - t0
    v = a.steps * per_step / dt
    line = {"impl": "reference", "metric": metric_name(a), "value": v, "unit": "images/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(a),
            "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": "port",
                             "sample": f"{per_step} images per step (of the {a.batch}-image batch), batch-1 loop as the "
                                       "reference runs it"},
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(a):
    return {"workload": f"BASELINE metric config (configs[1] at the metric's batch): YOLO-Nano-1.0x inference "
                        f"{a.size}x{a.size}, batch {a.batch} per GPU, COCO {CLASSES} classes, fp32 parity mode, "
                        "incl. decode+NMS",
            "input_size": a.size, "batch_per_gpu": a.batch, "total_batch_if_strong": getattr(a, "total_batch", a.batch)
            if getattr(a, "strong", False) else None, "num_classes": CLASSES, "conf_thresh": CONF,
            "nms_thresh": NMS_T, "weights": "reference random init (torch.manual_seed(3))" if a.weights == "refinit"
            else "calibrated synthetic (oracle/weights.py seed 2)",
            "gemm_mode": a.mode, "sharding": "batch-sharded, one process per GPU, no collective" +
            (" (strong scaling: the total batch is split over the ranks)" if getattr(a, "strong", False) else ""),
            "l2": f"inputs {a.batch * 3 * a.size * a.size * 4 / 1e6:.0f} MB per step (> 126 MB L2), "
                  f"4 rotating input batches; intermediate activations ~{a.batch * 24 * (a.size / 416) ** 2 / 1e3:.1f} GB per step"}


def run_train_workload(a):
    """BASELINE configs[4] through the same launch contract: hands over to tools/gpu_train_step_bench.py."""
    sys.path.insert(0, str(Path(__file__).resolve().parent / "tools"))
    import gpu_train_step_bench as tb
    argv = ["--steps", str(a.steps), "--warmup", str(max(a.warmup, 3)), "--size", str(a.size),
            "--batch", str(32 if a.batch == BATCH else a.batch)]
    if not a.no_cpu_baseline:
        argv.append("--cpu-baseline")
    sys.argv = [sys.argv[0]] + argv
    tb.main()


def main():
    a = parse()
    if a.workload == "train":
        if a.impl == "reference":
            raise SystemExit("--workload train has no --impl reference arm (its CPU baseline is in the line itself)")
        run_train_workload(a)
        return
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    a.total_batch = a.batch
    if a.strong:
        if a.batch % max(world, a.gpus):
            raise SystemExit(f"--strong: batch {a.batch} is not divisible by {max(world, a.gpus)} ranks")
        a.batch //= max(world, a.gpus)
    if a.impl == "reference":
        run_reference(a, rank, world)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    import torch.distributed as dist
    from oracle import weights as W                    # weights / inputs generators + CPU baseline only
    from oracle import yolo_nano_oracle as O
    from yolo_nano_b200 import _lib
    from yolo_nano_b200.engine import Engine
    from yolo_nano_b200.topology import conv_table

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)      # pinned host buffers are then allocated next to the GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    modes = {"ffma": _lib.GEMM_FP32_FFMA, "3xtf32": _lib.GEMM_TC_3XTF32, "tf32": _lib.GEMM_TC_TF32,
             "bf16": _lib.GEMM_TC_BF16}

    sd = W.reference_init(CLASSES, seed=3) if a.weights == "refinit" else W.calibrated(CLASSES, seed=2)
    eng = Engine(dev, a.size, CLASSES, W.anchors_for(CLASSES), CONF, NMS_T, False, modes[a.mode], a.batch)
    eng.load_weights(O.fold_state_dict(sd, conv_table(CLASSES)))

    nbuf = 4
    g = torch.Generator().manual_seed(100 + rank)
    host_x = [torch.randn(a.batch, 3, a.size, a.size, generator=g).pin_memory() for _ in range(nbuf)]
    dev_x = [h.to(dev) for h in host_x]
    out_dev = eng.alloc_outputs(a.batch)
    out_host = eng.alloc_outputs(a.batch, pinned_host=True)
    stream = torch.cuda.current_stream(dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        for i in range(steps):
            fn(i)
        e1.record(stream)
        torch.cuda.synchronize(dev)
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms, wall * 1e3], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        barrier()
        return float(t[0]), float(t[1])

    # ---- device-resident throughput (value) ------------------------------------------------
    def step_dev(i):
        eng.forward_detect(dev_x[i % nbuf], out_dev)

    for i in range(max(a.warmup, 3)):
        step_dev(i)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = eng.launch_count
    ms_dev, _ = timed(step_dev, a.steps)
    launches = eng.launch_count - l0
    counts = out_dev[3].cpu().numpy()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, out_dev)

    # ---- end to end through the host-buffer C-ABI call (e2e) ---------------------------------
    # streaming use of the host API: step i is submitted (H2D on the copy stream, compute behind
    # it) before step i-1 is collected, so PCIe and compute overlap; every step's H2D and D2H
    # still happen inside the timed region.
    out_host2 = [out_host, eng.alloc_outputs(a.batch, pinned_host=True)]

    def run_host(steps):
        for i in range(steps):
            eng.submit_host(i & 1, host_x[i % nbuf], out_host2[i & 1])
            if i > 0:
                eng.wait_host((i - 1) & 1)
        eng.wait_host((steps - 1) & 1)

    run_host(3)
    barrier()
    t0 = time.perf_counter()
    run_host(a.steps)
    torch.cuda.synchronize(dev)
    wall = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([wall], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    barrier()
    wall_e2e = float(t[0])
    if sampler:
        sampler.stop_flag.set()
        sampler.join(timeout=3)

    # ---- the same loop through the uint8 entry (SURVEY 8f row 1: Normalize + ToTensor on the device;
    # images cross PCIe as bytes).  Extra information next to `e2e`, which stays the float32 boundary.
    gu = torch.Generator().manual_seed(11 + rank)
    host_u8 = [torch.randint(0, 256, (a.batch, a.size, a.size, 3), dtype=torch.uint8, generator=gu).pin_memory()
               for _ in range(nbuf)]

    def run_host_u8(steps):
        for i in range(steps):
            eng.submit_host_u8(i & 1, host_u8[i % nbuf], out_host2[i & 1])
            if i > 0:
                eng.wait_host((i - 1) & 1)
        eng.wait_host((steps - 1) & 1)

    run_host_u8(3)
    barrier()
    t0 = time.perf_counter()
    run_host_u8(a.steps)
    torch.cuda.synchronize(dev)
    wall = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([wall], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    barrier()
    wall_u8 = float(t[0])
    run_host(2)      # leave the float32 results in the output buffers read below
    kept = int(out_host2[(a.steps - 1) & 1][3].sum())
    h2d = a.batch * 3 * a.size * a.size * 4
    kmax = int(out_host2[(a.steps - 1) & 1][3].max())
    d2h = a.batch * 4 + a.batch * kmax * 24      # rows [0, max count) of every image (strided copies)

    # ---- per-kernel roofline (CUDA events around every launch, same process) ----------------
    prof = {}
    rows = []
    for rep in range(3):
        rows = eng.profile(dev_x[rep % nbuf])
        for name, kind, ms, by, fl in rows:
            d = prof.setdefault(kind, {"ms": 0.0, "bytes": 0.0, "flops": 0.0, "launches": 0})
            d["ms"] += ms / 3; d["bytes"] += by / 3; d["flops"] += fl / 3; d["launches"] += 1 / 3
    if a.dump_profile and rank == 0:
        with open(a.dump_profile, "w") as f:
            json.dump({"per_launch_last_rep": rows, "per_kind_avg": prof}, f, indent=1)
    peak, peak_src = load_peaks()
    total_prof_ms = sum(d["ms"] for d in prof.values())
    dom = max(prof.items(), key=lambda kv: kv[1]["ms"])
    dk, dd = dom
    ach = dd["bytes"] / (dd["ms"] * 1e-3) / 1e9
    sass_name = {"pw_tcgen05": "tc_gemm_kernel", "conv3x3_tcgen05": "tc_gemm_kernel", "nms": "nms_segment_kernel",
                 "dwpw_tcgen05": "dwpw_tc_kernel",
                 "dwconv3x3": "dwconv3x3_kernel", "stem_pool": "stem_pool_kernel", "decode": "decode_level_kernel"}.get(dk, dk)
    roofline = {"bound": "hbm", "kernel": dk, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": load_traffic_by_kind(dk, traffic_file(a)),
                "traffic_note": "avg DRAM read+write bytes per launch of the `" + dk + "` launches (" + sass_name +
                f"; ncu, profiles/{traffic_file(a).name}); algorithmic bytes per launch = " +
                f"{dd['bytes'] / max(dd['launches'], 1e-9):.3e}", "peak_source": peak_src,
                "launches_per_step": dd["launches"], "ms_per_step": dd["ms"],
                "share_of_step": dd["ms"] / total_prof_ms,
                "achieved_tflops": dd["flops"] / (dd["ms"] * 1e-3) / 1e12,
                "whole_step": {"algorithmic_gb": sum(d["bytes"] for d in prof.values()) / 1e9,
                               "achieved_gbs": sum(d["bytes"] for d in prof.values()) / (ms_dev / a.steps * 1e-3) / 1e9},
                "by_kernel": {k: {"ms": round(v["ms"], 4), "gbs": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1),
                                  "tflops": round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 2),
                                  "launches": round(v["launches"])} for k, v in sorted(prof.items())}}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    cpu = None
    if not a.no_cpu_baseline and a.gpus == 1:
        cpu = cpu_baseline(sd, a.cpu_seconds, a.size)
    parity = None if a.no_parity else parity_check(eng, sd, host_x[0][:2], dev_x[0][:2].contiguous(), a.size, a.mode)
    latency = None if (a.no_latency or world > 1) else latency_b1(sd, dev, a.size, modes[a.mode])

    imgs = world * a.batch * a.steps
    line = {"metric": metric_name(a), "value": imgs / (ms_dev * 1e-3), "unit": "images/s", "n_gpus": world, "steps": a.steps,
            "warmup": max(a.warmup, 3), "ms_per_step": ms_dev / a.steps, "higher_is_better": True,
            "scaling": "strong" if a.strong else "weak",
            "vs_baseline": None, "dtype": {"3xtf32": "f32 (tcgen05 3xTF32 split, fp32 accumulate)", "ffma": "f32", "tf32": "tf32",
                      "bf16": "bf16 storage + tcgen05 kind::f16, fp32 accumulate (throughput mode, tolerance in "
                              "tests/test_gpu_forward.py::test_bf16_mode_*)"}[a.mode],
            "data": "synthetic", "config": workload_config(a),
            # the reference's real input is a uint8 image (data/transforms.py:445-458): that entry is the declared
            # end-to-end number; the float32 [B,3,S,S] entry (4x the bytes over PCIe) is kept beside it
            "e2e": {"value": imgs / (wall_u8 * 1e-3), "unit": "images/s",
                    "h2d_bytes_per_step": a.batch * 3 * a.size * a.size, "d2h_bytes_per_step": d2h,
                    "ms_per_step": wall_u8 / a.steps,
                    "call": "ynb_submit_host_u8 / ynb_wait_host, 2 slots: pinned uint8 HWC BGR images in, Normalize + "
                            "ToTensor of data/transforms.py on the device (bit-identical tensor), pinned host detections "
                            "out; step i's PCIe copy overlaps step i-1's compute"},
            "e2e_f32": {"value": imgs / (wall_e2e * 1e-3), "unit": "images/s", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": d2h, "ms_per_step": wall_e2e / a.steps,
                        "call": "ynb_submit_host / ynb_wait_host: the same with float32 [B,3,S,S] host input"},
            "parity": parity, "latency_b1": latency,
            "host_affinity": None if numa is None else {"first_cpu": numa[0], "cpus": numa[1]},
            "gpu_launches": launches, "clocks": sampler.summary() if sampler else None,
            "roofline": roofline, "cpu_baseline": cpu,
            "detections_per_image": float(counts.mean())}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
