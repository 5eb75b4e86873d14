#!/usr/bin/env python
"""bench.py -- ROIs/s of the GDRNPP per-ROI pose path (BASELINE.json metric) on N B200s of one node.

  python bench.py --gpus 1 --steps 20 --warmup 5
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
         bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...      (the CPU path on the host cores; oracle port, see DESIGN.md)
  python bench.py --workload fps|voting|nnd|flow|raster|upnp|refine|ycbv5|native   (one JSON line per record)

A step = one forward of the whole hot path (ConvNeXt-base + geometry head + Patch-PnP + pose lift) over one batch of 64
synthetic 256x256 ROIs per GPU (BASELINE.json configs[1]); ROIs are sharded across ranks with no data-path collective
except ONE all-gather of the [n,12] poses at the end of the timed region (configs[3]).

The number of record is measured in the PARITY precision mode ("bf16x3": split-bf16 tensor-core GEMMs, R within 1e-4 rad /
t within 1e-3 of the fp32 reference path, tests/test_gpu_parity.py::test_forward_vs_oracle_b64): CUDA-graph replay,
device-resident `value`, `e2e` with host buffers, `roofline`, `cpu_baseline`.  The bf16 throughput mode (R within ~0.03 rad)
is a SECONDARY record (`bf16_mode`).  Prints exactly one JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GFLOP_PER_ROI_REFERENCE = 56.45          # BASELINE.md §2: 28.225 GMAC, as the reference computes it
GFLOP_PER_ROI_EXECUTED = 53.51           # out conv computed for the ROI's own class only (70 of 1470 channels)
GEMM_GFLOP_PER_ROI_EXECUTED = 2 * (26.757 - 0.2986)  # executed work minus the depthwise convs (CUDA-core kernel)
BATCH = 64
CPU_SAMPLE_ROIS = 8                      # ROIs per step of the CPU arms (reference arm and cpu_baseline use the SAME sample)
METRIC = "ROIs/sec (256x256, ConvNeXt-base 'a6' + geo heads + Patch-PnP)"


def workload_config(world, precision):
    return {"workload": "batch=64 synthetic ROIs per GPU, ConvNeXt-a6 (convnext_base) + geometry heads + Patch-PnP + pose "
                        "lift (BASELINE configs[1]); ROIs sharded across ranks, one NCCL all-gather of [n,12] poses at "
                        "the end (configs[3])",
            "global_batch": BATCH * world,
            "l2": "inputs rotate over 4 distinct batches; per-step working set (~2 GB activations + 0.4 GB weights in "
                  "bf16x3) >> 126 MB L2",
            "parallelism": "roi-shard x%d" % world, "precision": precision}


def load_peaks(timed_region_s=None):
    """bf16 roofline denominator: the BURST figure for a timed region under ~1 s (the GPU has not hit its power-capped
    steady state yet), the sustained one for seconds-long regions (B200_PROFILING.md)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        burst = timed_region_s is None or timed_region_s < 1.0
        tf = d.get("bf16_tflops") if burst else d.get("bf16_tflops_sustained", d.get("bf16_tflops"))
        return {"bf16_tflops": tf, "hbm_gbs": d.get("hbm_gbs"), "sm_max_mhz": d.get("sm_max_mhz"),
                "source": "measured (MEASURED_PEAKS.json, %s; timed region %.2f s)" % ("burst" if burst else "sustained", timed_region_s or 0.0)}
    return {"bf16_tflops": 1590.0, "hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    """CPU threads this process may actually use (cgroup / affinity aware), capped at 64 for the torch CPU path."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(n, 64))


def bench_reference(args, rank, world):
    """--impl reference: the reference algorithm on the host cores (oracle port; the reference's own Python cannot be
    imported: timm/mmcv/detectron2 are absent, DESIGN.md §oracle).  Each step = a bounded sample of CPU_SAMPLE_ROIS ROIs
    of the 64-ROI batch."""
    if rank != 0:
        return
    from gdrnpp_bop2022_b200.synthetic import make_batch, make_state_dict
    from oracle import gdrn_model_oracle as O

    threads = host_threads()
    torch.set_num_threads(threads)
    n = CPU_SAMPLE_ROIS
    sd = make_state_dict()
    batches = [{k: v[:n] for k, v in make_batch(B=BATCH, seed=i).items()} for i in range(2)]   # the bench's own batches
    with torch.no_grad():
        for i in range(max(1, min(args.warmup, 3))):
            O.gdrn_forward(sd, batches[i % 2])
        t0 = time.perf_counter()
        for i in range(args.steps):
            O.gdrn_forward(sd, batches[i % 2])
        dt = time.perf_counter() - t0
    val = n * args.steps / dt
    sample = "%d ROIs of the 64-ROI batch per step x %d steps, torch CPU fp32, %d threads" % (n, args.steps, threads)
    out = {
        "impl": "reference", "metric": METRIC,
        "value": val, "unit": "ROIs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(max(world, 1), "f32 (reference arithmetic)"),
        "cpu_baseline": {"value": val, "unit": "ROIs/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "ROIs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def gpu_eager_baseline(dev):
    """BASELINE.md §3 R-GPU-5 / R-GPU-64 stand-in: the reference forward as eager fp32 PyTorch on this GPU (cuDNN convs,
    cuBLAS linears, native LN/GN/GELU -- the same torch ops the reference module makes; the reference module itself
    needs timm/mmcv/detectron2, absent), timed like engine/gdrn_evaluator.py:707-751 (perf_counter + cuda.synchronize,
    5 warm-up).  Backbone = torchvision.models.convnext_base().features (pinned bit-exact to the oracle by
    tests/test_oracle_pinning.py) when torchvision is importable.  A REPORTED BASELINE, not the product path."""
    from gdrnpp_bop2022_b200.synthetic import make_batch, make_state_dict
    from oracle import gdrn_model_oracle as O

    sd = {k: v.to(dev) for k, v in make_state_dict().items()}
    backbone = None
    try:
        backbone = O.torchvision_convnext(sd, "convnext_base").to(dev).eval()
    except Exception:  # noqa: BLE001
        backbone = None
    res = {"backbone": "torchvision.models.convnext_base().features" if backbone is not None else "oracle functional restatement",
           "timing": "perf_counter + cuda.synchronize, 5 warm-up, 10 timed batches (gdrn_evaluator.py:707-751 recipe)",
           "kind": "stand-in for the reference's own CUDA build (same torch/cuDNN/cuBLAS ops, eager)"}
    prev = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    for tf32 in (False, True):
        torch.backends.cudnn.allow_tf32 = tf32          # torch default: TF32 allowed for cuDNN convs, not for matmuls
        torch.backends.cuda.matmul.allow_tf32 = False
        for B in (5, 64):
            batch = {k: v.to(dev) for k, v in make_batch(B=B, seed=1).items()}
            cls_cpu = batch["roi_classes"].cpu()

            def fwd():
                feat = backbone(batch["roi_img"]) if backbone is not None else O.convnext_features(sd, batch["roi_img"])
                vis, full, cx, cy, cz, region = O.geo_head(sd, feat)
                vis, full, cx, cy, cz, region = O.class_gather(vis, full, cx, cy, cz, region, cls_cpu)
                coor = torch.cat([cx, cy, cz, batch["roi_coord_2d"]], dim=1)
                rs = torch.softmax(region[:, 1:], dim=1)
                rot6, t_ = O.conv_pnp_net(sd, coor, rs, batch["roi_extents"])
                return O.rot6d_to_mat_batch(rot6), t_

            with torch.no_grad():
                for _ in range(5):
                    fwd()
                torch.cuda.synchronize()
                n = 10
                t0 = time.perf_counter()
                for _ in range(n):
                    fwd()
                torch.cuda.synchronize()
                dt = (time.perf_counter() - t0) / n
            res["fp32%s_bs%d" % ("_tf32conv" if tf32 else "", B)] = {"ms_per_batch": dt * 1e3, "rois_per_s": B / dt}
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    return res


def dump_outputs(path, arrays):
    """--dump-outputs: what the timed path handed its caller in the last timed step, one float32 DIR/<name>.npy each.
    The inputs and weights are seeded, so two builds run with the same arguments can be compared output for output."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30, help="number of timed steps")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the bf16_mode / gpu_eager_baseline / native_ops records")
    ap.add_argument("--precision", default="bf16x3", choices=["bf16x3", "bf16"],
                    help="bf16x3 (default, the mode of record): split-bf16 GEMMs, fp32 parity; bf16: throughput mode")
    ap.add_argument("--workload", default="pose64",
                    help="pose64 (default) | native | fps | voting | nnd | flow | raster | upnp | refine | ycbv5")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the poses of the last one as DIR/rot.npy [N,3,3] and DIR/trans.npy [N,3] "
                         "(float32; N = 64 x GPUs, in rank order); pose64 workload, --impl ours")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "pose64"):
        ap.error("--dump-outputs writes the outputs of the pose64 workload of --impl ours")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        bench_reference(args, rank, world)
        return

    import torch.distributed as dist

    from gdrnpp_bop2022_b200 import _lib
    from gdrnpp_bop2022_b200.dist import all_gather_poses
    from gdrnpp_bop2022_b200.gdrn_model import GDRN_DoubleMask, default_cfg
    from gdrnpp_bop2022_b200.synthetic import make_batch, make_state_dict

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    if args.workload != "pose64":     # native-op micro-benchmarks / configs[2] / configs[4]: one JSON line per record
        if rank != 0:
            return
        import bench_native

        which = None if args.workload == "native" else [args.workload]
        for rec in bench_native.run(dev, load_peaks(), which, args.precision):
            print(json.dumps(rec), flush=True)
        return

    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()

    model = GDRN_DoubleMask(default_cfg(), max_batch=BATCH, precision=args.precision)
    model.load_state_dict(make_state_dict())
    model.to(dev)
    NB = 4  # distinct input batches: 4 x 50 MB of images + ~2 GB of activations per step >> 126 MB L2
    keys = ("roi_img", "roi_classes", "roi_coord_2d", "roi_cams", "roi_centers", "roi_whs", "resize_ratios",
            "roi_extents")
    host = []
    for i in range(NB):
        b = make_batch(B=BATCH, seed=rank * 100 + i)
        host.append({k: b[k].pin_memory() for k in keys})
    resident = [{k: v.to(dev) for k, v in hb.items()} for hb in host]
    staging = {k: torch.empty_like(v, device=dev) for k, v in host[0].items()}
    rot_host = torch.empty((BATCH, 3, 3), dtype=torch.float32).pin_memory()
    trans_host = torch.empty((BATCH, 3), dtype=torch.float32).pin_memory()
    h2d_bytes = sum(v.numel() * v.element_size() for v in host[0].values())
    d2h_bytes = rot_host.numel() * 4 + trans_host.numel() * 4

    def fwd_m(m, b):
        return m(b["roi_img"], roi_classes=b["roi_classes"], roi_coord_2d=b["roi_coord_2d"], roi_cams=b["roi_cams"],
                 roi_centers=b["roi_centers"], roi_whs=b["roi_whs"], roi_extents=b["roi_extents"],
                 resize_ratios=b["resize_ratios"])

    def fwd(b):
        return fwd_m(model, b)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    for i in range(args.warmup):
        fwd(resident[i % NB])
    torch.cuda.synchronize()
    # one CUDA graph per static input buffer: a step = one graph launch (~150 kernels)
    use_graphs = os.environ.get("GDRN_BENCH_GRAPHS", "1") != "0"

    def make_graphed(m):
        graphs = {}

        def graphed(b):
            if not use_graphs:
                return fwd_m(m, b)
            key = b["roi_img"].data_ptr()
            if key not in graphs:
                graphs[key] = m.capture_graph({k: b[k] for k in keys})
            replay, out = graphs[key]
            replay()
            return out

        return graphed

    graphed = make_graphed(model)
    for i in range(NB):
        graphed(resident[i])
    torch.cuda.synchronize()

    # ---------------- device-resident timing (value) ----------------
    # nvidia-smi needs ~0.3 s to deliver its first sample: start it while the (untimed) load is already running
    # so that every sample is taken under the same load as the timed region.
    sampler = ClockSampler(local_rank)
    sampler.start()
    t_spin = time.perf_counter()
    while len(sampler.lines) < 2 and time.perf_counter() - t_spin < 3.0:
        graphed(resident[0])
        torch.cuda.synchronize()
    launches0 = L.gdrn_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    rots, transes = [], []
    for i in range(args.steps):
        o = graphed(resident[i % NB])
        rots.append(o["rot"].clone() if use_graphs else o["rot"])
        transes.append(o["trans"].clone() if use_graphs else o["trans"])
    if world > 1:
        gathered = all_gather_poses(torch.cat(rots), torch.cat(transes))
    e1.record()
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        if world > 1:   # every rank's poses of every step, in rank order: keep each rank's last step
            last = [x.view(world, args.steps, BATCH, *x.shape[1:])[:, -1].reshape(world * BATCH, *x.shape[1:]) for x in gathered]
        else:
            last = [rots[-1], transes[-1]]
        dump_outputs(args.dump_outputs, {"rot": last[0], "trans": last[1]})
    launches = L.gdrn_launch_count() - launches0
    if use_graphs:  # graph replays do not pass through the launch counter: count the kernels of one captured forward
        c0_ = L.gdrn_launch_count()
        fwd(resident[0])
        launches = (L.gdrn_launch_count() - c0_) * args.steps
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    value = world * BATCH * args.steps / (ms_total / 1e3)

    # ---------------- end-to-end through the public API with host buffers ----------------
    # Every step: H2D of that step's inputs from pinned host memory, forward, D2H of that step's poses.
    # Double-buffered: the copy stream uploads step i+1 while the compute stream runs step i; the host reads
    # the poses of step i-1 (already on the host) while step i executes -- the serving loop a user would write.
    copy_stream = torch.cuda.Stream(device=dev)
    comp_stream = torch.cuda.current_stream()
    stagings = [staging, {k: torch.empty_like(v) for k, v in staging.items()}]
    rot_hosts = [rot_host, torch.empty_like(rot_host).pin_memory()]
    trans_hosts = [trans_host, torch.empty_like(trans_host).pin_memory()]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]

    def upload(i):
        sl = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[sl])       # the forward that last read this buffer has finished
            for k in keys:
                stagings[sl][k].copy_(host[i % NB][k], non_blocking=True)
            ready[sl].record(copy_stream)

    def run_e2e(nsteps):
        checksum = 0.0
        for sl in range(2):
            consumed[sl].record(comp_stream)
        upload(0)
        for i in range(nsteps):
            sl = i % 2
            if i + 1 < nsteps:
                upload(i + 1)
            comp_stream.wait_event(ready[sl])
            o = graphed(stagings[sl])
            consumed[sl].record(comp_stream)
            rot_hosts[sl].copy_(o["rot"], non_blocking=True)
            trans_hosts[sl].copy_(o["trans"], non_blocking=True)
            done[sl].record(comp_stream)
            if i > 0:                                   # read the previous step's poses on the host
                done[1 - sl].synchronize()
                checksum += float(trans_hosts[1 - sl][0, 2])
        done[(nsteps - 1) % 2].synchronize()
        checksum += float(trans_hosts[(nsteps - 1) % 2][0, 2])
        return checksum

    for sl in range(2):
        for k in keys:
            stagings[sl][k].copy_(host[sl][k])   # valid contents before the capture warm-up runs
        torch.cuda.synchronize()
        graphed(stagings[sl])
    run_e2e(2)
    barrier()
    e0.record()
    run_e2e(args.steps)
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    e2e_value = world * BATCH * args.steps / (ms_e2e / 1e3)

    # ---------------- roofline of the dominant kernel family (tcgen05 GEMMs), measured live with CUDA events ----------------
    import ctypes
    peaks = load_peaks(ms_total / 1e3)
    L.gdrn_model_set_profiling(model._handle, 1)
    ms3 = (ctypes.c_float * 3)()
    n3 = (ctypes.c_int * 3)()
    gemm_ms, gemm_n, dw_ms, other_ms = 0.0, 0, 0.0, 0.0
    reps = 3
    for i in range(reps):
        fwd(resident[i % NB])
        _lib.check(L.gdrn_model_get_profile(model._handle, ms3, n3), "get_profile")
        gemm_ms += ms3[0] / reps
        dw_ms += ms3[1] / reps
        other_ms += ms3[2] / reps
        gemm_n = n3[0]
    L.gdrn_model_set_profiling(model._handle, 0)
    x3 = args.precision == "bf16x3"
    gemm_tflops = BATCH * GEMM_GFLOP_PER_ROI_EXECUTED / gemm_ms if gemm_ms > 0 else 0.0  # GFLOP / ms = TFLOP/s (algorithmic)
    # DRAM bytes per GEMM launch from the committed ncu capture of this same command (profiles/, tools/make_traffic.py)
    traffic, traffic_src = None, None
    for tname in (("r02_traffic_x3.json" if x3 else "r02_traffic_bf16.json"), "r01_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", tname)
        if not os.path.exists(tpath) or (x3 and tname == "r01_traffic.json"):
            continue
        try:
            tj = json.load(open(tpath))
            fam = [v for k, v in tj["families"].items() if k.startswith("gemm")]
            if fam:
                traffic = fam[0]["dram_bytes_per_launch"]
                traffic_src = "profiles/%s (ncu dram__bytes_read.sum + dram__bytes_write.sum, mean over the %d tcgen05 GEMM " \
                              "launches of one step; build %s)" % (tname, fam[0]["launches"], tj.get("build", "see file"))
                break
        except Exception:  # noqa: BLE001
            traffic = None
    # tensor-pipe activity of the whole forward (BASELINE.json metric: "backbone tensor-pipe %") from the committed ncu
    # launch list of this same workload (profiles/r02_step_tensor.json, tools/r02b_ncu_step.sh + step_tensor_share.py)
    tensor_pipe = None
    tp_path = os.path.join(ROOT, "profiles", "r02_step_tensor.json")
    if x3 and os.path.exists(tp_path):
        try:
            tj = json.load(open(tp_path))
            tensor_pipe = {"forward_pct_of_elapsed": tj["tensor_pipe_pct_of_elapsed_forward"],
                           "tcgen05_kernels_pct_of_elapsed": tj["tensor_pipe_pct_of_elapsed_tcgen05_kernels"],
                           "tcgen05_kernels_pct_of_active": tj["tensor_pipe_pct_of_active_tcgen05_kernels"],
                           "tcgen05_time_share": tj["tcgen05_time_share"],
                           "source": "profiles/r02_step_tensor.json (ncu sm__pipe_tensor_cycles_active, time-weighted over the %d "
                                     "launches of one forward; build %s)" % (tj["launches"], tj.get("build"))}
        except Exception:  # noqa: BLE001
            tensor_pipe = None
    step_ms = ms_total / args.steps
    roofline = {
        "bound": "tensor",
        "kernel": ("gemm_pair_x3_kernel + gemm_tc_kernel (split-bf16 tcgen05/TMA implicit GEMM, all %d launches of a step)" if x3
                   else "gemm_tc_kernel + gemm_pair_kernel + mlp_fused_kernel (tcgen05/TMA implicit GEMM, all %d launches of a step)") % gemm_n,
        "achieved": gemm_tflops, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
        "frac": gemm_tflops / peaks["bf16_tflops"], "traffic": traffic, "traffic_source": traffic_src,
        "algorithmic_flop_per_launch": BATCH * GEMM_GFLOP_PER_ROI_EXECUTED * 1e9 / max(gemm_n, 1),
        "avg_launch_us": gemm_ms * 1e3 / max(gemm_n, 1), "peak_source": peaks["source"],
        "gemm_ms_per_step": gemm_ms, "dwconv_ms_per_step": dw_ms, "other_ms_per_step": other_ms,
        "whole_step_tflops_reference_flops": BATCH * GFLOP_PER_ROI_REFERENCE / step_ms,
        "whole_step_frac_reference_flops": BATCH * GFLOP_PER_ROI_REFERENCE / step_ms / peaks["bf16_tflops"],
        "whole_step_tflops_executed_flops": BATCH * GFLOP_PER_ROI_EXECUTED / step_ms,
        "tensor_pipe": tensor_pipe,
    }
    if x3:
        # `achieved` / `frac` count every multiply-add of the reference's fp32 GEMMs ONCE (algorithmic work).  The
        # tensor pipe issues three bf16 products per algorithmic MAC to reach fp32-class accuracy, so frac tops out at
        # 1/3; tensor_executed_* is what ncu's sm__pipe_tensor_cycles_active corresponds to.
        roofline.update({"products_per_mac": 3, "x3_ceiling_frac": 1.0 / 3.0,
                         "tensor_executed_tflops": 3 * gemm_tflops,
                         "tensor_executed_frac": 3 * gemm_tflops / peaks["bf16_tflops"]})

    # ---------------- secondary records (rank 0, one GPU): bf16 throughput mode, eager-GPU stand-in, native ops ----------------
    alt, eager, native, backbones = None, None, None, None
    if world == 1 and not args.no_secondary:
        other = "bf16" if x3 else "bf16x3"
        m2 = GDRN_DoubleMask(default_cfg(), max_batch=BATCH, precision=other)
        m2.load_state_dict(make_state_dict())
        m2.to(dev)
        g2 = make_graphed(m2)
        for i in range(NB):
            g2(resident[i])
        torch.cuda.synchronize()
        n2 = min(args.steps, 20)
        e0.record()
        for i in range(n2):
            g2(resident[i % NB])
        e1.record()
        torch.cuda.synchronize()
        ms2 = e0.elapsed_time(e1) / n2
        alt = {"precision": other, "value": BATCH / ms2 * 1e3, "unit": "ROIs/s", "ms_per_step": ms2, "steps": n2,
               "graph_replay": bool(use_graphs),
               "note": ("bf16 operands: R within ~0.03 rad / t within ~1e-3 of the fp32 oracle -- below the north-star parity bar, "
                        "a throughput mode only (tests/test_gpu_parity.py::test_forward_vs_oracle_b64[bf16])") if x3 else
                       "split-bf16 parity mode (R within 1e-4 rad / t within 1e-3)"}
        del m2, g2
        torch.cuda.empty_cache()
        # the other ConvNeXt widths the reference's backbone factory accepts (BASELINE configs[0] names convnext_tiny), same batch,
        # same precision mode; parity: tests/test_gpu_parity.py::test_forward_vs_oracle_convnext_tiny_small
        backbones = []
        for arch in ("convnext_tiny", "convnext_small"):
            try:
                m3 = GDRN_DoubleMask(default_cfg(arch=arch), arch=arch, max_batch=BATCH, precision=args.precision)
                m3.load_state_dict(make_state_dict(arch=arch))
                m3.to(dev)
                g3 = make_graphed(m3)
                for i in range(NB):
                    g3(resident[i])
                torch.cuda.synchronize()
                n3 = min(args.steps, 20)
                e0.record()
                for i in range(n3):
                    g3(resident[i % NB])
                e1.record()
                torch.cuda.synchronize()
                ms3 = e0.elapsed_time(e1) / n3
                backbones.append({"arch": arch, "precision": args.precision, "value": BATCH / ms3 * 1e3, "unit": "ROIs/s",
                                  "ms_per_step": ms3, "steps": n3, "graph_replay": bool(use_graphs)})
                del m3, g3
                torch.cuda.empty_cache()
            except Exception as e:  # noqa: BLE001
                backbones.append({"arch": arch, "error": "%s: %s" % (type(e).__name__, e)})
        try:
            eager = gpu_eager_baseline(dev)
        except Exception as e:  # noqa: BLE001
            eager = {"error": "%s: %s" % (type(e).__name__, e)}
        try:
            import bench_native

            native = bench_native.run(dev, peaks, ["fps", "voting", "nnd", "flow", "raster", "upnp", "refine", "ycbv5"], args.precision)
        except Exception as e:  # noqa: BLE001
            native = [{"error": "%s: %s" % (type(e).__name__, e)}]

    if world > 1:
        dist.barrier()
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            from oracle import gdrn_model_oracle as O

            threads = host_threads()
            torch.set_num_threads(threads)
            sd = make_state_dict()
            cb = {k: v[:CPU_SAMPLE_ROIS] for k, v in make_batch(B=BATCH, seed=0).items()}
            with torch.no_grad():
                O.gdrn_forward(sd, {k: v[:1] for k, v in cb.items()})  # warm the allocator / thread pool
                t0 = time.perf_counter()
                reps_cpu = 3
                for _ in range(reps_cpu):
                    O.gdrn_forward(sd, cb)
                dt = (time.perf_counter() - t0) / reps_cpu
            cpu = {"value": CPU_SAMPLE_ROIS / dt, "unit": "ROIs/s", "cores": threads, "kind": "port",
                   "sample": "%d ROIs of the 64-ROI batch (seed 0) x %d repetitions, oracle forward (torch CPU fp32), %.1f s per "
                             "repetition" % (CPU_SAMPLE_ROIS, reps_cpu, dt)}
        out = {
            "metric": METRIC,
            "value": value, "unit": "ROIs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.precision, "data": "synthetic",
            "config": workload_config(world, args.precision),
            "e2e": {"value": e2e_value, "unit": "ROIs/s", "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": d2h_bytes, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "parity": {"mode": args.precision,
                       "bar": "R within 1e-4 rad, t within 1e-3 of the fp32 reference path (BASELINE.json north_star)",
                       "met": bool(x3), "test": "tests/test_gpu_parity.py::test_forward_vs_oracle_b64 (this batch, these weights)"},
            "bf16_mode" if x3 else "bf16x3_mode": alt,
            "other_backbones": backbones,
            "gpu_eager_baseline": eager,
            "native_ops": native,
        }
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
