#!/usr/bin/env python
"""bench.py -- MonoRec hot-path benchmark (contract: task statement / SURVEY.md §8d).

Metric: keyframes/s (B x forwards / s) at 256x512, 32 depth planes, 4 source frames (BASELINE.json).
Workload at N=1: BASELINE config 2 -- synthetic KITTI-shaped inputs, batch 8, fused warp+SSIM cost-volume kernel only.
N>1: BASELINE config 4 -- one process per GPU (torchrun), 16 keyframes per GPU (weak scaling; the global batch is the
128 of config 4 at N=8), no data-path collective in the cost-volume path (it shards on independent keyframes, SURVEY.md §8e);
the whole-model objects (`full_model*`) include the NCCL all-gather of the per-rank `result` maps in their timed region.
`--config hires` is BASELINE config 5: 512x1024, 64 planes, 6 source frames, batch 4 per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config default|hires] [--dump-outputs DIR]

`--steps K` is the number of timed steps of the cost-volume path, on the device and through the host-buffer entry (e2e),
or of the reference arm (default 200; 5 for the slow reference arm).  The informational whole-model, loss and CPU-baseline
timings keep their own fixed counts.  `--dump-outputs DIR` writes what the last timed step computed (rank 0's cost volume and
single-frame volumes; the oracle port's in the reference arm) to DIR/<name>.npy, sampled as dump_outputs() describes, so
that two builds run with the same arguments can be compared.

`--impl reference` times the reference's CPU implementation of the path.  The reference is pure Python/PyTorch and
cannot travel to the GPU box, so this arm runs the oracle port (oracle/cost_volume_oracle.py: the same torch CPU
primitives in the same order, pinned on golden vectors from the reference) on the host cores.
"""
import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

H, W, D, F = 256, 512, 32, 4
B_PER_GPU = 8
B_PER_GPU_SHARDED = 16                     # BASELINE config 4: batch 128 sharded over 8 GPUs = 16 per GPU (used for every N > 1)
INV_LO, INV_HI = 0.0025, 0.33
METRIC = "keyframes_per_s_256x512_D32_F4"
ALG_BYTES_PER_KEYFRAME = 4 * H * W * (1 + F) * (3 + D)   # SURVEY.md §8d: every input read once, every output written once


def set_config(name):
    global H, W, D, F, B_PER_GPU, METRIC, ALG_BYTES_PER_KEYFRAME
    if name == "hires":                    # BASELINE config 5
        H, W, D, F, B_PER_GPU = 512, 1024, 64, 6, 4
        METRIC = "keyframes_per_s_512x1024_D64_F6"
    ALG_BYTES_PER_KEYFRAME = 4 * H * W * (1 + F) * (3 + D)


def k1_traffic(config, batch):
    """DRAM bytes per launch of the cost-volume kernel from the committed `ncu --set full` capture -- valid only for the
    kernel source it was taken from: the file stores the SHA-256 of csrc/cost_volume.cu and of the launch shape; any
    mismatch (a changed kernel, another batch) reports null instead of a stale number."""
    import hashlib
    p = ROOT / "profiles" / "r02_k1_traffic.json"
    if not p.exists():
        return None, "no capture committed"
    rec = json.loads(p.read_text())
    sha = hashlib.sha256((ROOT / "monorec_b200" / "csrc" / "cost_volume.cu").read_bytes()).hexdigest()
    ent = rec.get(f"{config}_b{batch}")
    if ent is None:
        return None, f"no capture for config {config} at batch {batch}"
    if ent.get("cost_volume_cu_sha256") != sha:
        return None, "capture predates the current cost_volume.cu"
    return float(ent["traffic_bytes_per_launch"]), "ncu --set full: dram__bytes_read.sum + dram__bytes_write.sum, " + ent.get("capture", "")


def pin_to_gpu_numa_node(index):
    """Runs this process on the CPUs NVML reports as local to GPU `index` before any pinned host buffer is allocated, so that
    first-touch places those buffers on the GPU's NUMA node (the e2e copies then stay off the inter-socket link)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n)
        cpus = [64 * i + b for i, w in enumerate(mask) for b in range(64) if (int(w) >> b) & 1]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """Samples SM clocks / throttle reasons through NVML every 20 ms while the timed region runs."""

    def __init__(self, index):
        self.index, self.rows, self.stop, self.t = index, [], threading.Event(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self.stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                    nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((sm, reasons))
            except Exception:
                pass
            time.sleep(0.02)

    def __enter__(self):
        if self.nv is not None:
            self.t = threading.Thread(target=self._run, daemon=True)
            self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        if self.t is not None:
            self.t.join(timeout=1)

    def summary(self):
        if self.nv is None or not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        nv = self.nv
        sm = sorted(r[0] for r in self.rows)
        bits = 0
        for r in self.rows:
            bits |= r[1]
        names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4}
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception:
            mx = None
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": [n for n, m in names.items() if bits & m],
                "samples": len(sm)}


def cpu_port_keyframes_per_s(repeats, threads=None):
    """The oracle port of CostVolumeModule.forward on the host cores, B=1 (the reference loops over the batch in
    Python, monorec_model.py:193, so its time is linear in B)."""
    from oracle import cost_volume_oracle as O
    from monorec_b200.synthetic import make_inputs
    if threads:
        torch.set_num_threads(threads)
    try:
        os.sched_setaffinity(0, range(os.cpu_count()))   # undo the NUMA pinning of the GPU part: use every host core
    except Exception:
        pass
    data = make_inputs(1, F, H, W, seed=0)
    O.cost_volume_torch(data, INV_HI, INV_LO, D)   # warm-up
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        O.cost_volume_torch(data, INV_HI, INV_LO, D)
        best = min(best, time.perf_counter() - t0)
    return 1.0 / best, torch.get_num_threads()


def run_reference(args, rank):
    if rank != 0:
        return
    steps = args.steps
    from oracle import cost_volume_oracle as O
    from monorec_b200.synthetic import make_inputs
    data = make_inputs(1, F, H, W, seed=0)
    # thread count: whichever of torch's default (physical cores) and every logical CPU is faster on this host, decided
    # by one untimed pass each (these double as warm-up); oversubscribing the hyper-threads usually loses
    candidates = sorted({torch.get_num_threads(), os.cpu_count() or 1})
    O.cost_volume_torch(data, INV_HI, INV_LO, D)
    trial = {}
    for n in candidates:
        torch.set_num_threads(n)
        t0 = time.perf_counter()
        O.cost_volume_torch(data, INV_HI, INV_LO, D)
        trial[n] = time.perf_counter() - t0
    torch.set_num_threads(min(trial, key=trial.get))
    t0 = time.perf_counter()
    for _ in range(steps):
        cv, sf = O.cost_volume_torch(data, INV_HI, INV_LO, D)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, cv, torch.stack(sf))
    val = steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "keyframes/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": 1 + len(candidates), "ms_per_step": 1e3 * dt / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"cost_volume_{H}x{W}_D{D}_F{F}, one keyframe per step "
                                   "(bounded sample: the reference is linear in batch)", "batch_per_step": 1},
            "cpu_baseline": {"value": val, "unit": "keyframes/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": f"{steps} x 1 keyframe, torch CPU ops, {torch.get_num_threads()} threads (fastest of {candidates})"},
            "e2e": {"value": val, "unit": "keyframes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


DUMP_BYTES = 48 << 20                     # at most this much float32 in one --dump-outputs directory


def dump_outputs(out_dir, cv, sfcv):
    """Writes the cost-volume outputs as float32 .npy files: cost_volume.npy [N, D] and single_frame_cvs.npy [N, F, D],
    the full depth-plane profile of N pixels (b, y, x).  The pixels are the first N of a permutation drawn from a CPU
    generator with a fixed seed, in ascending order, N as large as DUMP_BYTES allows (every pixel if all fit): the same
    arguments dump the same pixels on every run and every build."""
    import numpy as np
    nF, B, nD, h, w = sfcv.shape
    n = min(B * h * w, DUMP_BYTES // (4 * nD * (1 + nF)))
    pix = torch.randperm(B * h * w, generator=torch.Generator().manual_seed(0))[:n].sort().values.to(cv.device)
    b, y, x = pix // (h * w), pix // w % h, pix % w
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / "cost_volume.npy", cv[b, :, y, x].float().cpu().numpy())
    np.save(out_dir / "single_frame_cvs.npy", sfcv.permute(1, 3, 4, 0, 2)[b, y, x].float().cpu().numpy())


_REAL_STDOUT = None


def quiet_stdout():
    """Library chatter (NCCL's version banner, download messages, ...) must not end up next to the JSON line: everything
    written to fd 1 during the run goes to stderr; emit() writes the one result line to the real stdout."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 200; 5 with --impl reference)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="default", choices=["default", "hires"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-full-model", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 5 if args.impl == "reference" else 200
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    set_config(args.config)
    if args.impl == "reference":
        run_reference(args, rank)
        return
    args.warmup = max(args.warmup, 3)      # timing rules: at least 3 warm-up steps (the JSON line reports the number used)
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback in the product path)"
    numa_cpus = pin_to_gpu_numa_node(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from monorec_b200 import _lib
    from monorec_b200.synthetic import make_inputs, to_device
    lib = _lib.load()
    # N = 1: the configuration the metric is quoted on (batch 8); N > 1: BASELINE config 4's shard size, 16 keyframes per GPU
    # (global batch 16 N = 128 at N = 8; weak scaling); hires: 4 per GPU at every N
    B = B_PER_GPU if (world == 1 or args.config == "hires") else B_PER_GPU_SHARDED
    # rotating input sets whose images together exceed the 126 MB L2, so no step finds its inputs cached from the previous one
    set_bytes = B * (1 + F) * 3 * H * W * 4
    NSETS = max(2, min(4, -(-256 * 1024 * 1024 // set_bytes)))
    sets = []
    for i in range(NSETS):
        d = to_device(make_inputs(B, F, H, W, seed=100 * rank + i), dev)
        sets.append(d)
    proj = torch.empty(B, F, 3, 4, device=dev)
    depths = torch.empty(D, device=dev)
    cv = torch.empty(B, D, H, W, device=dev)
    sfcv = torch.empty(F, B, D, H, W, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    k_start = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    k_stop = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]

    def step(i, timed_idx=None):
        d = sets[i % NSETS]
        _lib.check(lib.mr_projection_tables(d["keyframe_pose"].data_ptr(), d["keyframe_intrinsics"].data_ptr(),
                                            _lib.ptr_array(d["poses"]), _lib.ptr_array(d["intrinsics"]), B, F, H, W,
                                            proj.data_ptr(), depths.data_ptr(), D, INV_LO, INV_HI, stream), "tables")
        if timed_idx is not None:
            k_start[timed_idx].record()
        _lib.check(lib.mr_cost_volume_fwd(d["keyframe"].data_ptr(), _lib.ptr_array(d["frames"]), proj.data_ptr(),
                                          depths.data_ptr(), cv.data_ptr(), sfcv.data_ptr(), B, F, D, H, W, 10.0, None,
                                          stream), "cost volume")
        if timed_idx is not None:
            k_stop[timed_idx].record()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    _lib.launch_count(reset=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        barrier()
        ev0.record()
        for i in range(args.steps):
            step(args.warmup + i, timed_idx=i)
        ev1.record()
        barrier()
    ms = ev0.elapsed_time(ev1)
    launches = _lib.launch_count(reset=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, cv, sfcv)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    kernel_ms = sum(a.elapsed_time(b) for a, b in zip(k_start, k_stop)) / args.steps
    value = world * B * args.steps / (ms * 1e-3)

    line = None
    if rank == 0:
        peak, peak_src = hbm_peak()
        achieved = ALG_BYTES_PER_KEYFRAME * B / (kernel_ms * 1e-3) / 1e9
        traffic, traffic_note = k1_traffic(args.config, B)
        cfg_name = ("BASELINE config 5 (hi-res)" if args.config == "hires" else
                    ("BASELINE config 2: fused warp+SSIM kernel only" if world == 1 else
                     f"BASELINE config 4 shard size: {B} keyframes per GPU, global batch {B * world} over {world} GPUs"))
        line = {"metric": METRIC, "value": value, "unit": "keyframes/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"cost_volume_{H}x{W}_D{D}_F{F} ({cfg_name})",
                           "batch_per_gpu": B, "global_batch": B * world, "src_frames": F, "depth_planes": D,
                           "height": H, "width": W, "parallelism": f"dp{world} (independent keyframes, no collective)",
                           "l2": f"inputs rotate over {NSETS} sets ({NSETS * set_bytes >> 20} MiB) > 126 MB L2; "
                                 f"{(1 + F) * B * D * H * W * 4 >> 20} MiB of outputs per step",
                           "host_numa_cpus": numa_cpus},
                "gpu_launches": launches,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_note, "peak_source": f"{peak_src} (burst copy)",
                             "kernel": "cost_volume_kernel (the events bracket mr_cost_volume_fwd: one launch)",
                             "kernel_ms": kernel_ms,
                             "algorithmic_bytes_per_launch": ALG_BYTES_PER_KEYFRAME * B},
                "clocks": clocks.summary()}

    # ---- e2e: the same path through the host-buffer C-ABI entry (pinned host memory, copies inside the timed region)
    if not args.no_e2e:
        host = make_inputs(B, F, H, W, seed=7 + rank)
        h_key = host["keyframe"].contiguous().pin_memory()
        h_frames = torch.stack(host["frames"]).contiguous().pin_memory()
        h_kp = host["keyframe_pose"].contiguous().pin_memory()
        h_kk = host["keyframe_intrinsics"].contiguous().pin_memory()
        h_poses = torch.stack(host["poses"]).contiguous().pin_memory()
        h_intr = torch.stack(host["intrinsics"]).contiguous().pin_memory()
        h_cv = torch.empty(B, D, H, W).pin_memory()
        ws_bytes = lib.mr_cost_volume_host_workspace(B, F, D, H, W)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)

        def e2e_step():
            _lib.check(lib.mr_cost_volume_host(h_key.data_ptr(), h_frames.data_ptr(), h_kp.data_ptr(), h_kk.data_ptr(),
                                               h_poses.data_ptr(), h_intr.data_ptr(), h_cv.data_ptr(), None,
                                               B, F, D, H, W, INV_LO, INV_HI, 10.0, ws.data_ptr(), ws_bytes), "e2e")
        for _ in range(3):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()      # synchronous: returns after the last D2H copy has landed
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if rank == 0:
            h2d = (1 + F) * B * 3 * H * W * 4 + (2 + 2 * F) * B * 64
            d2h = B * D * H * W * 4
            line["e2e"] = {"value": world * B * args.steps / float(t.item()), "unit": "keyframes/s",
                           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": args.steps,
                           "api": "mr_cost_volume_host (C ABI, pinned host buffers NUMA-local to the GPU; images and matrices "
                                  "uploaded, fused cost volume downloaded, single-frame volumes left on the device for the "
                                  "MaskModule as in monorec_model.py:693-699)"}

    # ---- informational: the whole MonoRecModel.forward (cost volume + ResNet-18 + mask/depth conv stacks on the tensor
    #      cores) replayed from a CUDA graph, batch sharded like above, per-rank result maps all-gathered over NCCL ----
    if not args.no_full_model:
        from monorec_b200 import conv as C
        from monorec_b200.dist import all_gather_batch
        from monorec_b200.model import GraphedMonoRec, MonoRecModel
        torch.manual_seed(0)
        model = MonoRecModel().to(dev).eval()          # random-init weights of the reference architecture
        default_mode = C.MODE
        for key, mode in (("full_model", "tf32"), ("full_model_f16", "f16")):
            C.set_mode(mode)
            C.FLOPS = [0]
            with torch.no_grad():
                model(dict(sets[0]))             # one eager forward: counts the conv stacks' multiply-adds
            conv_flops, C.FLOPS = C.FLOPS[0], None
            gm = GraphedMonoRec(model, sets[0])
            fm_steps = 20 if B <= 16 else 5
            for i in range(3):
                all_gather_batch(gm(sets[i % NSETS])["result"], equal_shards=True)
            barrier()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            for i in range(fm_steps):
                res = all_gather_batch(gm(sets[i % NSETS])["result"], equal_shards=True)
            f1.record()
            barrier()
            t = torch.tensor([f0.elapsed_time(f1)], device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            if rank == 0:
                fms = float(t.item()) / fm_steps
                tpeak = None
                pk = ROOT / "MEASURED_PEAKS.json"
                if pk.exists():
                    tpeak = float(json.loads(pk.read_text()).get("bf16_tflops_sustained", 0.0)) or None
                tach = conv_flops / (fms * 1e-3) / 1e12
                line[key] = {"value": world * B / (fms * 1e-3), "unit": "keyframes/s", "ms_per_forward": fms,
                             "batch_per_gpu": B, "global_batch": B * world, "conv_arithmetic": mode,
                             "gathered_result_shape": list(res.shape),
                             "roofline": {"bound": "tensor", "achieved": tach, "peak": tpeak if tpeak else 1400.0,
                                          "unit": "TFLOP/s", "frac": tach / (tpeak if tpeak else 1400.0),
                                          "peak_source": "measured (sustained bf16 GEMM)" if tpeak else "fallback",
                                          "flops_per_forward": conv_flops,
                                          "note": "MaskModule + DepthModule multiply-adds (x2) over the whole forward time "
                                                  "(cost volume, ResNet-18 trunk and the all-gather included in the time)"},
                             "what": "MonoRecModel.forward (CUDA-graph replay) + NCCL all-gather of result; "
                                     "inputs resident, random-init weights"}
            # the same forward from pinned HOST tensors to a HOST result (what example/test_monorec.py:45-53 does with
            # to(batch, device) ... .cpu()): H2D of the dict + graph replay + D2H of `result` inside the timed region.
            # Informational and guarded: a failure here must never cost the JSON line.
            try:
                hsets = []
                for i in range(2):
                    hd = make_inputs(B, F, H, W, seed=900 + 10 * rank + i)
                    hsets.append({k: ([t.contiguous().pin_memory() for t in v] if isinstance(v, (list, tuple)) else
                                      (v.contiguous().pin_memory() if torch.is_tensor(v) else v)) for k, v in hd.items()})
                h_res = torch.empty(B, 1, H, W).pin_memory()

                def host_step(i):
                    out = gm(hsets[i % 2])["result"]
                    h_res.copy_(out, non_blocking=True)
                    torch.cuda.synchronize()
                for i in range(2):
                    host_step(i)
                t0 = time.perf_counter()          # no collective in this guarded block: rank 0's own clock, x world
                for i in range(10):
                    host_step(i)
                dt = torch.tensor([time.perf_counter() - t0])
                if rank == 0:
                    h2d = sum(t.numel() * t.element_size() for v in hsets[0].values()
                              for t in (v if isinstance(v, (list, tuple)) else [v]) if torch.is_tensor(t))
                    line[key]["host_to_host"] = {"value": world * B * 10 / float(dt.item()), "unit": "keyframes/s",
                                                 "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": h_res.numel() * 4}
            except Exception as exc:   # noqa: BLE001
                if rank == 0 and line is not None and key in line:
                    line[key]["host_to_host_error"] = f"{type(exc).__name__}: {exc}"[:200]
            del gm
        # BASELINE config 3 proper: full model, batch 16, half arithmetic, one GPU (guarded, single-GPU runs only)
        if world == 1:
            try:
                C.set_mode("f16")
                B16 = 16
                sets16 = [to_device(make_inputs(B16, F, H, W, seed=500 + i), dev) for i in range(2)]
                gm = GraphedMonoRec(model, sets16[0])
                for i in range(3):
                    gm(sets16[i % 2])
                torch.cuda.synchronize()
                f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                f0.record()
                for i in range(10):
                    res = gm(sets16[i % 2])["result"]
                f1.record()
                torch.cuda.synchronize()
                fms = f0.elapsed_time(f1) / 10
                line["full_model_f16_b16"] = {"value": B16 / (fms * 1e-3), "unit": "keyframes/s", "ms_per_forward": fms,
                                              "batch_per_gpu": B16, "conv_arithmetic": "f16", "result_shape": list(res.shape),
                                              "what": "BASELINE config 3: MonoRecModel.forward (CUDA-graph replay), batch 16, "
                                                      "inputs resident (2 rotating sets), random-init weights"}
                del gm, sets16
            except Exception as exc:   # noqa: BLE001
                line["full_model_f16_b16_error"] = f"{type(exc).__name__}: {exc}"[:200]
        C.set_mode(default_mode)
        del model

    # SURVEY 8f row 4 (informational, single-GPU runs): the photometric reprojection loss, forward and forward + backward
    if world == 1 and not args.no_full_model:
        try:
            from monorec_b200 import losses as RL
            invd = (0.15 + 0.1 * torch.rand(B, 1, H, W, device=dev)).requires_grad_(True)
            rd = sets[0]

            def _fwd():
                with torch.no_grad():
                    RL.reprojection_loss(invd, rd, automasking=True, reduce=False)

            def _fwd_bwd():
                invd.grad = None
                RL.reprojection_loss(invd, rd, automasking=True, reduce=True).backward()

            times = []
            for fn in (_fwd, _fwd_bwd):
                for _ in range(3):
                    fn()
                torch.cuda.synchronize()
                r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                r0.record()
                for _ in range(20):
                    fn()
                r1.record()
                torch.cuda.synchronize()
                times.append(r0.elapsed_time(r1) / 20)
            line["reprojection_loss"] = {"forward_ms": times[0], "forward_backward_ms": times[1], "batch": B, "frames": F,
                                         "what": "monorec_b200.losses.reprojection_loss(automasking=True) on the bench inputs: "
                                                 "mr_reprojection_loss_fwd / _bwd through autograd (eager, incl. mr_projection_tables)"}
        except Exception as exc:   # noqa: BLE001
            line["reprojection_loss_error"] = f"{type(exc).__name__}: {exc}"[:200]

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, cores = cpu_port_keyframes_per_s(repeats=2)
        line["cpu_baseline"] = {"value": v, "unit": "keyframes/s", "cores": cores, "kind": "port",
                                "sample": "1 keyframe (B=1, F=4, D=32, 256x512), best of 2 after 1 warm-up"}
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
