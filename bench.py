#!/usr/bin/env python
"""Benchmark of the SceneEgo volumetric lifting stage (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W                # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...      # reference algorithm on the host CPU (oracle port)
    python bench.py --impl reference-gpu --frames-per-gpu 256    # reference algorithm with stock torch CUDA ops, fp32
                                                                 # (the denominator of north_star's ">= 50x" target)

A "step" is one pass of the hot path (everything VoxelNetwork_depth.forward does after
the backbone) over one batch of synthetic input: per GPU 64 frames of backbone features
(64,256,64,64) f32 + depth maps (64,1024,1280) f32, V=64, 15 joints, random-init weights
(BASELINE.json configs[1]).  Frames are sharded over ranks (weak scaling: 64 frames per
GPU; `--global-frames` shards a fixed total instead) with no data-path collective; the
poses of all timed steps are all-gathered over NCCL ONCE, at the end of the timed region
(north_star: "NCCL only for the final gather of poses").  Rank 0 prints ONE JSON line.

Other BASELINE configs: `--frames-per-gpu B` / `--global-frames B` (configs[2] sweep; `--sweep a,b,c` runs several
totals in one process, one JSON line each), `--volume-size 128` (configs[3]), `--graph` (CUDA-graph lift for the
batch-1 demo.py case), tools/microbench_geometry.py (configs[4]).

`--dump-outputs DIR` writes the 4-tuple that the last timed step returned (keypoints_3d, features, volumes,
coord_volumes) as DIR/<name>.npy in float32, so that two builds can be compared output for output on identical
seeded inputs.  An output larger than DUMP_SAMPLE elements is written as a fixed, seeded sample of its elements.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "frames/s VoxelNetDepth volumetric stage"
UNIT = "frames/s"
FRAMES_PER_GPU = 64
J = 15
FEATURES_BYTES_PER_FRAME = 32 * 1024 * 1280 * 4            # output #2 of the reference forward
FEATURES_BUDGET_BYTES = 100e9                              # above this, output #2 is not materialised (says so)
DUMP_SAMPLE = 1 << 21                                      # --dump-outputs: at most 8 MB per output, 32 MB in all


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--frames-per-gpu", type=int, default=FRAMES_PER_GPU)
    ap.add_argument("--global-frames", type=int, default=0, help="fixed total, sharded over the ranks (strong scaling)")
    ap.add_argument("--sweep", default="", help="comma-separated global frame counts: one JSON line each")
    ap.add_argument("--sweep-frames-cap", type=int, default=2560,
                    help="sweep lines time min(--steps, max(2, cap / frames per GPU)) steps (the default line always times --steps)")
    ap.add_argument("--volume-size", type=int, default=64)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-table", action="store_true", help="skip the per-kernel roofline pass")
    ap.add_argument("--chunk", type=int, default=64, help="frames per V2V launch group")
    ap.add_argument("--graph", action="store_true", help="replay the lift as a CUDA graph (batches <= 16)")
    ap.add_argument("--no-features", action="store_true", help="do not materialise output #2 (168 MB per frame)")
    ap.add_argument("--persistent-features", action="store_true", help="output #2 in one reused buffer")
    ap.add_argument("--raw-depth", action="store_true",
                    help="e2e ships raw 512x640 depth maps; the dataset's resize + clamp run inside the voxelisation")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--act-dtype", default="bf16", choices=["bf16", "f16"],
                    help="storage type of V2V activations / weights (bf16 = BASELINE configs[1]; f16 = the fp16 build)")
    ap.add_argument("--profile-ops", default="", help="write the per-op V2V timing table to this file")
    ap.add_argument("--out", default="", help="also append the JSON line(s) to this file")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the outputs of the last timed step (rank 0's frames) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def workload_config(frames, world, V=64, chunk=64, strong=False, features=True, graph=False):
    return {"workload": f"VoxelNetDepth post-backbone stage, batch {frames} frames/GPU, {V}^3 voxel cube, 15 joints, "
                        f"features (B,256,64,64) f32 + depth (B,1024,1280) f32, bf16 V2V, fp32 unprojection and "
                        f"soft-argmax (BASELINE.json configs[{1 if V == 64 else 3}])",
            "frames_per_gpu": frames, "global_frames": frames * world, "volume_size": V, "joints": J,
            "parallelism": f"frame-shard x{world}, one NCCL all-gather of the poses at the end of the timed region",
            "weights": "random init (seeded), BatchNorm statistics randomised",
            "outputs": ("reference-identical 4-tuple (features and softmaxed volumes materialised; the 168 MB/frame "
                        "features tensor is written on a side stream inside the timed region)") if features else
                       "poses + softmaxed volumes; output #2 (168 MB/frame features tensor) NOT materialised at this batch",
            "v2v_chunk_frames": min(chunk, frames),
            "cuda_graph": bool(graph),
            "l2_policy": "inputs (9.4 MB/frame) and activations (>1 GB/layer at 64 frames) exceed the 126 MB L2" if frames >= 16
                         else "L2 flushed (256 MB memset) between timed steps"}


def emit(line, args):
    s = json.dumps(line)
    print(s, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(s + "\n")


def dump_outputs(out_dir, outputs):
    """Write each output tensor (None: not materialised, skipped) as out_dir/<name>.npy in float32.  One with more
    than DUMP_SAMPLE elements is written flat, as its elements at DUMP_SAMPLE ascending flat indices drawn from a
    CPU generator seeded with 0: the same indices in every run with the same arguments."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        if t is None:
            continue
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randint(t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.float().cpu().numpy())


# --------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def wait_first_sample(self, timeout=8.0):
        # nvidia-smi's start-up (NVML initialisation over every GPU of the box) holds driver locks that stall kernel
        # launches for tens of milliseconds: wait for its first sample so that only the 100 ms polling overlaps the
        # timed region
        t = time.time()
        while self.proc is not None and not self.rows and time.time() - t < timeout:
            time.sleep(0.05)
        time.sleep(0.1)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def window(self, t0, t1):
        rows = [r for t, r in self.rows if t0 <= t <= t1 and len(r) >= 9] or [r for _, r in self.rows if len(r) >= 9]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[1]) for r in rows)
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "reasons": sorted(reasons),
                "samples": len(rows), "power_w_max": max(float(r[3]) for r in rows)}

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        return self.window(t0 if t0 is not None else 0.0, t1 if t1 is not None else time.time())


# --------------------------------------------------------------------------------------
# reference algorithm on the host CPU (oracle port -- the only place bench.py runs oracle/ on the CPU)
# --------------------------------------------------------------------------------------
def cpu_reference_frames_per_s(n_frames, repeats=1, warmup=0, V=64):
    import torch
    from oracle import sceneego_oracle as orc
    from sceneego_b200 import DEFAULT_CALIBRATION
    from sceneego_b200.utils import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    tables = orc.StageTables(DEFAULT_CALIBRATION, V, 2.0)
    sd = synth.synthetic_state_dict(synth.stage_state_shapes(), seed=0, mode="random_bn")
    feat = synth.synthetic_features(n_frames)
    depth = synth.synthetic_depth_room(n_frames, tables.ray)
    times = []
    for i in range(warmup + repeats):
        t0 = time.perf_counter()
        with torch.no_grad():
            orc.stage_forward(tables, sd, feat, depth_batch=depth)
        times.append(time.perf_counter() - t0)
    times = times[warmup:]
    return n_frames * len(times) / sum(times), cores, times


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # each step = ONE frame of the batch (bounded sample: the reference's voxelisation loop is serial per frame,
    # network/voxel_net_depth.py:252-256, and its torch CPU ops already use every core at B = 1, so frames/s
    # does not depend on the batch)
    fps, cores, times = cpu_reference_frames_per_s(1, repeats=args.steps, warmup=min(args.warmup, 1), V=args.volume_size)
    ms = 1000.0 * sum(times) / len(times)
    sample = ("1 frame per step of the same workload (oracle/sceneego_oracle.py, torch CPU threads = all host cores); "
              "the reference's per-frame loop makes frames/s independent of the batch size")
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.frames_per_gpu, args.gpus, args.volume_size, args.chunk),
            "frames_run_per_step": 1, "sample": sample,
            "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line, args)


# --------------------------------------------------------------------------------------
# reference algorithm on ONE GPU with stock torch CUDA ops, fp32, TF32 off, host NumPy voxelisation loop kept
# (network/voxel_net_depth.py:224-275 on device='cuda'): the denominator of north_star's ">= 50x" target
# --------------------------------------------------------------------------------------
def reference_gpu_arm(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import sceneego_oracle as orc
    from sceneego_b200 import DEFAULT_CALIBRATION
    from sceneego_b200.utils import synth
    if not torch.cuda.is_available():
        emit({"impl": "reference-gpu", "unavailable": "no CUDA device"}, args)
        return
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    V = args.volume_size
    B = args.frames_per_gpu if args.frames_per_gpu != FRAMES_PER_GPU else 256      # north_star: batch 256
    tables = orc.StageTables(DEFAULT_CALIBRATION, V, 2.0)
    sd = {k: v.to(dev) for k, v in synth.synthetic_state_dict(synth.stage_state_shapes(), seed=0, mode="random_bn").items()}
    feat = synth.synthetic_features(B).to(dev)
    depth = synth.synthetic_depth_room(B, tables.ray).to(dev)
    steps = max(1, min(args.steps, 3))
    res = None
    while B >= 1:
        try:
            with torch.no_grad():
                orc.stage_forward_device(tables, sd, feat[:B], depth[:B], dev)        # warm-up (cuDNN autotune, allocator)
                torch.cuda.synchronize()
                tot, host, vox_gpu_free = [], [], []
                for _ in range(steps):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    t0 = time.perf_counter()
                    e0.record()
                    _, _, _, tim = orc.stage_forward_device(tables, sd, feat[:B], depth[:B], dev, timings=True)
                    e1.record()
                    torch.cuda.synchronize()
                    tot.append(time.perf_counter() - t0)
                    host.append(tim["voxel_loop_s"])
            res = (B, tot, host)
            break
        except torch.cuda.OutOfMemoryError:
            torch.cuda.empty_cache()
            B //= 2
    if res is None:
        emit({"impl": "reference-gpu", "unavailable": "out of memory at every batch size"}, args)
        return
    B, tot, host = res
    t = sum(tot) / len(tot)
    th = sum(host) / len(host)
    cfg = workload_config(B, 1, V, args.chunk)
    cfg["workload"] = cfg["workload"].replace("bf16 V2V", "fp32 cuDNN V2V (TF32 off)")
    line = {"impl": "reference-gpu", "metric": METRIC, "value": B / t, "unit": UNIT, "n_gpus": 1, "steps": len(tot),
            "warmup": 1, "ms_per_step": 1000 * t, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "what": "the reference's op sequence (oracle/sceneego_oracle.py::stage_forward_device: nn.Conv2d + Upsample + "
                    "ConstantPad2d, F.grid_sample, per-frame host NumPy voxelisation with D2H/H2D like "
                    "network/voxel_net_depth.py:251-257, cuDNN fp32 Conv3d V2V, softmax + einsum) on one B200",
            "host_voxel_loop_ms_per_step": 1000 * th,
            "value_without_host_voxel_loop": B / max(t - th, 1e-9),
            "host_cores": os.cpu_count(),
            "e2e": {"value": B / t, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line, args)


# --------------------------------------------------------------------------------------
# this repo's arm
# --------------------------------------------------------------------------------------
def ours_arm(args):
    import torch
    import torch.distributed as dist
    from sceneego_b200 import parallel
    from sceneego_b200.network.voxel_net_depth import VoxelNetwork_depth
    from sceneego_b200.pipeline import HostStagePipeline
    from sceneego_b200.utils import cfg as cfgmod
    from sceneego_b200.utils import synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (this arm has no CPU fallback; use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = None if args.no_numa_bind else parallel.bind_to_gpu_numa_node(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    V = args.volume_size
    totals = [int(x) for x in args.sweep.split(",") if x] if args.sweep else [None]

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        sampler.wait_first_sample()

    import contextlib
    import io
    net = None
    steps_req = args.steps
    for total_req in totals:
        if total_req is not None:
            B = max(1, total_req // world)
            strong = True
        elif args.global_frames:
            B = max(1, args.global_frames // world)
            strong = True
        else:
            B = args.frames_per_gpu
            strong = False
        total = B * world
        features = not args.no_features and B * FEATURES_BYTES_PER_FRAME <= FEATURES_BUDGET_BYTES
        graph = args.graph and B <= 16
        if net is None:
            with contextlib.redirect_stdout(io.StringIO()):
                net = VoxelNetwork_depth(cfgmod.default_config(batch_size=max(B, 1), volume_size=V), device=f"cuda:{local}",
                                         v2v_chunk=args.chunk, persistent_features=args.persistent_features,
                                         graph_max_batch=16 if args.graph else 0).eval()
            sd = synth.synthetic_state_dict(synth.stage_state_shapes(), seed=0, mode="random_bn")
            full = net.state_dict()
            full.update(sd)
            net.load_state_dict(full, strict=True)
        net.materialize_features = features
        if total_req is not None:
            args.steps = max(2, min(steps_req, args.sweep_frames_cap // B))
        line = run_config(args, net, B, total, world, rank, local, dev, V, strong, features, graph, sampler, numa)
        if rank == 0:
            emit(line, args)
    if rank == 0:
        sampler.stop()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_config(args, net, B, total, world, rank, local, dev, V, strong, features, graph, sampler, numa):
    import torch
    import torch.distributed as dist
    from sceneego_b200 import parallel
    from sceneego_b200.pipeline import HostStagePipeline
    from sceneego_b200.utils import synth

    def pinned(t):
        return t.pin_memory()
    feat_h = pinned(synth.synthetic_features(B, seed=1234 + rank))
    depth_h = pinned(synth.synthetic_depth_room(B, net.ray, seed=7 + rank))
    feat_d, depth_d = feat_h.to(dev), depth_h.to(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev) if B < 16 else None

    last = {}

    def step(keep=False):
        if flush is not None:
            flush.zero_()                     # small batches fit the 126 MB L2: flush it between timed steps
        with torch.no_grad():
            out = net.lift(feat_d, net.grid_coord_proj_batch, net.coord_volumes, depth_map_batch=depth_d)
        if keep:
            last.update(zip(("keypoints_3d", "features", "volumes", "coord_volumes"), out))
        return out[0]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    for _ in range(warm):
        kp = step()
    if world > 1:
        parallel.gather_poses(kp, total)       # NCCL communicator set-up outside the timed region
    barrier()
    # ---- device-resident timing ----------------------------------------------------------
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    e0.record()
    launches = 0
    kps = []
    for i in range(args.steps):
        kps.append(step(keep=bool(args.dump_outputs) and i == args.steps - 1))
        launches += net.last_launches
    all_kp = torch.stack(kps)                              # (steps, B, J, 3)
    if world > 1:                                          # the ONE collective: final gather of the poses
        all_kp = parallel.gather_poses(all_kp.transpose(0, 1).contiguous(), total)
    e1.record()
    barrier()
    t_wall1 = time.time()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    if flush is not None:                                  # the flush memsets are not part of the stage: subtract them
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(args.steps):
            flush.zero_()
        f1.record()
        torch.cuda.synchronize()
        ms_total = max(ms_total - f0.elapsed_time(f1), 1e-3)
    clocks = sampler.window(t_wall0, t_wall1) if rank == 0 else None
    value = total * args.steps / (ms_total / 1000.0)
    assert torch.isfinite(all_kp).all()
    if last and rank == 0:
        dump_outputs(args.dump_outputs, last)
    last.clear()

    # ---- end to end: pinned host buffers -> H2D -> lift -> D2H, through the public pipeline ----
    if args.raw_depth:
        # what the reference's datasets read from disk: 512x640 maps (data/demo/depths/*.exr); their nearest resize to
        # 1024x1280 and the 10 m clamp (dataset/demo_dataset.py:86-91) run inside the voxelisation kernel
        raw_h = pinned(depth_h[:, ::2, ::2].contiguous())
        net.depth_preprocess = (1024, 1280, 10.0)
        e2e_inputs = (feat_h, raw_h)
    else:
        e2e_inputs = (feat_h, depth_h)
    pipe = HostStagePipeline(net, gather_fn=(lambda kp: parallel.gather_poses(kp, kp.shape[0] * world)) if world > 1 else None)
    pipe.run([e2e_inputs] * args.steps)       # same batch count as the timed call: pinned result buffers exist
    barrier()
    pipe.h2d_bytes = pipe.d2h_bytes = 0
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    outs = pipe.run([e2e_inputs] * args.steps)
    f1.record()
    barrier()
    ms2 = torch.tensor([f0.elapsed_time(f1)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_value = total * args.steps / (float(ms2.item()) / 1000.0)
    assert torch.isfinite(outs[-1]).all()
    net.depth_preprocess = None
    # the host->device copy of one step alone (explains the gap between `value` and `e2e`: PCIe / host memory, not kernels)
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stage_d = [torch.empty_like(t, device=dev) for t in e2e_inputs]
    barrier()
    g0.record()
    for _ in range(3):
        for d, h in zip(stage_d, e2e_inputs):
            d.copy_(h, non_blocking=True)
    g1.record()
    barrier()
    h2d_ms = torch.tensor([g0.elapsed_time(g1) / 3], device=dev)
    if world > 1:
        dist.all_reduce(h2d_ms, op=dist.ReduceOp.MAX)
    h2d_ms = float(h2d_ms.item())
    del stage_d

    if rank != 0:
        return None
    peaks = {}
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk_path):
        peaks = json.load(open(pk_path))
    cfg = workload_config(B, world, V, args.chunk, strong, features, graph)
    h2d_bytes = sum(t.numel() * 4 for t in e2e_inputs)
    ms_step = ms_total / args.steps
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": args.act_dtype, "data": "synthetic",
            "config": cfg, "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": pipe.h2d_bytes // args.steps,
                    "d2h_bytes_per_step": pipe.d2h_bytes // args.steps,
                    "api": "sceneego_b200.pipeline.HostStagePipeline.run (pinned host -> poses on host)",
                    "inputs": "features f32 + raw 512x640 depth (dataset resize/clamp fused into the voxelisation)"
                              if args.raw_depth else "features f32 + preprocessed 1024x1280 depth",
                    "h2d_alone_ms_per_step": h2d_ms,
                    "h2d_alone_GB_per_s": h2d_bytes / (h2d_ms * 1e-3) / 1e9,
                    "limiter": "host->device copy (PCIe / host memory)" if h2d_ms > ms_step else "GPU kernels",
                    "numa_node": numa},
            "gpu_launches": launches, "frames_per_s_per_gpu": value / world,
            "latency_ms_per_batch": ms_step}
    if not args.no_kernel_table:
        hbm_burst = float(peaks.get("hbm_gbs", 6650.0))
        tc_burst = float(peaks.get("bf16_tflops", 1590.0))
        tc_sust = float(peaks.get("bf16_tflops_sustained", 1400.0))
        peak_src = "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"
        kern = stage_kernel_timings(net, feat_d, depth_d, B, args, V, hbm_burst, tc_burst)
        line["kernels"] = kern
        line["roofline"] = roofline_block(kern, tc_burst, tc_sust, peak_src, V, ms_step, B)
    if world == 1 and not args.no_cpu_baseline and not args.sweep:
        fps, cores, times = cpu_reference_frames_per_s(2, repeats=1, warmup=0, V=V)
        line["cpu_baseline"] = {"value": fps, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"2 frames of the same workload through oracle/sceneego_oracle.py "
                                          f"(torch CPU, {cores} threads), {sum(times):.1f} s"}
    return line


def ncu_traffic(kernel_prefix, frames_per_launch, V):
    """dram bytes per launch of the dominant kernel from a committed ncu summary whose launch size matches this run
    (profiles/*_ncu_traffic.json, written by tools/ncu_summarise.py from an `ncu --set full` capture)."""
    import glob
    best = None
    for p in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_traffic.json"))):
        try:
            d = json.load(open(p))
        except Exception:
            continue
        for e in d.get("kernels", []):
            if e.get("kernel", "").startswith(kernel_prefix) and e.get("frames_per_launch") == frames_per_launch \
                    and e.get("volume_size", 64) == V:
                best = (e, os.path.relpath(p, ROOT))
    return best


def roofline_block(kern, tc_burst, tc_sust, peak_src, V, ms_step, B):
    v2v = kern["v2v"]
    fam = v2v["families"]
    c32 = fam["conv3_32_32_full_res"]
    n = v2v["chunk_frames"]
    launch_ms = c32["ms_per_frame"] * n / max(c32["launches"], 1)
    traffic, traffic_src = None, None
    hit = ncu_traffic("conv_march_kernel<2, 0, 2, 1>", n, V)     # the plain 32 -> 32 instantiation (6 of the 9 launches)
    if hit:
        traffic = hit[0]["dram_bytes_read"] + hit[0]["dram_bytes_write"]
        traffic_src = hit[1]
    stage_fl = v2v["conv_flops_per_frame"]
    return {"kernel": "conv_march_kernel (tcgen05 x-marching banded implicit-GEMM Conv3d 3x3x3 32->32 at full resolution, "
                      f"N=96 MMAs into a ring of TMEM slots, resident weights; {c32['launches']} launches per {n}-frame chunk)",
            "bound": "tensor", "achieved": c32["tflops"], "peak": tc_burst, "unit": "TFLOP/s",
            "frac": c32["tflops"] / tc_burst,
            "peak_kind": "bf16_tflops (burst): the durations are per-launch CUDA events in a ~20 ms profiling pass after idle",
            "frac_of_sustained_peak": c32["tflops"] / tc_sust, "sustained_peak": tc_sust,
            "traffic": traffic, "traffic_source": traffic_src,
            "algorithmic_bytes_per_launch": 2 * 32 * V ** 3 * 2 * n,
            "peak_source": peak_src,
            "how": f"algorithmic 2*32*32*27*{V}^3 = {2 * 32 * 32 * 27 * V ** 3 / 1e9:.2f} GFLOP per frame x {n} frames per launch "
                   "/ mean CUDA-event duration of those launches on the launching stream (sceneego_v2v_run_profile)",
            "launch_ms": launch_ms,
            "share_of_step": c32["ms_per_frame"] * B / ms_step,
            "stem": {"kernel": "stem kernel (7x7x7 Conv3d 33->16)", "achieved": fam["stem7_33_16"]["tflops"],
                     "frac": fam["stem7_33_16"]["tflops"] / tc_burst,
                     "share_of_step": fam["stem7_33_16"]["ms_per_frame"] * B / ms_step},
            "all_tensor_convs": {"achieved": stage_fl / (v2v["conv_ms_per_frame"] * 1e-3) / 1e12,
                                 "frac": stage_fl / (v2v["conv_ms_per_frame"] * 1e-3) / 1e12 / tc_burst,
                                 "how": "algorithmic FLOPs of every tcgen05 conv of V2V / sum of their durations"},
            "whole_step": {"achieved": stage_fl * B / (ms_step * 1e-3) / 1e12,
                           "frac_of_sustained_peak": stage_fl * B / (ms_step * 1e-3) / 1e12 / tc_sust,
                           "how": "V2V algorithmic FLOPs x frames / ms_per_step of the timed region (seconds long: sustained peak)"}}


def stage_kernel_timings(net, feat_d, depth_d, B, args, V, hbm_peak, tc_peak):
    """Time each kernel of the stage alone with CUDA events (after warm-up, L2 flushed) and relate it to its
    algorithmic bytes / FLOPs; every entry carries its roofline fraction (`frac`) against the burst peak."""
    import torch
    from sceneego_b200 import _lib
    vn = net.volume_net
    pg = vn.program(V, min(vn.max_chunk, B), feat_d.device)
    conv = net.process_features[0]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=feat_d.device)

    def timed(fn, reps=5):
        ts = []
        for _ in range(reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ts.sort()
        return ts[len(ts) // 2]

    out = {}
    n = min(pg.chunk, B)
    feat32 = _lib.feature_conv1x1(feat_d[:n], conv.weight, conv.bias)
    grid = net.grid_coord_proj_batch[0].reshape(-1, 2).contiguous()
    in_buf = pg.buffers[pg.in_buf]
    logits = torch.empty(n, J, V, V, V, dtype=torch.float32, device=feat_d.device)
    N = V ** 3

    def rec(name, ms, bytes_per_frame, note, bound="hbm"):
        gbs = bytes_per_frame * n / (ms * 1e-3) / 1e9
        out[name] = {"ms_per_frame": ms / n, "algorithmic_MB_per_frame": bytes_per_frame / 1e6, "GB_per_s": gbs,
                     "frac": gbs / hbm_peak, "bound": bound, "note": note}

    ms = timed(lambda: _lib.feature_conv1x1(feat_d[:n], conv.weight, conv.bias))
    rec("feature_conv1x1", ms, 256 * 64 * 64 * 4 + 64 * 64 * 32 * 4, "read (256,64,64) f32 + write (64,64,32) f32")
    ms = timed(lambda: _lib.unproject(feat32, grid, None, V, 2.0, 1024, 1280, None, in_buf, pg.lay_in,
                                      extra_zero_planes=pg.extra_zero_planes))
    rec("unproject", ms, 64 * 64 * 32 * 4 + N * 32 * 2 + N * 16 * pg.extra_zero_planes + N * 8,
        "read 0.524 MB features + the grid table, write 32 bf16 channels" +
        (" + the cleared occupancy plane" if pg.extra_zero_planes else ""))
    d = depth_d[:n]
    if pg.zwin:
        # lift()'s path for the marching stem: one store per pixel into the program's plain f32 grid, then one pass
        # that builds the whole z-window occupancy plane from it and re-zeroes the grid
        scratch = pg.occ_scratch[:n]
        ms = timed(lambda: _lib.voxelize_depth(d, net._ray_dev, 1024, 1280, V, 2.0, scratch, None, pg.lay_in, channel=32))
        rec("voxelize", ms, 1024 * 1280 * 4,
            "read (1024,1280) f32 depth; ray table (31.5 MB) shared by all frames; sparse f32 scatter; bound by fp64 instruction issue, not HBM")
        ms = timed(lambda: _lib.occ_expand_zwin(scratch, in_buf, pg.lay_in, 32))
        rec("occ_expand_zwin", ms, N * 4 + N * 16, "read the (V,V,V) f32 grid, write the z-window occupancy plane (16 B per voxel)")
    else:
        ms = timed(lambda: _lib.voxelize_depth(d, net._ray_dev, 1024, 1280, V, 2.0, None, in_buf, pg.lay_in, channel=32))
        rec("voxelize", ms, 1024 * 1280 * 4,
            "read (1024,1280) f32 depth; ray table (31.5 MB) shared by all frames; sparse bf16 scatter")
    vn.profile_chunk(pg, n, logits)     # warm-up
    prof = vn.profile_chunk(pg, n, logits)
    conv_ms = sum(ms for m, ms in prof if m["kind"] == "conv")
    conv_fl = sum(m["flops"] for m, ms in prof if m["kind"] == "conv")
    other_ms = sum(ms for m, ms in prof if m["kind"] != "conv")

    def mem_bytes(m):
        s = m["side"]
        if m["kind"] == "pool":
            return m["cin"] * (s ** 3 + (s // 2) ** 3) * 2
        if m["kind"] == "deconv":
            return m["cin"] * s ** 3 * 2 + 2 * m["cout"] * (2 * s) ** 3 * 2
        if m["kind"] == "tail":
            return s ** 3 * (32 * 2 + m["cout"] * 4)
        return None
    table = []
    for i, (m, ms) in enumerate(prof):
        e = {"op": i, "kind": m["kind"], "cin": m["cin"], "cout": m["cout"], "k": m["k"], "side": m["side"],
             "ms_per_frame": ms / n}
        if m["flops"] and m["kind"] == "conv":
            e["tflops"] = m["flops"] * n / (ms * 1e-3) / 1e12
            e["frac"] = e["tflops"] / tc_peak
        mb = mem_bytes(m)
        if mb:
            e["GB_per_s"] = mb * n / (ms * 1e-3) / 1e9
            e["frac"] = e["GB_per_s"] / hbm_peak
        table.append(e)

    def family(pred, bound="tensor"):
        sel = [(m, ms) for m, ms in prof if pred(m)]
        t = sum(ms for _, ms in sel)
        f = sum(m["flops"] for m, _ in sel)
        r = {"launches": len(sel), "ms_per_frame": t / n, "flops_per_frame": f,
             "tflops": f * n / (t * 1e-3) / 1e12 if t else 0.0, "bound": bound}
        if bound == "tensor":
            r["frac"] = r["tflops"] / tc_peak
        else:
            by = sum(mem_bytes(m) or 0 for m, _ in sel)
            r["algorithmic_MB_per_frame"] = by / 1e6
            r["GB_per_s"] = by * n / (t * 1e-3) / 1e9 if t else 0.0
            r["frac"] = r["GB_per_s"] / hbm_peak
        return r
    full = lambda m: m["kind"] == "conv" and m["k"] == 3 and m["cin"] == 32 and m["cout"] == 32 and m["side"] == V  # noqa: E731
    fams = {"conv3_32_32_full_res": family(full),
            "stem7_33_16": family(lambda m: m["kind"] == "conv" and m["k"] == 7),
            "other_tensor_convs": family(lambda m: m["kind"] == "conv" and m["k"] != 7 and not full(m)),
            "tail_1x1_fused": family(lambda m: m["kind"] == "tail", "hbm"),
            "deconv": family(lambda m: m["kind"] == "deconv", "hbm"),
            "maxpool": family(lambda m: m["kind"] == "pool", "hbm")}
    out["v2v"] = {"conv_ms_per_frame": conv_ms / n, "conv_flops_per_frame": conv_fl, "pool_deconv_tail_ms_per_frame": other_ms / n,
                  "bound": "tensor", "launches_per_chunk": len(prof), "chunk_frames": n, "families": fams,
                  "peaks": {"hbm_GB_per_s": hbm_peak, "bf16_TFLOP_per_s_burst": tc_peak}}
    if args.profile_ops:
        os.makedirs(os.path.dirname(os.path.abspath(args.profile_ops)), exist_ok=True)
        json.dump(table, open(args.profile_ops, "w"), indent=1)
    ms = timed(lambda: _lib.softargmax3d(logits, 1.0, True, net._axis, None, False))
    rec("softargmax", ms, J * N * 4, f"read ({J},{V},{V},{V}) f32 logits once (online softmax)")
    ms_full = timed(lambda: _lib.softargmax3d(logits, 1.0, True, net._axis, None, True))
    rec("softmax_volume_write", max(ms_full - ms, 1e-6), 2 * J * N * 4,
        "output #3 of the reference forward: read logits again + write the softmaxed volume f32")
    ms = timed(lambda: _lib.features_upsample_pad(feat32, 1024, 128))
    rec("features_upsample_pad", ms, 32 * 1024 * 1280 * 4 + 64 * 64 * 32 * 4,
        "output #2 of the reference forward: write (32,1024,1280) f32")
    return out


if __name__ == "__main__":
    a = parse()
    os.environ["SCENEEGO_ACT_DTYPE"] = a.act_dtype          # read by sceneego_b200._lib when the library is first loaded
    if a.impl == "reference":
        reference_arm(a)
    elif a.impl == "reference-gpu":
        reference_gpu_arm(a)
    else:
        ours_arm(a)
