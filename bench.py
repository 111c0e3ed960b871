#!/usr/bin/env python
"""bench.py -- headline benchmark of the MoreFusion volumetric-pose hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this framework
    python bench.py --impl reference --gpus N --steps K ...  # reference algorithm on host CPU cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's poses

Metric (BASELINE.json): objects/sec, volumetric pose (32^3).  Workload at every N:
BASELINE config[1] "singleview_3d inference, 32^3 occupancy 3D-CNN, batch=8 objects" -- one
step = one pass of the hot path (per-point MLP -> average_voxelization_3d 32^3 -> occupancy
stencils -> conv3/conv4 -> trilinear gathers -> 3 pose heads -> per-point poses) over a batch
of 8 synthetic YCB-shaped objects x 1000 points per rank (weak scaling: objects are
independent, no data-path collective; SURVEY.md 8e).  The 2-D ResNet18/PSPNet extractor is the
adjacent "next" row (SURVEY.md 8f-1): its 32-channel per-point output is the synthetic input.

Printed JSON (one line, rank 0): value = device-resident throughput; e2e = same metric through
the public Runner API with pinned HOST buffers in and out (H2D + D2H inside the timed region);
roofline = conv3 tcgen05 implicit GEMM (dense algorithmic FLOPs / CUDA-event duration measured
inside the timed steps) against the measured bf16 peak; cpu_baseline = the oracle port of the
same path timed on this box's host cores on a bounded sample.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

B_PER_RANK = 8
P = 1000
METRIC = "objects/sec volumetric pose (32^3)"
WORKLOAD = "singleview_3d inference hot path: 3D-CNN over 32^3 grid, batch=8 objects x 1000 pts per GPU"
CONV3_FLOPS_PER_OBJECT = 2.0 * 4096 * 256 * (160 * 64)     # SURVEY.md 8d: 21.47 GFLOP


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(bf16=d["bf16_tflops"], bf16_sustained=d["bf16_tflops_sustained"],
                    hbm=d["hbm_gbs"], source="measured (MEASURED_PEAKS.json)")
    return dict(bf16=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "50", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except Exception:
                continue
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for nm, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), samples=len(sm),
                    reasons=sorted(reasons))


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        backend = "nccl" if torch.cuda.is_available() else "gloo"
        if torch.cuda.is_available():
            torch.cuda.set_device(local)
        if backend == "nccl":
            dist.init_process_group(backend, device_id=torch.device("cuda", local))
        else:
            dist.init_process_group(backend)
    return rank, world, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()


def max_over_ranks(x, world, device):
    if world == 1:
        return x
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


# ------------------------------------------------------------------ reference arm / cpu baseline
def cpu_port_step(weights, batch, n_obj):
    from oracle import cnn as ocnn
    sub = {k: v[:n_obj] for k, v in batch.items()}
    t0 = time.perf_counter()
    ocnn.forward(weights, n_fg_class=21, bf16=False, **sub)
    return time.perf_counter() - t0


def pick_threads(weights, batch):
    """torch-CPU convolutions on small 3-D grids do not scale to every core of a large host
    (oversubscription makes 128 threads slower than 16): time one object at a few thread counts
    and use the fastest, reporting the number actually used."""
    n = os.cpu_count() or 1
    best_t, best = 1, float("inf")
    for t in sorted({min(8, n), min(16, n), min(32, n), min(64, n), n}):
        torch.set_num_threads(t)
        cpu_port_step(weights, batch, 1)
        dt = cpu_port_step(weights, batch, 1)
        if dt < best:
            best_t, best = t, dt
    torch.set_num_threads(best_t)
    return best_t


def run_reference(args, rank, world):
    """The reference's algorithm for this path on the host CPU cores.  The reference's own code
    cannot run here (chainer/cupy absent, SURVEY.md 8c) so this is the oracle port
    (kind="port"): torch-CPU fp32 convs + the NumPy restatements of the reference kernels."""
    if rank != 0:
        return
    from morefusion_b200 import synthetic
    weights = synthetic.init_weights(21, seed=1)
    n_obj = 2                                       # bounded sample per step
    batch = synthetic.make_cnn_batch(B_PER_RANK, P, seed=0)
    threads = pick_threads(weights, batch)
    warm = [cpu_port_step(weights, batch, n_obj) for _ in range(max(args.warmup, 1))]
    if min(warm) * args.steps > 240.0:
        n_obj = 1                                   # keep the whole run within a few minutes
        cpu_port_step(weights, batch, n_obj)
    ts = [cpu_port_step(weights, batch, n_obj) for _ in range(args.steps)]
    total = sum(ts)
    value = n_obj * args.steps / total
    line = dict(
        impl="reference", metric=METRIC, value=value, unit="objects/s", n_gpus=args.gpus,
        steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * total / args.steps,
        higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
        config=dict(workload=WORKLOAD, sample=f"{n_obj} of the {B_PER_RANK} objects per step"),
        cpu_baseline=dict(value=value, unit="objects/s", cores=threads, kind="port",
                          host_cores=os.cpu_count(),
                          sample=f"{n_obj} objects x {args.steps} steps, torch-CPU fp32 + NumPy oracle"),
        e2e=dict(value=value, unit="objects/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
        gpu_launches=0)
    print(json.dumps(line), flush=True)



# ------------------------------------------------------------------ sub-records
def _graph_time_us(fn, flush, reps=20, warm=3):
    """Median CUDA-event time of a CUDA-graph replay of fn(), L2 flushed between replays."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(warm):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        keep = fn()
    for _ in range(warm):
        g.replay()
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); g.replay(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    del keep
    ts.sort()
    return ts[len(ts) // 2], ts[0]


def bench_avg_vox(dev, pk, flush):
    """average_voxelization_3d through the public operator at the model shape (B8 x P1000 x C144
    -> 32^3) and at BASELINE config 1 (P1024, C4): algorithmic bytes (SURVEY.md 8d) / time."""
    import morefusion_b200 as mf
    from morefusion_b200 import synthetic
    out = {}
    for tag, B, Pn, C in (("model_shape", 8, 1000, 144), ("config1_unit", 1, 1024, 4)):
        D = 32
        sb = synthetic.make_cnn_batch(B, Pn, seed=1)
        pts = torch.as_tensor(np.ascontiguousarray(sb["points"].transpose(0, 2, 1).reshape(B * Pn, 3)),
                              device=dev)
        vals = torch.randn(B * Pn, C, device=dev)
        bi = torch.arange(B, device=dev, dtype=torch.int32).repeat_interleave(Pn)
        us, mn = _graph_time_us(lambda: mf.functions.average_voxelization_3d(
            vals, pts, bi, batch_size=B, origin=(0, 0, 0), pitch=1.0, dimensions=(D, D, D)), flush)
        byts = 4 * (B * Pn * C + 4 * B * Pn) + 4 * (B * C * D ** 3 + B * D ** 3)
        out[tag] = dict(us=us, min_us=mn, algorithmic_bytes=byts, achieved_gbs=byts / us / 1e3,
                        frac_of_hbm_peak=byts / us / 1e3 / pk["hbm"])
    out.update(bound="hbm", peak_gbs=pk["hbm"], kernels="k_avg_prepass + k_avg_fused (gather + single-pass fill)",
               timed="CUDA-graph replay of the public operator, 192 MiB L2 flush between replays, median of 20")
    return out


def bench_icc(dev, pk, quick):
    """Fused ICC (BASELINE config 4): 8-object scene, 32^3 grids, 100 fused iterations; single
    scene latency and batched-scene throughput; stateless byte model of SURVEY.md 8d."""
    from morefusion_b200 import synthetic
    from morefusion_b200.contrib.iterative_collision_check_link import ICCBatch
    n_iter = 100
    scenes = [synthetic.make_icc_scene(N=8, seed=10 + i) for i in range(4)]

    def run(S, reps):
        batch = ICCBatch([scenes[i % 4] for i in range(S)], sdf_offset=0.02, device=dev)
        q0, t0 = batch.quaternion.clone(), batch.translation.clone()
        ts = []
        for _ in range(reps + 1):
            batch.quaternion.copy_(q0); batch.translation.copy_(t0)
            batch.adam_state.zero_(); batch.adam_t = 0
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); batch.refine(n_iter=n_iter); e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return min(ts[1:]), batch
    ms1, b1 = run(1, 2 if quick else 4)
    sc = scenes[0]
    n_pts = sum(p.shape[0] for p in sc["points"])
    bytes_iter = sum(16 * p.shape[0] + 2 * 4 * 32 ** 3 for p in sc["points"]) + 84 * 8
    out = dict(single_scene=dict(ms_100_iter=ms1, us_per_iter=ms1 * 1e3 / n_iter,
                                 scene_iter_per_s=n_iter / (ms1 * 1e-3)),
               objects=8, points_per_scene=n_pts, n_iter=n_iter,
               stateless_bytes_per_scene_iter=bytes_iter,
               pair_tests_per_scene_iter=8 * n_pts, bound="hbm (stateless-iteration model, SURVEY.md 8d)")
    best = 0.0
    for S in ((16, 74) if quick else (8, 16, 37, 74, 148)):
        ms, _ = run(S, 1 if quick else 2)
        rate = S * n_iter / (ms * 1e-3)
        out[f"batch_{S}"] = dict(ms=ms, scene_iter_per_s=rate)
        best = max(best, rate)
    out.update(best_scene_iter_per_s=best, achieved_gbs=best * bytes_iter / 1e9,
               frac_of_hbm_peak=best * bytes_iter / 1e9 / pk["hbm"],
               pair_tests_per_s=best * 8 * n_pts,
               note="working set is L2 resident; the stateless model charges every iteration the "
                    "points + both 32^3 grids once; candidate-key atomics <= 27 per in-range pair test")
    return out


def bench_mapping(dev, pk, quick):
    """Occupancy-grid producer (SURVEY.md 8f-3): per 640x480 frame, 8 instance scans + the
    background scan into the device hash map (MultiInstanceOctreeMapping.integrate), then the three
    32^3 grids of all 8 targets from one launch.  Inputs resident in HBM; CUDA events."""
    from morefusion_b200 import synthetic
    from morefusion_b200.contrib import MultiInstanceOctreeMapping
    n_frames = 3 if quick else 6
    frames = []
    for i in range(n_frames):
        pcd, label, _, pitches = synthetic.make_depth_frame(seed=i)
        frames.append((torch.as_tensor(pcd, device=dev), torch.as_tensor(label, device=dev)))
    ids = sorted(i for i in pitches if i != 0) + [0]          # foreground instances, then background
    masks = [[(lab == ins) for ins in ids] for _, lab in frames]
    m = MultiInstanceOctreeMapping(device=dev)
    for ins in ids:
        m.initialize(ins, pitch=pitches[ins])
    ts = []
    for f, (pcd, lab) in enumerate(frames):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for k, ins in enumerate(ids):
            m.integrate(ins, masks[f][k], pcd)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    tids = [i for i in ids if i != 0]
    pcd0, lab0 = frames[0][0].cpu().numpy(), frames[0][1].cpu().numpy()
    origins = [np.nanmedian(pcd0[lab0 == t], axis=0) - 15.5 * pitches[t] for t in tids]
    q = []
    for _ in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g = m.get_target_grids_batch(tids, dimensions=(32, 32, 32), pitches=[pitches[t] for t in tids],
                                     origins=origins)
        e1.record()
        torch.cuda.synchronize()
        q.append(e0.elapsed_time(e1))
    steady = sorted(ts[1:])[len(ts[1:]) // 2]
    # the same frames as ONE labelled scan each (two launches per frame)
    m2 = MultiInstanceOctreeMapping(device=dev)
    for ins in ids:
        m2.initialize(ins, pitch=pitches[ins])
    labs = [lab.to(torch.int32) for _, lab in frames]
    tl = []
    for f, (pcd, _) in enumerate(frames):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        m2.integrate_labels(labs[f], pcd)
        e1.record()
        torch.cuda.synchronize()
        tl.append(e0.elapsed_time(e1))
    steady_l = sorted(tl[1:])[len(tl[1:]) // 2]
    assert m2.n_cells() == m.n_cells()
    n_valid = int((~torch.isnan(frames[-1][0]).any(-1)).sum().item())
    out = dict(frame="640x480, 8 instances (class pitch) + background (1 cm), OctoMap sensor model",
               ms_per_frame_labelled_scan=steady_l, first_frame_ms_labelled=tl[0],
               rays_per_s=n_valid / (steady_l * 1e-3),
               ms_per_frame_9_integrate_calls=steady, first_frame_ms=ts[0], rays_per_frame=n_valid,
               map_cells=m.n_cells(), table_slots=m._cap,
               query_ms_8_targets_32cubed=min(q), occupied_target_voxels=int((g[0] > 0).sum().item()),
               lookups_per_query=8 * 32 ** 3 * len(ids),
               kernels="k_map_scan_hits + k_map_scan_free per scan; k_map_query_grids per query",
               bound="L2 / atomic latency (random probes of a hash table; not a streaming kernel)",
               timed="CUDA events around integrate_labels() of a frame / around the 9 integrate() calls "
                     "of a frame (median of frames 2..n) and around get_target_grids_batch (min of 4); "
                     "inputs resident in HBM")
    # CPU side: the oracle's restatement of the OctoMap calls on a bounded sample of rays
    import time
    from oracle import octomap as oc
    tree = oc.OcTree(pitches[0])
    sample = pcd0[lab0 == 0]
    sample = sample[~np.isnan(sample).any(1)][:: max(1, len(sample) // 400)]
    t0 = time.time()
    tree.insertPointCloud(sample, origin=np.zeros(3))
    dt = time.time() - t0
    out["cpu_port"] = dict(rays_per_s=len(sample) / dt, rays=len(sample), cores=1, kind="port",
                           sample="oracle/octomap.py insertPointCloud on a strided sample of the "
                                  "background scan (pure Python; OctoMap itself is not in the image)")
    return out


def bench_chain(dev, model, runner, rank, world, quick):
    """BASELINE config 5: per-frame chain voxelise -> 3D-CNN -> ICC through HOST buffers.  A frame
    = 8 objects: H2D of the frame's CNN inputs and of its two 32^3 grids per object, the CNN step
    (one CUDA graph), per-object best pose = argmax confidence, ICC refinement of the 8-object
    scene (30 fused iterations, the per-frame budget of evaluate.py:274 / the ROS node), D2H of
    the refined poses.  Frames are sharded round-robin over the ranks (no collective)."""
    from morefusion_b200 import synthetic
    from morefusion_b200.contrib.iterative_collision_check_link import ICCBatch
    n_frames = 8 if quick else 32
    icc_iter = 30
    scenes = [synthetic.make_icc_scene(N=8, seed=20 + i) for i in range(2)]
    batches = [ICCBatch([sc], sdf_offset=0.02, device=dev) for sc in scenes]
    inits = [(b.quaternion.clone(), b.translation.clone()) for b in batches]
    grids = []          # pinned host copies of the per-frame grids (grid_target | gne)
    for sc in scenes:
        h = torch.from_numpy(np.stack([sc["grid_target"], sc["grid_nontarget_empty"]]).astype(np.float32))
        grids.append(h.pin_memory())
    cnn_blobs = []
    for i in range(2):
        runner.load_host(synthetic.make_cnn_batch(B_PER_RANK, P, seed=500 + i))
        blob, _ = runner.new_host_blob()
        blob.copy_(runner.host_in_blob)
        cnn_blobs.append(blob)
    out_pose = torch.empty((8, 14), dtype=torch.float32).pin_memory()
    torch.cuda.synchronize()

    def frame(i):
        k = i % 2
        b = batches[k]
        runner.upload(cnn_blobs[k])                                   # H2D CNN inputs
        b.prob.grid_target.copy_(grids[k][0].reshape(b.prob.grid_target.shape), non_blocking=True)
        b.prob.gne.copy_(grids[k][1].reshape(b.prob.gne.shape), non_blocking=True)
        runner.run()                                                  # voxelise -> 3D-CNN -> poses
        best = runner.out["conf"].argmax(dim=1)                       # [B]
        ar = torch.arange(B_PER_RANK, device=dev)
        cnn_pose = torch.cat([runner.out["rot"][ar, best], runner.out["trans"][ar, best]], 1)
        # random-init weights give meaningless CNN poses: ICC starts from the scene's perturbed
        # ground truth (same sizes, same work); the CNN pose is still produced and returned
        b.quaternion.copy_(inits[k][0]); b.translation.copy_(inits[k][1])
        b.adam_state.zero_(); b.adam_t = 0
        b.refine(n_iter=icc_iter)
        dev_pose = torch.cat([cnn_pose, b.quaternion, b.translation], 1)   # [8, 7 + 7]
        out_pose.copy_(dev_pose, non_blocking=True)                   # D2H

    for i in range(2):
        frame(i)
    torch.cuda.synchronize()
    my = list(range(rank, n_frames * world, world))
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in my:
        frame(i)
    e1.record()
    torch.cuda.synchronize()
    barrier(world)
    ms = max_over_ranks(e0.elapsed_time(e1), world, dev)
    h2d = cnn_blobs[0].numel() + grids[0].numel() * 4

    # ---- throughput mode: F frames in flight share ONE ICC launch (their scenes are independent
    # groups of the same persistent kernel): every frame still goes H2D -> CNN -> pose -> ICC -> D2H
    # through host buffers; what changes is that the refinement of F frames runs together, which
    # is where the fused ICC kernel's throughput comes from (a single scene is barrier-bound).
    F = 4
    fb = ICCBatch([scenes[j % 2] for j in range(F)], sdf_offset=0.02, device=dev)
    fq0, ft0 = fb.quaternion.clone(), fb.translation.clone()
    out_pose_f = torch.empty((F * 8, 14), dtype=torch.float32).pin_memory()
    gt_rows = fb.prob.grid_target.reshape(F, -1)
    gne_rows = fb.prob.gne.reshape(F, -1)

    def frames(i0):
        cnn_poses = []
        for j in range(F):
            k = (i0 + j) % 2
            runner.upload(cnn_blobs[k])
            gt_rows[j].copy_(grids[k][0].reshape(-1), non_blocking=True)
            gne_rows[j].copy_(grids[k][1].reshape(-1), non_blocking=True)
            runner.run()
            best = runner.out["conf"].argmax(dim=1)
            ar = torch.arange(B_PER_RANK, device=dev)
            cnn_poses.append(torch.cat([runner.out["rot"][ar, best], runner.out["trans"][ar, best]], 1))
        fb.quaternion.copy_(fq0); fb.translation.copy_(ft0)
        fb.adam_state.zero_(); fb.adam_t = 0
        fb.refine(n_iter=icc_iter)
        dev_pose = torch.cat([torch.cat(cnn_poses), fb.quaternion, fb.translation], 1)
        out_pose_f.copy_(dev_pose, non_blocking=True)

    frames(0)
    torch.cuda.synchronize()
    n_groups = max(1, len(my) // F)
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for g in range(n_groups):
        frames(g * F)
    e1.record()
    torch.cuda.synchronize()
    barrier(world)
    ms_f = max_over_ranks(e0.elapsed_time(e1), world, dev)
    per_frame_f = ms_f / (n_groups * F)

    # ---- the same with the map front end in every frame (SURVEY.md 8f-2 / 8f-3): depth + instance
    # label H2D (2 x 1.2 MB), depth -> point image, labelled OctoMap scan into the persistent device
    # map, the 3 x 8 target grids, grid_nontarget_empty composed as the evaluation transform does
    # (train.py:50-54,92-105).  The synthetic generators are not ONE consistent scene: the map
    # stage runs on its own 640x480 frames and its grids are produced and combined every frame,
    # while the CNN / ICC consume the scene's precomputed grids (same sizes, same work).
    from morefusion_b200 import geometry as mgeo
    from morefusion_b200.contrib import MultiInstanceOctreeMapping
    fr = [synthetic.make_depth_frame(seed=40 + j) for j in range(2)]
    pitches = fr[0][3]
    ids = sorted(i for i in pitches if i != 0) + [0]
    mp = MultiInstanceOctreeMapping(device=dev)
    for ins in ids:
        mp.initialize(ins, pitch=pitches[ins])
    h_depth = [torch.from_numpy(np.ascontiguousarray(f[0][..., 2])).pin_memory() for f in fr]
    h_label = [torch.from_numpy(np.ascontiguousarray(f[1])).pin_memory() for f in fr]
    d_depth = torch.empty(tuple(h_depth[0].shape), dtype=torch.float32, device=dev)
    d_label = torch.empty(tuple(h_label[0].shape), dtype=torch.int32, device=dev)
    Hh, Ww = h_depth[0].shape
    tids = [i for i in ids if i != 0]
    t_orig = [np.nanmedian(fr[0][0][fr[0][1] == t], axis=0) - 15.5 * pitches[t] for t in tids]
    t_pit = [pitches[t] for t in tids]

    def frontend(i):
        k = i % 2
        d_depth.copy_(h_depth[k], non_blocking=True)
        d_label.copy_(h_label[k], non_blocking=True)
        pcd = mgeo.pointcloud_from_depth(d_depth, fx=600.0, fy=600.0, cx=Ww / 2, cy=Hh / 2)
        mp.integrate_labels(d_label, pcd)
        gt, gn, ge = mp.get_target_grids_batch(tids, dimensions=(32, 32, 32), pitches=t_pit, origins=t_orig)
        tgt = gt > 0.5
        return ((gn > 0.5) ^ tgt) | ((ge > 0.5) ^ tgt)               # grid_nontarget_empty [8,32,32,32]

    def frames_full(i0):
        keep = [frontend(i0 + j) for j in range(F)]
        frames(i0)
        return keep

    frames_full(0)
    torch.cuda.synchronize()
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for g in range(n_groups):
        frames_full(g * F)
    e1.record()
    torch.cuda.synchronize()
    barrier(world)
    ms_full = max_over_ranks(e0.elapsed_time(e1), world, dev)
    with_map = dict(value=n_groups * F * world * 8 / (ms_full * 1e-3), ms_per_frame=ms_full / (n_groups * F),
                    extra_h2d_bytes_per_frame=int(h_depth[0].numel() * 4 + h_label[0].numel() * 4),
                    map_cells=mp.n_cells(),
                    stages="depth+label H2D -> k_pointcloud_from_depth -> k_map_scan_hits/free (all "
                           "instances) -> k_map_query_grids (8 targets) -> gne -> [CNN -> ICC as above]")
    return dict(metric="objects/sec per-frame chain voxelise->3D-CNN->ICC",
                value=n_groups * F * world * 8 / (ms_f * 1e-3), unit="objects/s",
                frames=n_groups * F * world, objects_per_frame=8, icc_iterations=icc_iter,
                ms_per_frame=per_frame_f, frames_per_icc_launch=F,
                latency_of_a_frame_group_ms=ms_f / n_groups,
                single_frame_mode=dict(value=len(my) * world * 8 / (ms * 1e-3), ms_per_frame=ms / len(my),
                                       frames=len(my) * world, frames_per_icc_launch=1),
                with_map_frontend=with_map,
                h2d_bytes_per_frame=int(h2d), d2h_bytes_per_frame=int(out_pose.numel() * 4),
                n_gpus=world,
                timed="CUDA events around the frame loop incl. H2D/D2H, max over ranks; `value` = "
                      f"{F} frames in flight per ICC launch (each frame: H2D, CNN graph, pose select, "
                      "then one fused 30-iteration ICC launch over the group's scenes, D2H); "
                      "single_frame_mode = one frame per ICC launch (lowest latency)")


# ------------------------------------------------------------------ our arm
def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy, so that two builds run with the same arguments
    (hence the same seeded inputs) can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args, rank, world, local):
    assert torch.cuda.is_available(), "bench.py (our arm) needs a CUDA device; no CPU fallback"
    import morefusion_b200 as mf
    from morefusion_b200 import synthetic
    from morefusion_b200.contrib.singleview_3d.models import Model
    mf.config.check_nan = False
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    pk = peaks()

    weights = synthetic.init_weights(21, seed=1)
    model = Model(n_fg_class=21, with_occupancy=True).to(dev).load_reference_weights(weights)
    runner = model.make_runner(B_PER_RANK, P, dev, graph=not args.no_graph)
    n_sets = 4                                       # rotate input batches
    batches = [synthetic.make_cnn_batch(B_PER_RANK, P, seed=100 * rank + i) for i in range(n_sets)]
    dev_sets = []
    for b in batches:
        runner.load_host(b)
        torch.cuda.synchronize()
        dev_sets.append({k: v.clone() for k, v in runner.st.items()})
    pinned_blobs = []                                 # one pinned host blob per rotating batch
    for b in batches:
        runner.load_host(b)
        blob, _ = runner.new_host_blob()
        blob.copy_(runner.host_in_blob)
        pinned_blobs.append(blob)
    torch.cuda.synchronize()
    flush = torch.empty(192 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def set_inputs(i):
        for k, v in dev_sets[i % n_sets].items():
            runner.st[k].copy_(v)

    # ---- device-resident throughput
    for i in range(max(args.warmup, 3)):
        set_inputs(i)
        runner.run()
    torch.cuda.synchronize()
    K = args.steps
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    cev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    sampler = ClockSampler(local)
    barrier(world)
    torch.cuda.synchronize()
    if rank == 0:
        sampler.start()
    n0 = model.n_launches
    for i in range(K):
        set_inputs(i)
        flush.zero_()                     # L2 flush between timed iterations (untimed)
        ev[i][0].record()
        runner.run()                      # whole step = one captured graph
        ev[i][1].record()
    torch.cuda.synchronize()
    barrier(world)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # the poses of the last timed step; later passes overwrite runner.out
        dump_outputs(args.dump_outputs, runner.out)
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = max_over_ranks(sum(step_ms), world, dev)
    # second pass over the same K steps with the step split into three graphs so that the
    # dominant kernel (conv3) is bracketed by events on the launching stream (roofline)
    for i in range(K):
        set_inputs(i)
        flush.zero_()
        runner.set_events(*cev[i])
        runner.run()
    torch.cuda.synchronize()
    conv3_ms = [a.elapsed_time(b) for a, b in cev]
    launches = runner.launches_per_step * K if runner.graphs is not None else model.n_launches - n0
    runner.ev = None
    value = world * B_PER_RANK * K / (total_ms * 1e-3)

    # ---- end to end: pinned host buffers in, pinned host poses out, copies inside the timing
    # Runner.run_e2e(): ONE graph launch = H2D of the small inputs + occupancy grid, H2D of `values`
    # under the occupancy branch, the step, poses written by the last kernel into pinned host memory.
    for i in range(3):
        runner.host_in_blob.copy_(pinned_blobs[i % n_sets]); runner.run_e2e()
        torch.cuda.synchronize()
    ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    barrier(world)
    torch.cuda.synchronize()
    for i in range(K):
        # the caller fills the runner's pinned staging blob (host memcpy, before the timed region;
        # the previous step has completed)
        runner.host_in_blob.copy_(pinned_blobs[i % n_sets])
        flush.zero_()
        ev2[i][0].record()
        runner.run_e2e()                                       # H2D + step + D2H inside the graph
        ev2[i][1].record()
        torch.cuda.synchronize()
    barrier(world)
    e2e_ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in ev2), world, dev)
    e2e_value = world * B_PER_RANK * K / (e2e_ms * 1e-3)

    # ---- per-frame chain (BASELINE config 5): frames sharded over ALL ranks, so every rank runs it
    records = {}
    try:
        records["chain"] = bench_chain(dev, model, runner, rank, world, args.quick)
    except Exception as e:
        records["chain"] = dict(error=f"{type(e).__name__}: {e}")
    # ---- training step (BASELINE config 3): data parallel, NCCL gradient all-reduce at N > 1
    try:
        tl = train_bench(rank, world, local, 6 if args.quick else 12, 3)
        records["train"] = {k: tl[k] for k in ("metric", "value", "unit", "ms_per_step", "scaling",
                                                 "n_gpus", "steps", "config", "gemms", "loss_last")}
    except Exception as e:
        records["train"] = dict(error=f"{type(e).__name__}: {e}")
    if rank != 0:
        return
    # ---- roofline of the dominant kernel (conv3 tcgen05 implicit GEMM)
    conv3_avg_ms = float(np.mean(conv3_ms))
    flops = CONV3_FLOPS_PER_OBJECT * B_PER_RANK
    achieved = flops / (conv3_avg_ms * 1e-3) / 1e12
    traffic = None
    prof = os.path.join(ROOT, "profiles", "r02_conv3_pair_ncu_summary.json")
    if os.path.exists(prof):
        try:
            traffic = json.load(open(prof)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    roof = dict(bound="tensor", kernel="k_gemm_tc_pair<6> (conv3 160->256 k4 s2, implicit GEMM M=32768 N=256 K=10240, cta_group::2, stream-K)",
                achieved=achieved, peak=pk["bf16"], unit="TFLOP/s",
                frac=achieved / pk["bf16"], frac_of_sustained_peak=achieved / pk["bf16_sustained"],
                peak_source=pk["source"] + ", burst figure (0.14 ms kernel between L2 flushes); "
                            "sustained figure kept as frac_of_sustained_peak",
                avg_launch_us=conv3_avg_ms * 1e3, share_of_step=conv3_avg_ms / float(np.mean(step_ms)),
                timed="CUDA events around the conv3 launch in a second pass over the same K steps "
                      "(step split into 3 graphs); `value` times the one-graph step",
                traffic=traffic,
                traffic_source="profile constant: dram__bytes_read+write per launch from the committed "
                               "ncu --set full capture (profiles/r02_conv3_pair_ncu_summary.json), not measured in this run")
    # ---- the two HBM-bound targets north_star names + the per-frame chain (BASELINE configs 1/4/5)
    for name, fn in (("avg_vox", lambda: bench_avg_vox(dev, pk, flush)),
                     ("icc", lambda: bench_icc(dev, pk, args.quick)),
                     ("mapping", lambda: bench_mapping(dev, pk, args.quick))):
        try:
            records[name] = fn()
        except Exception as e:      # a sub-record must not take the headline line down
            records[name] = dict(error=f"{type(e).__name__}: {e}")
    # ---- CPU baseline: oracle port on the host cores, bounded sample
    if world == 1:
        threads = pick_threads(weights, batches[0])
        n_obj = 2
        reps, t_cpu = 0, 0.0
        while t_cpu < 8.0 and reps < 6:
            t_cpu += cpu_port_step(weights, batches[0], n_obj)
            reps += 1
        cpu = dict(value=n_obj * reps / t_cpu, unit="objects/s", cores=threads, host_cores=os.cpu_count(),
                   kind="port",
                   sample=f"{n_obj} objects x {reps} passes of the oracle port (torch-CPU fp32 convs + NumPy kernels)")
    else:       # the host-core baseline is a 1-GPU figure: N ranks would time each other's threads
        cpu = dict(value=None, unit="objects/s", kind="port", sample="measured at N=1 only (see the 1-GPU line)")
    line = dict(
        metric=METRIC, value=value, unit="objects/s", n_gpus=world, steps=K, warmup=max(args.warmup, 3),
        ms_per_step=total_ms / K, higher_is_better=True, scaling="weak", vs_baseline=None,
        dtype="bf16", data="synthetic",
        config=dict(workload=WORKLOAD, objects_per_gpu_per_step=B_PER_RANK, points_per_object=P,
                    voxel_dim=32, n_fg_class=21, parallelism=f"objects sharded over {world} GPU(s), no collective",
                    cuda_graph=runner.graphs is not None,
                    l2="192 MiB buffer written between timed iterations (untimed); 4 rotating input sets"),
        e2e=dict(value=e2e_value, unit="objects/s", h2d_bytes_per_step=runner.h2d_bytes,
                 d2h_bytes_per_step=runner.d2h_bytes, ms_per_step=e2e_ms / K,
                 timed="CUDA events around Runner.run_e2e(): one graph launch = H2D copy of the small inputs "
                       "+ occupancy grid, H2D copy of `values` while the occupancy branch runs, the step, "
                       "the last kernel writing the poses in place into the pinned host output (UVA); "
                       "every input / output byte crosses PCIe inside the timed region"),
        gpu_launches=int(launches), clocks=clocks, roofline=roof, cpu_baseline=cpu, **records)
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ training arm (BASELINE config 3)
def train_bench(rank, world, local, steps, warmup):
    """singleview_3d training step, data parallel (train.py:229-233,342-344,361): global batch 16
    split over the ranks, forward + CUDA backward of the 3-D section, bucketed NCCL gradient
    all-reduce overlapped with the backward, fused 1/world + Chainer-Adam update.  Per-point
    features stand in for the 2-D extractor's output (as in the inference line)."""
    assert torch.cuda.is_available(), "bench.py --mode train needs a CUDA device"
    import morefusion_b200 as mf
    from morefusion_b200 import _lib, synthetic
    from morefusion_b200.contrib.singleview_3d.models import Model, training
    mf.config.check_nan = False
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    pk = peaks()
    G = 16
    assert G % world == 0
    Bl = G // world
    model = Model(n_fg_class=21, with_occupancy=True).to(dev).load_reference_weights(
        synthetic.init_weights(21, seed=1)).train()
    tr = training.Trainer(model, alpha=1e-4)
    rs = np.random.RandomState(100 + rank)
    batches = []
    models = synthetic.SyntheticYCBModels()
    t = lambda x: torch.as_tensor(np.ascontiguousarray(x), device=dev)   # noqa: E731
    for i in range(2):
        b = synthetic.make_cnn_batch(Bl, P, seed=1000 * rank + i)
        q = rs.normal(size=(Bl, 4)).astype(np.float32)
        q /= np.linalg.norm(q, axis=1, keepdims=True)
        cam = b["points"] * b["pitch"][:, None, None] + b["origin"][:, :, None]
        batches.append(dict(dev={k: t(v) for k, v in b.items()}, class_id=b["class_id"],
                            q=t(q), tt=t(cam.mean(axis=2).astype(np.float32))))
    cur = {}

    def predict(**kw):
        d = cur["b"]["dev"]
        return training.forward_features_with_grad(
            model, class_id=cur["b"]["class_id"], values=d["values"], points=d["points"],
            pitch=d["pitch"], origin=d["origin"], grid_nontarget_empty=d["grid_nontarget_empty"])
    model.predict = predict

    def step(i):
        cur["b"] = batches[i % 2]
        return tr.step(class_id=cur["b"]["class_id"], rgb=None, pcd=None,
                       quaternion_true=cur["b"]["q"], translation_true=cur["b"]["tt"])
    for i in range(max(warmup, 3)):
        step(i)
    torch.cuda.synchronize()
    K = steps
    sampler = ClockSampler(local)
    barrier(world)
    torch.cuda.synchronize()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        loss = step(i)
    e1.record()
    torch.cuda.synchronize()
    barrier(world)
    clocks = sampler.stop() if rank == 0 else None
    ms = max_over_ranks(e0.elapsed_time(e1), world, dev)
    # ---- tensor-pipe fractions of the four conv gradient GEMMs (events around single launches)
    L = _lib.lib()
    tb = training._train_buffers(model, Bl, P, dev)
    buf = model._work_buffers(Bl, P, dev)
    tw = training._train_pack(model)

    def timed(fn, reps=5):
        fn()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts))
    ptr, s = _lib.ptr, _lib.stream
    gemms = {}
    for name, flops, fn in (
        ("conv3_wgrad", 2.0 * Bl * 4096 * 256 * 10240, lambda: L.mf_train_conv_wgrad(
            ptr(tb["dY3p"]), ptr(buf["x3"]), Bl, 16, 256, 1280, ptr(tb["gw3"]), 0, s())),
        ("conv3_dgrad", 2.0 * Bl * 4096 * 256 * 10240, lambda: L.mf_train_conv_dgrad(
            ptr(tb["dY3p"]), ptr(tw["conv3/Wd"]), Bl, 16, 256, 160, 2, ptr(tb["dx3"]), 160,
            Bl * 4096 * 160, s())),
        ("conv4_wgrad", 2.0 * Bl * 512 * 512 * 16384, lambda: L.mf_train_conv_wgrad(
            ptr(tb["dY4p"]), ptr(buf["x4"]), Bl, 8, 512, 2048, ptr(tb["gw4"]), 0, s())),
        ("conv4_dgrad", 2.0 * Bl * 512 * 512 * 16384, lambda: L.mf_train_conv_dgrad(
            ptr(tb["dY4p"]), ptr(tw["conv4/Wd"]), Bl, 8, 512, 256, 1, ptr(tb["dgrid3"]), 256, 0, s()))):
        t_ms = timed(fn)
        gemms[name] = dict(us=t_ms * 1e3, tflops=flops / (t_ms * 1e-3) / 1e12,
                           frac_of_bf16_burst_peak=flops / (t_ms * 1e-3) / 1e12 / pk["bf16"])
    model.flush_reports()
    n_params = int(tr.flat_p.numel())
    line = dict(
        metric="objects/sec training step, 3-D section of singleview_3d (global batch 16)",
        value=G * K / (ms * 1e-3), unit="objects/s", n_gpus=world, steps=K,
        warmup=max(warmup, 3), ms_per_step=ms / K, higher_is_better=True, scaling="strong",
        vs_baseline=None, dtype="bf16", data="synthetic", mode="train",
        config=dict(workload="singleview_3d training step: forward + backward of the 3-D section, "
                             "Chainer-Adam(1e-4), global batch 16 x 1000 pts",
                    per_gpu_batch=Bl, parallelism=f"dp{world}: fp32 gradient all-reduce over NCCL in "
                    f"{len(tr.buckets)} buckets overlapped with the backward, fused unscale + Adam",
                    parameters=n_params, allreduce_bytes_per_step=4 * n_params if world > 1 else 0,
                    l2="working set (activations + 124 MB of gradients) exceeds L2"),
        loss_last=float(loss.detach()), clocks=clocks, gemms=gemms,
        roofline=dict(bound="tensor", kernel="k_gemm_train<256,4> conv3 wgrad (MN-major implicit GEMM)",
                      achieved=gemms["conv3_wgrad"]["tflops"], peak=pk["bf16"], unit="TFLOP/s",
                      frac=gemms["conv3_wgrad"]["frac_of_bf16_burst_peak"], traffic=None),
        gpu_launches=None)
    del tr, model
    torch.cuda.empty_cache()
    return line


def run_train(args, rank, world, local):
    line = train_bench(rank, world, local, args.steps, args.warmup)
    if rank == 0:
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--quick", action="store_true", help="shorter sub-records (icc / chain)")
    ap.add_argument("--mode", default="infer", choices=["infer", "train"],
                    help="infer: BASELINE config 2 (headline); train: config 3 (data-parallel step)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the poses of the last timed step (rot, trans, conf of rank 0) "
                         "as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.mode != "infer"):
        ap.error("--dump-outputs applies to the inference arm (--impl ours --mode infer)")
    if args.impl == "reference":
        # host-CPU arm: rank 0 alone works; other ranks exit 0 without joining any group
        run_reference(args, int(os.environ.get("RANK", "0")), 1)
        return
    rank, world, local = dist_setup(args.gpus)
    try:
        if args.impl == "reference":
            run_reference(args, rank, world)
        elif args.mode == "train":
            run_train(args, rank, world, local)
        else:
            run_ours(args, rank, world, local)
    finally:
        if world > 1:
            import torch.distributed as dist
            if dist.is_initialized():
                dist.destroy_process_group()


if __name__ == "__main__":
    main()
