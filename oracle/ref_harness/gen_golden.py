#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the REFERENCE's own operator code.

TEST INFRASTRUCTURE ONLY.  Run in the dev container (needs /root/reference):

    python -m oracle.ref_harness.gen_golden

Every array named ``ref_*`` in a golden file was produced by reference code
executed through oracle/ref_harness/shim.py (``*_cpu`` = the reference's NumPy
``forward_cpu``/``backward_cpu``; ``*_gpu`` = its CuPy kernel source string run
serially on the CPU).  Inputs are seeded; nothing here reads the oracle except
``quaternion_from_matrix`` (a trimesh stand-in used only to initialise the ICC
link, see shim.install) and, for ``octree_mapping``, the OctoMap stand-in
(oracle/octomap.py: the library is absent, so the reference's own
``MultiInstanceOctreeMapping`` code runs on the restated ``OcTree``).
"""

import hashlib
import json
import os
import sys

import numpy as np

from . import shim

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
OUT = os.path.join(ROOT, "tests", "golden")
F32 = np.float32
# SHA-256 of every array the generator wrote, so that the committed fixtures can be checked
# against the reference's output where the reference itself is not available
DIGESTS = "reference_digests.json"
_WRITTEN = []


def _save(name, **kw):
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **kw)
    _WRITTEN.append(name + ".npz")
    print("wrote", path, os.path.getsize(path), "bytes")


def array_digest(a):
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def file_digests(path):
    with np.load(path) as z:
        return {k: array_digest(z[k]) for k in sorted(z.files)}


def _geo(name):
    return shim.ref_module("functions.geometry." + name)


# ---------------------------------------------------------------- voxelization
def voxelization_cases():
    """(name, values, points, batch_indices, intensities, B, origin, pitch, dims)."""
    cases = []
    rs = np.random.RandomState(0)
    # mirrors tests/functions_tests/geometry_tests/test_average_voxelization_3d.py:20-38
    P, C, B, D = 128, 4, 3, 32
    cases.append(dict(
        name="unit32", values=rs.uniform(-1, 1, (P, C)).astype(F32),
        points=rs.uniform(-1, 1, (P, 3)).astype(F32),
        batch_indices=rs.randint(0, B, P).astype(np.int32),
        intensities=rs.uniform(0, 1, P).astype(F32),
        B=B, origin=np.array([-1, -1, -1], F32), pitch=F32(2.0 / D), dims=(D, D, D)))
    # dense collisions + out-of-bounds + exact .5 ties (round half away vs half even)
    P, C, B = 600, 5, 2
    pts = rs.uniform(-0.2, 4.4, (P, 3)).astype(F32)
    pts[:100] = (np.floor(pts[:100]) + 0.5).astype(F32)       # exact ties at pitch=1
    pts[100:140] = rs.uniform(-3, 8, (40, 3)).astype(F32)     # many out of bounds
    cases.append(dict(
        name="ties_oob", values=rs.uniform(-1, 1, (P, C)).astype(F32), points=pts,
        batch_indices=rs.randint(0, B, P).astype(np.int32),
        intensities=rs.randint(0, 4, P).astype(F32),           # exact intensity ties
        B=B, origin=np.zeros(3, F32), pitch=F32(1.0), dims=(4, 5, 6)))
    return cases


def gen_voxelization():
    av = _geo("average_voxelization_3d")
    mv = _geo("max_voxelization_3d")
    for c in voxelization_cases():
        out = {k: v for k, v in c.items() if k != "name"}
        out["dims"] = np.array(c["dims"])
        gy = np.random.RandomState(1).uniform(
            -1, 1, (c["B"], c["values"].shape[1]) + c["dims"]).astype(F32)
        out["gy_seed"] = 1   # gy = RandomState(1).uniform(-1, 1, (B, C)+dims).astype(f32)
        for mode in ("cpu", "gpu"):
            shim.set_mode(mode)
            f = av.AverageVoxelization3D(
                batch_size=c["B"], origin=c["origin"], pitch=c["pitch"], dimensions=c["dims"])
            y = np.asarray(f(c["values"], c["points"], c["batch_indices"]))
            g = f.backward((c["values"], c["points"], c["batch_indices"]), (gy,))[0]
            out[f"ref_avg_matrix_{mode}"] = y
            out[f"ref_avg_counts_{mode}"] = np.asarray(f.counts)
            out[f"ref_avg_gvalues_{mode}"] = np.asarray(g)
            f = mv.MaxVoxelization3D(
                batch_size=c["B"], origin=c["origin"], pitch=c["pitch"], dimensions=c["dims"])
            y = np.asarray(f(c["values"], c["points"], c["batch_indices"], c["intensities"]))
            g = f.backward(
                (c["values"], c["points"], c["batch_indices"], c["intensities"]), (gy,))[0]
            out[f"ref_max_matrix_{mode}"] = y
            out[f"ref_max_indices_{mode}"] = np.asarray(f.indices)
            out[f"ref_max_gvalues_{mode}"] = np.asarray(g)
        _save("voxelization_" + c["name"], **out)


# ---------------------------------------------------------------- interpolate
def gen_interpolate():
    m = _geo("interpolate_voxel_grid")
    rs = np.random.RandomState(2)
    B, C, D, P = 3, 4, 16, 128
    vox = rs.uniform(-1, 1, (B, C, D, D, D)).astype(F32)
    pts = rs.uniform(0, D - 1, (P, 3)).astype(F32)
    pts[:8] = rs.uniform(-1.5, 0, (8, 3)).astype(F32)         # negative: (int) vs floor
    pts[8:16] = rs.uniform(D - 1, D + 1, (8, 3)).astype(F32)  # upper border
    pts[16:20] = np.array([[0, 0, 0], [D - 1, D - 1, D - 1], [3, 4, 5], [2.5, 2.5, 2.5]], F32)
    bi = rs.randint(0, B, P).astype(np.int32)
    gy = rs.uniform(-1, 1, (P, C)).astype(F32)
    out = dict(voxelized=vox, points=pts, batch_indices=bi, gy=gy)
    shim.set_mode("cpu")
    out["ref_values_cpu"] = np.asarray(m.InterpolateVoxelGrid()(vox, pts, bi))
    shim.set_mode("gpu")
    f = m.InterpolateVoxelGrid()
    out["ref_values_gpu"] = np.asarray(f(vox, pts, bi))
    out["ref_gvoxelized_gpu"] = np.asarray(f.backward((vox, pts, bi), (gy,))[0])
    _save("interpolate_16", **out)


# ---------------------------------------------------------------- TDF / pseudo occupancy
def tdf_cases():
    rs = np.random.RandomState(3)
    cases = []
    # the reference's own __main__ self-check inputs (truncated_distance_function.py:222-231)
    cases.append(dict(name="main5", points=np.array([[0.5, 0.5, 0.5], [1.48, 1.48, 1.48]], F32),
                      pitch=F32(0.5), origin=np.zeros(3, F32), dims=(5, 5, 5), truncation=F32(1.2)))
    # ICC-shaped: threshold 2 => ksize 3, 27 offsets; points on a sphere shell + interior
    P = 700
    d = rs.normal(size=(P, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
    pts = (d * rs.uniform(0.0, 0.045, (P, 1))).astype(F32) + np.array([0.3, -0.1, 0.7], F32)
    pitch = F32(0.006296589104319322)
    origin = (np.array([0.3, -0.1, 0.7], F32) - pitch * F32(7.5)).astype(F32)
    cases.append(dict(name="ball16", points=pts, pitch=pitch, origin=origin, dims=(16, 16, 16),
                      truncation=F32(2) * pitch))
    # lattice points exactly on voxel centres / faces -> exact distance ties
    g = np.stack(np.meshgrid(*(np.arange(0, 6, 0.5),) * 3, indexing="ij"), -1).reshape(-1, 3)
    cases.append(dict(name="lattice_ties", points=g.astype(F32), pitch=F32(1.0),
                      origin=np.zeros(3, F32), dims=(6, 6, 6), truncation=F32(2.0)))
    return cases


def gen_tdf():
    m = _geo("truncated_distance_function")
    shim.set_mode("gpu")
    rs = np.random.RandomState(4)
    for c in tdf_cases():
        f = m.TruncatedDistanceFunction(
            pitch=c["pitch"], origin=c["origin"], dims=c["dims"], truncation=c["truncation"])
        tdf = np.asarray(f(c["points"]))
        K = f._ksize ** 3
        idx = np.asarray(f._indices) // K
        gy = rs.uniform(-1, 1, c["dims"]).astype(F32)
        gp = np.asarray(f.backward((c["points"],), (gy,))[0])
        sdf = rs.uniform(-0.01, 0.03, c["points"].shape[0]).astype(F32)
        thr = 2
        po = m.pseudo_occupancy_voxelization(
            c["points"], sdf, pitch=c["pitch"], origin=c["origin"], dims=c["dims"],
            threshold=thr, sdf_offset=0.02)
        po0 = m.pseudo_occupancy_voxelization(
            c["points"], sdf, pitch=c["pitch"], origin=c["origin"], dims=c["dims"],
            threshold=thr)
        out = {k: v for k, v in c.items() if k != "name"}
        out["dims"] = np.array(c["dims"])
        out.update(gy=gy, sdf=sdf, threshold=thr, sdf_offset=F32(0.02), ksize=f._ksize,
                   ref_tdf=tdf, ref_indices=idx, ref_gpoints=gp,
                   ref_po_grid=np.asarray(po[0]), ref_po_surface=np.asarray(po[1]),
                   ref_po_inside=np.asarray(po[2]),
                   ref_po0_surface=np.asarray(po0[1]), ref_po0_inside=np.asarray(po0[2]))
        _save("tdf_" + c["name"], **out)


# ---------------------------------------------------------------- occupancy_grid_3d
def gen_occupancy():
    m = _geo("occupancy_grid_3d")
    shim.set_mode("cpu")
    rs = np.random.RandomState(5)
    # known-answer inputs of tests/.../test_occupancy_grid_3d.py:13-38
    kat_pts = np.array([[0, 0.05, 0.1], [3.9, 3.95, 4]], F32)
    kat = np.asarray(m.occupancy_grid_3d(kat_pts, pitch=1, origin=(0, 0, 0), dims=(5, 5, 5)))
    pts = rs.uniform(0.1, 0.5, (40, 3)).astype(F32)
    pitch, origin, dims, thr = F32(0.05), np.array([0.05, 0.1, 0.0], F32), (8, 7, 6), 2
    y = np.asarray(m.occupancy_grid_3d(pts, pitch=pitch, origin=origin, dims=dims, threshold=thr))
    f = m.OccupancyGrid3D(pitch=pitch, origin=origin, dims=dims)
    d = [np.asarray(x) for x in f(pts)]
    gd = [rs.uniform(-1, 1, x.shape).astype(F32) for x in d]
    gp = np.asarray(f.backward((pts,), gd)[0])
    _save("occupancy_grid_3d", kat_points=kat_pts, ref_kat=kat, points=pts, pitch=pitch,
          origin=origin, dims=np.array(dims), threshold=thr, ref_grid=y,
          gd0=gd[0], gd1=gd[1], gd2=gd[2], ref_gpoints_from_gd=gp)


# ---------------------------------------------------------------- transforms
def gen_transforms():
    shim.set_mode("cpu")
    rs = np.random.RandomState(6)
    qm = _geo("quaternion_matrix")
    ct = _geo("compose_transform")
    tm = _geo("translation_matrix")
    tfm = _geo("transformation_matrix")
    tp = _geo("transform_points")
    q = rs.normal(size=(7, 4)).astype(F32)       # deliberately NOT unit norm
    t = rs.uniform(-1, 1, (7, 3)).astype(F32)
    R = np.asarray(qm.quaternion_matrix(q))
    R1 = np.asarray(qm.quaternion_matrix(q[0]))
    gR = rs.uniform(-1, 1, (7, 4, 4)).astype(F32)
    Q = rs.uniform(-1, 1, (7, 4, 4)).astype(F32)
    table_fwd = np.asarray(qm.QuaternionMatrix()(Q))
    table_bwd = np.asarray(qm.QuaternionMatrix().backward((Q,), (gR,))[0])
    T = np.asarray(tfm.transformation_matrix(q, t))
    T1 = np.asarray(tfm.transformation_matrix(q[1], t[1]))
    Tc = np.asarray(ct.compose_transform(R[:, :3, :3], t))
    Tt = np.asarray(tm.translation_matrix(t))
    gc = ct.ComposeTransform().backward((R[:, :3, :3], t), (gR,))
    pts = rs.uniform(-1, 1, (50, 3)).astype(F32)
    X = np.asarray(tp.transform_points(pts, T))
    X1 = np.asarray(tp.transform_points(pts, T[2]))
    _save("transforms", q=q, t=t, gR=gR, Q=Q, points=pts, ref_R=R, ref_R_single=R1,
          ref_table_fwd=table_fwd, ref_table_bwd=table_bwd, ref_T=T, ref_T_single=T1,
          ref_compose=Tc, ref_translation=Tt, ref_compose_gR=np.asarray(gc[0]),
          ref_compose_gt=np.asarray(gc[1]), ref_points_M=X, ref_points_single=X1)


# ---------------------------------------------------------------- ICC forward (loss)
def icc_scene(seed=7, N=3, D=16):
    """Small synthetic contact scene: N balls of lattice points with analytic sdf."""
    rs = np.random.RandomState(seed)
    pitch = np.array([0.0063, 0.0087, 0.0064, 0.0044][:N], F32)
    centers = np.array([[0.00, 0.00, 0.60], [0.055, 0.01, 0.61], [0.02, 0.06, 0.59], [0.0, -0.05, 0.6]][:N], F32)
    points, sdf, T0, origin, gt, gne = [], [], [], [], [], []
    for i in range(N):
        r = F32(pitch[i] * D * 0.30)
        ax = np.arange(-r, r + 1e-9, pitch[i])
        g = np.stack(np.meshgrid(ax, ax, ax, indexing="ij"), -1).reshape(-1, 3)
        d = np.linalg.norm(g, axis=1)
        keep = d <= r
        points.append(g[keep].astype(F32))
        sdf.append((r - d[keep]).astype(F32))
        ang = rs.uniform(-0.3, 0.3, 3)
        q = np.array([1.0, *ang]); q /= np.linalg.norm(q)
        w, x, y, z = q
        R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                      [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                      [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
        T = np.eye(4); T[:3, :3] = R; T[:3, 3] = centers[i] + rs.normal(0, 0.004, 3)
        T0.append(T.astype(F32))
        origin.append((centers[i] - pitch[i] * (D / 2.0 - 0.5)).astype(F32))
        ijk = np.stack(np.meshgrid(*(np.arange(D),) * 3, indexing="ij"), -1).astype(F32)
        c = ijk * pitch[i] + origin[-1]
        dist = np.linalg.norm(c - centers[i], axis=-1)
        gt.append(((dist < r) & (dist > r - 1.5 * pitch[i]) & (c[..., 2] < centers[i][2])).astype(F32))
        gne.append(((dist > r + pitch[i]) & (rs.uniform(size=dist.shape) < 0.7)).astype(F32))
    return dict(points=points, sdf=sdf, transform_init=np.stack(T0), pitch=pitch,
                origin=np.stack(origin), grid_target=np.stack(gt),
                grid_nontarget_empty=np.stack(gne), voxel_dim=D)


def gen_icc():
    shim.load_functions_namespace()
    shim.set_mode("gpu")
    link_mod = shim.ref_module("contrib.iterative_collision_check_link")
    for name, kw in [("contact3", dict(seed=7, N=3)), ("isolated2", dict(seed=8, N=2)),
                     ("single1", dict(seed=9, N=1))]:
        s = icc_scene(**kw)
        if name == "isolated2":      # far apart: grid_other is NaN -> F.maximum skipped (:82)
            s["transform_init"][1, :3, 3] += np.array([0.5, 0, 0], F32)
            s["origin"][1] += np.array([0.5, 0, 0], F32)
        link = link_mod.IterativeCollisionCheckLink(
            s["transform_init"], voxel_dim=s["voxel_dim"], voxel_threshold=2, sdf_offset=0.02)
        with np.errstate(invalid="ignore", divide="ignore"):
            loss = link(s["points"], s["sdf"], s["pitch"], s["origin"], s["grid_target"],
                        s["grid_nontarget_empty"])
        out = dict(transform_init=s["transform_init"], pitch=s["pitch"], origin=s["origin"],
                   grid_target=s["grid_target"], grid_nontarget_empty=s["grid_nontarget_empty"],
                   voxel_dim=s["voxel_dim"], sdf_offset=F32(0.02), voxel_threshold=2,
                   ref_quaternion=np.asarray(link.quaternion), ref_translation=np.asarray(link.translation),
                   ref_loss=np.asarray(loss, dtype=F32), n_objects=len(s["points"]))
        for i, (p, d) in enumerate(zip(s["points"], s["sdf"])):
            out[f"points_{i}"] = p
            out[f"sdf_{i}"] = d
        _save("icc_forward_" + name, **out)


# ---------------------------------------------------------------- average_distance loss
def gen_average_distance():
    shim.load_functions_namespace()
    shim.set_mode("cpu")
    m = shim.ref_module("functions.loss.average_distance")
    rs = np.random.RandomState(11)
    # mirrors tests/functions_tests/loss_tests/test_average_distance.py:13-21 (128 points, 5 preds)
    P, M = 128, 5

    def rand_T():
        q = rs.normal(size=4); q /= np.linalg.norm(q)
        w, x, y, z = q
        T = np.eye(4)
        T[:3, :3] = [[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]]
        T[:3, 3] = rs.uniform(-1, 1, 3)
        return T.astype(F32)
    points = rs.uniform(-1, 1, (P, 3)).astype(F32)
    T1 = rand_T()
    T2 = np.stack([rand_T() for _ in range(M)])
    T2[0] = T1                       # identical pose: distance exactly 0
    T2[1, :3, 3] = T1[:3, 3]; T2[1, :3, :3] = T1[:3, :3] @ np.diag([1, -1, -1]).astype(F32)  # 180 deg flip
    out = dict(points=points, T1=T1, T2=T2)
    out["ref_add"] = np.asarray(m.average_distance(points, T1, T2, symmetric=False))
    out["ref_add_s"] = np.asarray(m.average_distance(points, T1, T2, symmetric=True))
    _save("average_distance", **out)


# ---------------------------------------------------------------- occupancy-grid producer
def octree_mapping_scene(seed=21, H=48, W=64):
    """Two depth frames (second one from a shifted sensor origin) of three objects in front of a
    tilted background; instance label image; NaN dropout."""
    rs = np.random.RandomState(seed)
    u, v = np.meshgrid(np.arange(W), np.arange(H))
    f = 90.0
    frames = []
    for fr, org in enumerate(((0.0, 0.0, 0.0), (0.021, -0.013, 0.006))):
        z = 0.62 + 0.12 * (u / W) + 0.004 * rs.rand(H, W)
        label = np.zeros((H, W), np.int32)
        for ins, (cu, cv, ru, rv, zz) in {1: (16, 14, 9, 8, 0.40), 2: (40, 24, 11, 9, 0.45),
                                          3: (28, 36, 8, 7, 0.36)}.items():
            m = (np.abs(u - cu - 2 * fr) < ru) & (np.abs(v - cv) < rv)
            z = np.where(m, zz + 0.02 * ((u - cu) / ru) ** 2 + 0.003 * rs.rand(H, W), z)
            label[m] = ins
        pcd = np.stack([(u - W / 2) * z / f, (v - H / 2) * z / f, z], -1).astype(F32)
        pcd = pcd + np.asarray(org, F32)
        pcd[rs.rand(H, W) < 0.04] = np.nan
        frames.append((pcd, label, np.asarray(org, np.float64)))
    return frames


def gen_octree_mapping():
    shim.install()
    mod = shim.ref_module("contrib.multi_instance_octree_mapping")
    frames = octree_mapping_scene()
    pitches = {1: 0.006, 2: 0.0075, 3: 0.005, 0: 0.01}
    mapping = mod.MultiInstanceOctreeMapping()
    for ins in (1, 2, 3, 0):                          # build_octomap order: foreground, then background
        mapping.initialize(ins, pitch=pitches[ins])
    for pcd, label, org in frames:
        for ins in (1, 2, 3, 0):
            mapping.integrate(ins, label == ins, pcd, origin=org)
    out = dict(instance_ids=np.array([1, 2, 3, 0]), pitches=np.array([pitches[i] for i in (1, 2, 3, 0)]))
    for n, (pcd, label, org) in enumerate(frames):
        out[f"pcd{n}"], out[f"label{n}"], out[f"origin{n}"] = pcd, label, org
    pcd0, label0, _ = frames[0]
    for tid in (1, 3):
        center = np.nanmedian(pcd0[label0 == tid], axis=0)
        origin = center - (32 / 2 - 0.5) * pitches[tid]       # datasets/rgbd_pose_estimation/base.py:153-156
        gt, gn, ge = mapping.get_target_grids(tid, dimensions=(32, 32, 32), pitch=pitches[tid], origin=origin)
        out[f"grid_origin_{tid}"] = origin
        out[f"ref_grid_target_{tid}"], out[f"ref_grid_nontarget_{tid}"], out[f"ref_grid_empty_{tid}"] = gt, gn, ge
    for ins in (1, 2, 3, 0):                          # the map itself: keys and float32 log-odds
        cells = mapping._octrees[ins].cells
        keys = np.array(sorted(cells), dtype=np.int32).reshape(-1, 3)
        out[f"cells_keys_{ins}"] = keys
        out[f"cells_logodds_{ins}"] = np.array([cells[tuple(k)] for k in keys], dtype=F32)
    occ, emp = mapping.get_target_pcds(2)
    order = lambda a: a[np.lexsort(a.T[::-1])]
    out["ref_pcd_occupied_2"], out["ref_pcd_empty_2"] = order(occ), order(emp)
    _save("octree_mapping", **out)


def gen_octree_mapping_update():
    """The reference class's ``update`` (multi_instance_octree_mapping.py:29-34: updateNodes on
    every row, then updateInnerOccupancy) after one scan, and the grids it leads to."""
    shim.install()
    mod = shim.ref_module("contrib.multi_instance_octree_mapping")
    pcd, label, org = octree_mapping_scene(seed=33, H=24, W=32)[0]
    mapping = mod.MultiInstanceOctreeMapping()
    mapping.initialize(1, pitch=0.006)
    mapping.initialize(0, pitch=0.012)
    mapping.integrate(1, label == 1, pcd, origin=org)
    mapping.integrate(0, label != 1, pcd, origin=org)
    rs = np.random.RandomState(5)
    centre = np.nanmedian(pcd[label == 1], axis=0).astype(np.float64)
    occupied = centre + rs.uniform(-0.03, 0.03, (400, 3))
    occupied[:12] = occupied[0]                     # 12 rows in one cell: the clamp is reached
    mapping.update(1, occupied)
    cells = mapping._octrees[1].cells
    keys = np.array(sorted(cells), dtype=np.int32).reshape(-1, 3)
    origin = centre - 7.5 * 0.006
    gt, gn, ge = mapping.get_target_grids(1, dimensions=(16, 16, 16), pitch=0.006, origin=origin)
    _save("octree_mapping_update", pcd=pcd, label=label, origin=org, occupied=occupied,
          cells_keys_1=keys, cells_logodds_1=np.array([cells[tuple(k)] for k in keys], dtype=F32),
          grid_origin=origin, ref_grid_target=gt, ref_grid_nontarget=gn, ref_grid_empty=ge)


def main():
    assert shim.reference_available(), "needs /root/reference"
    _WRITTEN.clear()
    gen_octree_mapping()
    gen_octree_mapping_update()
    gen_average_distance()
    gen_voxelization()
    gen_interpolate()
    gen_tdf()
    gen_occupancy()
    gen_transforms()
    gen_icc()
    digests = {f: file_digests(os.path.join(OUT, f)) for f in sorted(_WRITTEN)}
    with open(os.path.join(OUT, DIGESTS), "w") as f:
        json.dump(digests, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    sys.exit(main())
