"""Generate tests/golden/icc_closed_loop_*.npz: oracle trajectories of the ICC driver loop
(check_iterative_collision_check_link.py:44-79: Adam(0.01), translation alpha x0.1, 100
iterations, sdf_offset=0.02) that the GPU closed-loop parity tests compare with.

TEST INFRASTRUCTURE ONLY:

    python -m oracle.ref_harness.gen_icc_closed_loop [seed3 seed4 ref3]

  seed3 / seed4   BASELINE config 4: morefusion_b200.synthetic.make_icc_scene(N=8, seed) -- the
                  inputs are regenerated from the seed at test time, only the oracle's outputs
                  (q, t, loss history) and a checksum of the inputs are stored.
  ref3            the reference's committed 3-object scene
                  (examples/ycb_video/pose_refinement/data/0000000{0,1,2}.npz, stored under
                  tests/golden/pose_refinement_scene/:
                  transform_init, pitch, origin, grid_target, grid_nontarget_empty copied
                  verbatim).  The fixture lacks the SDF samples (models.get_sdf needs the YCB
                  download, check_iterative_collision_check_link.py:30), so points/sdf are an
                  analytic stand-in: the three objects are YCB boxes (class 3 sugar_box, 2
                  cracker_box, 9 gelatin_box); lattice points at the class pitch inside the
                  bounding box of `pcd_cad`, sdf = signed distance to that box, positive inside
                  (datasets/ycb_video/models.py:66-79 convention).
"""

import hashlib
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import icc as oicc  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
# the reference's examples/ycb_video/pose_refinement/data/0000000{0,1,2}.npz, stored verbatim
REF_DATA = os.path.join(OUT, "pose_refinement_scene")
F32 = np.float32


def checksum(arrays):
    h = hashlib.sha1()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def box_sdf_lattice(pcd_cad, pitch):
    lo, hi = pcd_cad.min(0).astype(np.float64), pcd_cad.max(0).astype(np.float64)
    c, half = (lo + hi) / 2, (hi - lo) / 2
    ax = [np.arange(-h, h + 1e-9, pitch) for h in half]
    g = np.stack(np.meshgrid(*ax, indexing="ij"), -1).reshape(-1, 3)
    q = np.abs(g) - half
    d = -(np.linalg.norm(np.maximum(q, 0), axis=-1) + np.minimum(q.max(axis=-1), 0))
    return (g + c).astype(F32), d.astype(F32)


def ref3_scene():
    inst = [np.load(os.path.join(REF_DATA, f"{i:08d}.npz")) for i in range(3)]
    points, sdf = zip(*[box_sdf_lattice(d["pcd_cad"], float(d["pitch"])) for d in inst])
    return dict(
        class_id=np.array([int(d["class_id"]) for d in inst], np.int32),
        points=list(points), sdf=list(sdf),
        pitch=np.array([d["pitch"] for d in inst]).astype(F32),
        origin=np.stack([d["origin"] for d in inst]).astype(F32),
        grid_target=np.stack([d["grid_target"] for d in inst]).astype(F32),
        grid_nontarget_empty=np.stack([d["grid_nontarget_empty"] for d in inst]).astype(F32),
        transform_init=np.stack([d["transform_init"] for d in inst]).astype(F32))


def scene(name):
    from morefusion_b200 import synthetic
    if name == "seed3":
        return synthetic.make_icc_scene(N=8, seed=3, kinds=("box",))
    if name == "seed4":
        return synthetic.make_icc_scene(N=8, seed=4, kinds=("box", "cylinder", "sphere"))
    if name == "ref3":
        return ref3_scene()
    raise KeyError(name)


def inputs_checksum(sc):
    return checksum(list(sc["points"]) + list(sc["sdf"]) + [
        sc["pitch"], sc["origin"], sc["grid_target"], sc["grid_nontarget_empty"],
        sc["transform_init"]])


def main(names):
    for name in names:
        sc = scene(name)
        t0 = time.time()
        # the initial (q, t) are part of the fixture: quaternion_from_matrix uses LAPACK eigh,
        # whose last bits are CPU dependent, and the loop is chaotic in them
        q0 = np.stack([oicc.tfm.quaternion_from_matrix(T) for T in sc["transform_init"]]).astype(F32)
        t0_ = np.stack([np.asarray(T)[:3, 3] for T in sc["transform_init"]]).astype(F32)
        q, t, hist = oicc.icc_refine(
            sc["transform_init"], sc["points"], sc["sdf"], sc["pitch"], sc["origin"],
            sc["grid_target"], sc["grid_nontarget_empty"], n_iter=100, sdf_offset=0.02,
            return_history=True, q0=q0, t0=t0_)
        out = dict(q=q, t=t, q0=q0, t0=t0_, loss=np.array(hist, F32), n_iter=100,
                   sdf_offset=F32(0.02),
                   inputs_sha1=inputs_checksum(sc), oracle_cpu_s=time.time() - t0)
        if name == "ref3":
            sizes = np.array([p.shape[0] for p in sc["points"]], np.int64)
            out.update(
                class_id=sc["class_id"], sizes=sizes, points=np.concatenate(sc["points"]),
                sdf=np.concatenate(sc["sdf"]), pitch=sc["pitch"], origin=sc["origin"],
                grid_target=sc["grid_target"].astype(np.uint8),
                grid_nontarget_empty=sc["grid_nontarget_empty"].astype(np.uint8),
                transform_init=sc["transform_init"])
        path = os.path.join(OUT, f"icc_closed_loop_{name}.npz")
        np.savez_compressed(path, **out)
        print("wrote", path, os.path.getsize(path), "bytes", f"{time.time() - t0:.1f}s",
              "loss", hist[0], "->", hist[-1], flush=True)


if __name__ == "__main__":
    main(sys.argv[1:] or ["ref3", "seed3", "seed4"])
