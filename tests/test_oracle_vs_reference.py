"""The committed golden vectors are the reference's OWN output: its NumPy paths and CuPy kernel
source strings, run through oracle/ref_harness (serial C++ emulation), wrote every array of
tests/golden/*.npz.  oracle/ref_harness/gen_golden.py records a SHA-256 of each array it wrote
in tests/golden/reference_digests.json; the fixtures are checked against that record, and the
reference's committed ICC scene is stored verbatim under tests/golden/pose_refinement_scene/."""

import json
import os

import numpy as np

from oracle.ref_harness import gen_golden as gg


def test_goldens_regenerate_bit_identically():
    committed = gg.OUT
    with open(os.path.join(committed, gg.DIGESTS)) as f:
        recorded = json.load(f)
    # icc_closed_loop_* are ORACLE trajectories (oracle/ref_harness/gen_icc_closed_loop.py, minutes
    # of NumPy each); their reference-derived inputs are checked below
    names = sorted(f for f in os.listdir(committed)
                   if f.endswith(".npz") and not f.startswith("icc_closed_loop_"))
    assert names == sorted(recorded), "generator and committed fixture sets differ"
    for f in names:
        got = gg.file_digests(os.path.join(committed, f))
        assert set(got) == set(recorded[f]), f
        for k in got:
            assert got[k] == recorded[f][k], (f, k)


def test_icc_ref3_fixture_inputs_come_from_the_reference():
    """tests/golden/icc_closed_loop_ref3.npz carries the reference's committed 3-object scene
    (examples/ycb_video/pose_refinement/data/0000000{0,1,2}.npz) verbatim."""
    from oracle.ref_harness import gen_icc_closed_loop as gen
    g = np.load(os.path.join(gen.OUT, "icc_closed_loop_ref3.npz"))
    sc = gen.ref3_scene()
    assert gen.inputs_checksum(sc) == str(g["inputs_sha1"])
    for i in range(3):
        d = np.load(os.path.join(gen.REF_DATA, f"{i:08d}.npz"))
        assert np.array_equal(g["transform_init"][i], d["transform_init"])
        assert np.array_equal(g["grid_target"][i], d["grid_target"])
        assert np.array_equal(g["grid_nontarget_empty"][i], d["grid_nontarget_empty"])
        assert np.array_equal(g["origin"][i], d["origin"])
        assert g["pitch"][i] == np.float32(d["pitch"])
