"""The C++ host's OBJ/MTL reader (cedec-2024-rt_b200/host/obj_scene.hpp) against the reference's own loader
(common/loader.hpp:11-66 + tinyobjloader 1.0.6): primitive order and vertex/material bits must be identical.
The committed fixture's golden was produced by oracle/_ref/libref_loader.so (the reference loader itself):
    python -c "import sys; sys.path.insert(0,'oracle'); import orc, numpy as np; \
      np.save('tests/golden/obj/tricky_reference_loader.npy', orc.load_obj_reference('tests/golden/obj/tricky.obj','tests/golden/obj/'))"
cornellbox1.obj and blocks_ao.obj (+ .mtl) hold two of the scenes the examples load, written back from the reference loader's
Triangle[] in golden/scenes_small.npz (the original asset files are not part of the repository): one `v` per distinct
position and one material per distinct (Kd, Ke), every value as printf("%.9g") of its float, faces in triangle order.
"""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOOL = os.path.join(ROOT, "cedec-2024-rt_b200", "obj_to_tri")
OBJ = os.path.join(ROOT, "tests", "golden", "obj")


def _convert(obj, tmp_path):
    if not os.path.exists(TOOL):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "cedec-2024-rt_b200", "csrc")], check=True)
    out = str(tmp_path / "out.tri")
    subprocess.run([TOOL, obj, out], check=True, capture_output=True)
    return open(out, "rb").read()


def test_fixture_matches_reference_loader(tmp_path):
    """polygons (fan order), negative indices, exponents, '.5' (unparsable for tinyobj -> 0), v/vt/vn forms"""
    want = np.load(os.path.join(OBJ, "tricky_reference_loader.npy"))
    got = _convert(os.path.join(OBJ, "tricky.obj"), tmp_path)
    assert len(got) == want.nbytes and got == want.tobytes()


def test_missing_file_is_an_error(tmp_path):
    r = subprocess.run([TOOL, str(tmp_path / "nope.obj"), str(tmp_path / "o.tri")], capture_output=True, text=True)
    assert r.returncode == 1 and "cannot open" in r.stderr


@pytest.mark.parametrize("scene", ["cornellbox1", "blocks_ao"])
def test_reference_scenes_match_staged_caches(scene, tmp_path):
    """two of the scenes the examples load: identical to the bytes of the reference loader (golden/scenes_small.npz)"""
    want = np.load(os.path.join(ROOT, "tests", "golden", "scenes_small.npz"))[scene].tobytes()
    got = _convert(os.path.join(OBJ, scene + ".obj"), tmp_path)
    assert got == want
