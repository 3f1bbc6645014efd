"""Host BVH builds over boxes whose planes tie at -0.0 against +0.0: the signs of zero in the flattened nodes are part of the
tree fw_scene_build_host returns, so they are pinned here (with the SAH interior and with FW_BVH_SAH=0)."""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import REPO

VALS = [0.0, -0.0, 1e-45, -1e-45, 1e-40, -1e-40, 1e-38]
PINS = {  # n: (md5 of fw_scene_bvh_nodes with the SAH interior, the same with FW_BVH_SAH=0)
    33: ("af93d8a274d6e22ff89e31974da83f17", "82799739132db4c4e34dba159a2fcffd"),
    200: ("bf3465a382af272591fffaf90e554415", "10974c8ca9a139fd64437c8ed9de02b1"),
    2500: ("0b87146ed8df6d0c9c748667400375c9", "96c9e87167cdafac919834d03a14837b"),
}


def _hashes():
    from firework_b200.engine import NativeScene
    rng = np.random.default_rng(7)
    out = {}
    for n in PINS:
        objs = []
        for i in range(n):
            x, y, z = (VALS[k] for k in rng.integers(0, len(VALS), 3))
            r = [0.0, -0.0, 1e-45][i % 3]
            objs.append("  - obj:\n      object_type: Sphere\n      radius: %r\n      material: 0\n    position:\n      x: %r\n      y: %r\n"
                        "      z: %r\n    rotation:\n      s: 1.0\n      bv:\n        xy: 0.0\n        xz: 0.0\n        yz: 0.0\n"
                        "    flip_normals: false\n" % (r, x, y, z))
        text = ("---\nrender_objects:\n" + "".join(objs) + "materials:\n  - material: LambertianMat\n    albedo:\n"
                "      texture: ConstantTexture\n      color:\n        x: 0.5\n        y: 0.5\n        z: 0.5\n"
                "environment:\n  environment: ColorEnv\n  color:\n    x: 0.0\n    y: 0.0\n    z: 0.0\n")
        s = NativeScene(text, commit=False)
        s.build_host()
        out[n] = hashlib.md5(s.bvh_nodes()[0].tobytes()).hexdigest()
        s.close()
    return out


@pytest.mark.parametrize("sah", [1, 0])
def test_signed_zero_ties_keep_their_node_bytes(sah):
    if sah:
        got = _hashes()
    else:
        prog = ("import sys, json; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
                "from test_bvh_zero_signs import _hashes\nprint(json.dumps(_hashes()))\n" % (REPO, os.path.join(REPO, "tests")))
        import json
        out = subprocess.run([sys.executable, "-c", prog], env=dict(os.environ, FW_BVH_SAH="0"), capture_output=True, text=True,
                             check=True).stdout
        got = {int(k): v for k, v in json.loads(out.strip().splitlines()[-1]).items()}
    assert got == {n: PINS[n][0 if sah else 1] for n in PINS}
