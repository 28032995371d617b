"""GPU: the drop-in boundary of SURVEY 8b exercised the way a maintainer would use it -- the reference's own FaceRecon.py
(staged unmodified in oracle/_ref/pyref) with `network.fs_net_repo.gcn3d` swapped for `tgpose_b200.gcn3d`."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def test_reference_face_enc_runs_unchanged_on_our_gcn3d():
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "pyref", "network", "fs_net_repo", "FaceRecon.py")):
        pytest.skip("needs the original project's FaceRecon.py, staged into oracle/_ref/pyref by build() from the "
                    "unmodified reference sources, which this repository does not ship")
    # a fresh interpreter: the module swap must happen before the reference's FaceRecon is imported
    p = subprocess.run([sys.executable, os.path.join(HERE, "dropin_face_enc.py")], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    r = json.loads(p.stdout.strip().splitlines()[-1])
    print(r)
    assert r["shape"] == [2, 128, 1286] and r["global_shape"] == [2, 1286, 128] and r["finite"]
    assert r["same_init"] and r["state_keys_equal_golden"]        # same constructor order / parameter names as the reference
    # the reference's call sequence on the plain API and our fused encoder run the same kernels: they agree up to the
    # BatchNorm folding of the fused path (and the index flips that can seed); the reference golden is the T3 comparison
    assert r["frac_vs_fused"] > 0.99
    assert r["frac_vs_reference_golden"] > 0.90
