"""The drop-in claim of INTEGRATION.md, checked: with this package first on the path and FETAL_REFERENCE_ROOT pointing at
the reference checkout, the imports and `getattr` look-ups that fetal/train_fetal.py:5-39 and fetal/predict.py:5 perform
resolve - hot-path names to the B200 implementation, everything else to the reference's own files. Keras / TensorFlow /
nibabel / tables are absent in this image and are stubbed exactly as oracle/ref_harness.py stubs them (test
infrastructure); the test runs in a subprocess so that the stubs and the overlay environment cannot leak.

Where oracle/ref_harness.py finds no reference checkout, the overlay is checked against a stand-in checkout written to a
temporary directory: the
reference's `fetal_net` layout with the names fetal/train_fetal.py imports from the modules this package does not define,
and hot-path namesakes that raise when imported (so resolving one of them to the stand-in fails the test)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_SHADOWED = "raise ImportError('the reference module %s was imported instead of the B200 one')\n"
STAND_IN = {
    "fetal_net/__init__.py": "",
    "fetal_net/preprocess.py": "",
    "fetal_net/data.py": "def write_data_to_file(*a, **k):\n    pass\n\n\ndef open_data_file(*a, **k):\n    pass\n",
    "fetal_net/generator.py": "from .utils.patches import get_patch_from_3d_data  # noqa: F401\n"
                              "from .utils.utils import pickle_load  # noqa: F401\n\n\n"
                              "def get_training_and_validation_generators(*a, **k):\n    pass\n",
    "fetal_net/model/__init__.py": "",
    "fetal_net/model/fetal_net.py": "def fetal_envelope_model(*a, **k):\n    pass\n",
    "fetal_net/utils/__init__.py": "",
    "fetal_net/utils/utils.py": "def pickle_load(*a, **k):\n    pass\n",
}
for _m in ("training", "prediction", "metrics", "model/unet3d", "utils/patches"):
    STAND_IN["fetal_net/%s.py" % _m] = _SHADOWED % _m


@pytest.fixture
def reference_root(tmp_path):
    """The reference checkout where oracle.ref_harness finds it, else the stand-in checkout under tmp_path."""
    from oracle.ref_harness import REFERENCE_ROOT as ref
    if os.path.isdir(os.path.join(ref, "fetal_net")):
        return ref
    for rel, text in STAND_IN.items():
        path = tmp_path / rel
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_text(text)
    return str(tmp_path)

SCRIPT = r"""
import json, os, sys, types
root, pkg, ref = sys.argv[1:4]
sys.path.insert(0, root); sys.path.insert(0, pkg)
sys.path.append(ref)                                # `python -m fetal.train_fetal` is started from the checkout: its
                                                    # root (package `fetal`) is on the path, AFTER the B200 package
import numpy as np
np.int, np.float = int, float                       # removed NumPy aliases the reference still uses
from oracle.ref_harness import _Anything, _STUBBED
for name in _STUBBED:
    sys.modules.setdefault(name, _Anything(name))
import fetal_net, fetal_net.metrics, fetal_net.model
out = {}
out["pkg_file"] = fetal_net.__file__
# fetal/train_fetal.py:5-13
import fetal_net.preprocess
from fetal_net.data import write_data_to_file, open_data_file
from fetal_net.generator import get_training_and_validation_generators
from fetal_net.model.fetal_net import fetal_envelope_model
from fetal_net.training import load_old_model, train_model
out["preprocess"] = fetal_net.preprocess.__file__
out["data"] = sys.modules["fetal_net.data"].__file__
out["generator"] = sys.modules["fetal_net.generator"].__file__
out["model_fetal_net"] = sys.modules["fetal_net.model.fetal_net"].__file__
out["training"] = sys.modules["fetal_net.training"].__file__
# fetal/train_fetal.py:31-32 with the shipped config values (fetal/config_utils.py:73-79, SURVEY.md §8b)
for model_name in ("unet_model_3d", "isensee2017_model_3d", "unet_model_2d"):
    out["builder/" + model_name] = getattr(fetal_net.model, model_name).__module__
for loss in ("dice_coefficient_loss", "binary_crossentropy_loss", "dice_and_xent"):
    out["loss/" + loss] = getattr(fetal_net.metrics, loss).__module__
# fetal/predict.py:5
from fetal_net.prediction import run_validation_cases, patch_wise_prediction
import fetal_net.prediction as fp
out["prediction"] = fp.__file__
out["pwp_module"] = patch_wise_prediction.__module__
# the generator module of the reference found OUR patches module (it slices with get_patch_from_3d_data)
out["patches"] = sys.modules["fetal_net.utils.patches"].__file__
out["utils_utils"] = sys.modules["fetal_net.utils.utils"].__file__
print(json.dumps(out))
"""


def test_reference_scripts_resolve_through_the_overlay(reference_root):
    REF = reference_root
    pkg = os.path.join(ROOT, "fetal-mri-segmentation_b200")
    env = dict(os.environ, FETAL_REFERENCE_ROOT=REF)
    r = subprocess.run([sys.executable, "-c", SCRIPT, ROOT, pkg, REF], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    ours = os.path.join(pkg, "fetal_net")
    theirs = os.path.join(REF, "fetal_net")
    assert out["pkg_file"].startswith(ours)
    for k in ("training", "prediction", "patches"):                 # hot-path modules: the B200 mirror
        assert out[k].startswith(ours), (k, out[k])
    for k in ("preprocess", "data", "generator", "model_fetal_net", "utils_utils"):   # everything else: the reference
        assert out[k].startswith(theirs), (k, out[k])
    for k, v in out.items():
        if k.startswith("builder/"):
            assert v == "fetal_net.model.unet3d", (k, v)
        if k.startswith("loss/"):
            assert v == "fetal_net.metrics", (k, v)
    assert out["pwp_module"] == "fetal_net.prediction"


def test_without_the_overlay_missing_modules_fail_loudly():
    pkg = os.path.join(ROOT, "fetal-mri-segmentation_b200")
    env = {k: v for k, v in os.environ.items() if k != "FETAL_REFERENCE_ROOT"}
    code = "import sys; sys.path.insert(0, %r); import fetal_net.model, fetal_net.prediction; import fetal_net.generator" % pkg
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "No module named 'fetal_net.generator'" in r.stderr
