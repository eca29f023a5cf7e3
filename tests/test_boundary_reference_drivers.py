"""Drop-in boundary (SURVEY.md 8(b)): with ``clifford-vae_b200/`` ahead of the reference checkout on PYTHONPATH,
every reference driver, model file and script must import -- i.e. ``utils.vsa`` / ``dists.clifford`` /
``hyperspherical_vae`` here export every name the reference's callers pull from them
(mnist/mnist_clifpws.py:20-37, mnist/mnist_vmf.py:19-33, cnn/cifar10_train.py:23-39, cnn/fashion_train.py:24-42,
scripts/*.py) -- and the hot-path modules they end up with must be this repo's, not the reference's.

With the reference checkout present, every driver is imported in a subprocess; matplotlib may be absent, so tests/stubs/
holds a permissive stand-in.  Without the checkout, the drop-in modules are checked against the names those drivers, model
files and utils/wandb_utils.py import from them, recorded in tests/golden/reference_imports.json.
scripts/surface_area_plot.py is a module-level matplotlib figure with no hot-path import and is not covered."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("CLIFFORD_VAE_REFERENCE_ROOT", "/root/reference")

MODULES = [
    "mnist.mlp_vae", "mnist.mnist_clifpws", "mnist.mnist_vmf",
    "cnn.models", "cnn.cliffordar_model", "cnn.cifar10_train", "cnn.fashion_train",
    "scripts.binding_depth_heatmap", "scripts.bundle_heatmap", "scripts.rolefiller_heatmap",
    "scripts.sample_viz", "scripts.paper_bind_bundle_figure",
]

_PROG = r"""
import importlib, os, sys
mods = os.environ["CVB_TEST_MODULES"].split(",")     # not argv: scripts/sample_viz.py parses sys.argv at import
for m in mods:
    try:
        importlib.import_module(m)
    except Exception as e:
        # scripts/sample_viz.py draws samples from CPU-resident distributions at import time (:181); its imports
        # (:20-27) have resolved by then and the drop-in refuses CPU tensors by design (no CPU fallback)
        if m == "scripts.sample_viz" and type(e).__name__ == "CliffordB200Error":
            print("NOTE sample_viz stopped at its CPU sampling call:", str(e)[:60])
            continue
        raise
import utils.vsa, dists.clifford, hyperspherical_vae.distributions as hv, utils.wandb_utils as wu
print("VSA", utils.vsa.__file__)
print("DISTS", dists.clifford.__file__)
print("VMF", hv.__file__)
print("WANDB", wu.__file__)
for name in ("test_bundle_capacity", "test_binding_unbinding_pairs", "test_per_class_bundle_capacity_k_items",
             "hrr_init", "unitary_init", "normalize_vectors", "bind", "invert", "unbind", "bundle",
             "permute_vector", "unpermute_vector", "similarity"):
    assert callable(getattr(utils.vsa, name)), name
import mnist.mlp_vae as mv, cnn.models as cm
from clifford_b200 import distributions as D
assert mv.CliffordPowerSphericalDistribution is D.CliffordPowerSphericalDistribution
assert cm.CliffordPowerSphericalDistribution is D.CliffordPowerSphericalDistribution
assert cm.PowerSpherical is D.PowerSpherical
print("ALL-OK")
"""


def _recorded_imports_are_exported():
    import importlib
    import json
    with open(os.path.join(ROOT, "tests", "golden", "reference_imports.json")) as f:
        want = json.load(f)
    pkg = os.path.join(ROOT, "clifford-vae_b200")
    for mod_name, names in want.items():
        mod = importlib.import_module(mod_name)
        assert mod.__file__.startswith(pkg), (mod_name, mod.__file__)
        for name in names:
            assert callable(getattr(mod, name, None)), (mod_name, name)
    import dists.clifford as dc
    from clifford_b200 import distributions as D
    assert dc.CliffordPowerSphericalDistribution is D.CliffordPowerSphericalDistribution
    assert dc.PowerSpherical is D.PowerSpherical


def test_every_reference_driver_imports_on_the_drop_in_modules():
    if not os.path.isdir(os.path.join(REF, "mnist")):
        _recorded_imports_are_exported()
        return
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "clifford-vae_b200"), os.path.join(ROOT, "tests", "stubs"),
                                         REF, os.path.join(REF, "vmf")])
    env.pop("CLIFFORD_VAE_REFERENCE_ROOT", None)       # the checkout must be found through sys.path alone
    env["CVB_TEST_MODULES"] = ",".join(MODULES)
    out = subprocess.run([sys.executable, "-c", _PROG], env=env, cwd="/tmp", capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = dict(l.split(" ", 1) for l in out.stdout.strip().splitlines() if " " in l)
    pkg = os.path.join(ROOT, "clifford-vae_b200")
    assert lines["VSA"].startswith(pkg) and lines["DISTS"].startswith(pkg) and lines["VMF"].startswith(pkg)
    assert lines["WANDB"].startswith(REF)              # plots/logging stay the reference's
    assert "ALL-OK" in out.stdout


def test_harness_entry_points_keep_the_reference_signatures():
    """Argument names, order and defaults of the three harness functions (reference utils/vsa.py:99-113, 224-238,
    402-418), checked against the reference when it is present, else against the recorded lists."""
    import inspect
    from utils import vsa
    want = {
        "test_bundle_capacity": ["d", "n_items", "k_range", "n_trials", "normalize", "device", "plot", "decoder",
                                 "save_dir", "item_memory", "use_braiding", "bind_with_random", "baseline_d"],
        "test_binding_unbinding_pairs": ["d", "n_items", "k_range", "n_trials", "normalize", "device", "plot",
                                         "unbind_method", "save_dir", "item_memory", "use_braiding",
                                         "bind_with_random", "baseline_d"],
        "test_per_class_bundle_capacity_k_items": ["d", "n_items", "n_classes", "items_per_class", "n_trials",
                                                   "normalize", "device", "plot", "save_dir", "item_memory", "labels",
                                                   "item_images", "use_braiding", "per_class_braid", "class_names"],
    }
    for name, params in want.items():
        sig = inspect.signature(getattr(vsa, name))
        got = [p for p in sig.parameters if not p.startswith("_")]
        assert got == params, (name, got)
    assert inspect.signature(vsa.test_binding_unbinding_pairs).parameters["bind_with_random"].default is True
    assert inspect.signature(vsa.test_bundle_capacity).parameters["bind_with_random"].default is False
    assert inspect.signature(vsa.hrr_init).parameters["device"].default == "cpu"
