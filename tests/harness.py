"""Boundary harness: runs the reference's UNMODIFIED host code ({training,pattern_class,dataset,divide_lr}.py of a
checkout of github.com/neurospin-projects/2022_pauriau_unetsulc) with `deepsulci.*` / `soma` / `sigraph` injected
through sys.modules (unetsulc_b200.deepsulci_shim).  The checkout is not part of this repository: set
UNETSULC_REFERENCE to its directory to use it.  Without it the tests use the fixtures under tests/golden/.
"""
import contextlib
import importlib
import io
import os
import random
import sys

import numpy as np
import torch

REF = os.environ.get("UNETSULC_REFERENCE", "")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def reference_available():
    return bool(REF) and os.path.isdir(REF)


def synthetic_cohort(n_subjects=3, shape=(16, 16, 16), n_classes=6, seed=0):
    """dict_bck2 / dict_names / sulci_side_list in the form the reference caches them (main.py:87-94)."""
    from oracle.synth import synth_points
    names = ['S%02d_left' % i for i in range(n_classes - 1)] + ['unknown']
    dict_bck2, dict_names = {}, {}
    for s in range(n_subjects):
        pts, nm = synth_points(shape, n_classes, seed + s, occupancy=0.08, names=names)
        g = 'subject%02d.arg' % s
        dict_bck2[g], dict_names[g] = pts, nm
    return dict_bck2, dict_names, sorted(set(names))


@contextlib.contextmanager
def reference_modules(unet3d=None, cutting=None, esi_score=None, early_stopping=None):
    """Imports the reference's modules fresh, bound to the given implementations of the five deepsulci symbols."""
    import unetsulc_b200  # noqa: F401
    from unetsulc_b200 import deepsulci_shim
    saved = {k: sys.modules.get(k) for k in list(sys.modules)
             if k.split(".")[0] in ("deepsulci", "soma", "sigraph", "training", "pattern_class", "dataset",
                                    "divide_lr", "fine_tunning")}
    for k in list(saved):
        sys.modules.pop(k, None)
    deepsulci_shim.install(unet3d=unet3d, cutting=cutting, esi_score=esi_score, early_stopping=early_stopping)
    sys.path.insert(0, REF)
    try:
        mods = {n: importlib.import_module(n) for n in ("dataset", "divide_lr", "fine_tunning", "pattern_class",
                                                        "training")}
        yield mods
    finally:
        sys.path.remove(REF)
        for k in list(sys.modules):
            if k.split(".")[0] in ("deepsulci", "soma", "sigraph", "training", "pattern_class", "dataset",
                                   "divide_lr", "fine_tunning"):
                sys.modules.pop(k, None)
        for k, v in saved.items():
            if v is not None:
                sys.modules[k] = v


def run_reference_training(workdir, unet3d, n_epochs=2, lr=1e-2, momentum=0.9, patience=None, seed=7,
                           cuda=-1, quiet=True):
    """reference training.py::UnetTrainingSulciLabelling.learning() on a synthetic cohort.  Returns results dict."""
    from oracle.cutting_ref import cutting_ref
    from oracle.stats_ref import esi_score_ref
    from oracle.early_stopping_ref import EarlyStoppingRef
    bck2, names, sslist = synthetic_cohort()
    files = sorted(bck2)
    with reference_modules(unet3d=unet3d, cutting=cutting_ref, esi_score=esi_score_ref,
                           early_stopping=EarlyStoppingRef) as mods:
        random.seed(seed); np.random.seed(seed); torch.manual_seed(seed)
        out = io.StringIO()
        with (contextlib.redirect_stdout(out) if quiet else contextlib.nullcontext()):
            method = mods["training"].UnetTrainingSulciLabelling(
                files, 'L', cuda=cuda, working_path=workdir, dict_model={'name': 'harness'},
                dict_names=names, dict_bck2=bck2, sulci_side_list=sslist)
            method.learning(lr, momentum, n_epochs, files[:2], files[2:], batch_size=1,
                            patience=patience or {})
        return method
