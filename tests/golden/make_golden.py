"""Regenerates the fixtures under tests/golden/.  Needs a checkout of the reference (see tests/harness.py):

    UNETSULC_REFERENCE=<checkout> python tests/golden/make_golden.py

Fixtures (small, committed):
  plateau_traces.json ........ decisions of the REFERENCE's own DivideLr / FineTunning (divide_lr.py, fine_tunning.py)
                               on fixed loss sequences -> pins our restated trackers
  dataset_cases.npz .......... volumes produced by the REFERENCE's own SulciDataset (dataset.py) for seeded inputs,
                               with and without rotation augmentation -> pins our SulciDataset
  reference_training.json .... results dict of the REFERENCE's unmodified training.py::learning() driven by the
                               oracle UNet3D on CPU (2 epochs, synthetic cohort) -> pins the host-side training semantics
  oracle_unet3d.npz .......... oracle forward/backward on a seeded 16x24x16 volume -> pins the oracle against drift
  cutting_cases.npz, esi_cases.json ... oracle integer pass on seeded inputs (bit-exact expectations for the GPU path)
"""
import json
import os
import random
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from tests import harness  # noqa: E402
from oracle.cutting_ref import cutting_ref  # noqa: E402
from oracle.stats_ref import esi_score_ref, esi_counts_ref  # noqa: E402
from oracle.synth import synth_scores, synth_volume  # noqa: E402
from oracle.unet3d_ref import UNet3DRef  # noqa: E402

LOSS_SEQS = {
    "improving": [1.0, 0.9, 0.8, 0.7, 0.6, 0.5],
    "plateau": [1.0, 0.9, 0.95, 0.96, 0.97, 0.5, 0.6, 0.7, 0.8, 0.9, 1.0],
    "noisy": [0.5, 0.6, 0.4, 0.45, 0.46, 0.47, 0.3, 0.31, 0.32, 0.33, 0.34, 0.35],
    "flat": [1.0] * 8,
}


def plateau_traces():
    out = {}
    with harness.reference_modules() as mods:
        import contextlib
        import io
        for name, seq in LOSS_SEQS.items():
            for patience in (1, 2, 3):
                for repeat in (1, 2):
                    d = mods["divide_lr"].DivideLr(patience=patience, repeat=repeat)
                    tr = []
                    with contextlib.redirect_stdout(io.StringIO()):
                        for v in seq:
                            d(v, None)
                            tr.append([bool(d.divide_lr), bool(d.stop), int(d.counter)])
                    out["divide_lr/%s/p%d/r%d" % (name, patience, repeat)] = tr
                f = mods["fine_tunning"].FineTunning(patience=patience)
                tr = []
                with contextlib.redirect_stdout(io.StringIO()):
                    for v in seq:
                        f(v, None)
                        tr.append([bool(f.ft_start), bool(f.stop), int(f.counter)])
                out["fine_tunning/%s/p%d" % (name, patience)] = tr
    return {"loss_sequences": LOSS_SEQS, "traces": out}


def dataset_cases():
    bck2, names, sslist = harness.synthetic_cohort(n_subjects=2, shape=(12, 14, 10), n_classes=5, seed=3)
    dict_sulci = {s: i for i, s in enumerate(sslist)}
    files = sorted(bck2)
    arrays = {}
    with harness.reference_modules() as mods:
        DS = mods["dataset"].SulciDataset
        for train in (False, True):
            random.seed(11); np.random.seed(11)
            ds = DS(files, dict(dict_sulci), train=train, dict_bck2=bck2, dict_names=names)
            for i in range(len(files)):
                for rep in range(2 if train else 1):
                    x, y = ds[i]
                    arrays["x_train%d_s%d_r%d" % (train, i, rep)] = x.numpy().astype(np.uint8)
                    arrays["y_train%d_s%d_r%d" % (train, i, rep)] = y.numpy().astype(np.int16)
        ds = DS(files, dict(dict_sulci), train=False, dict_bck2=bck2, dict_names=names, img_size=[16, 16, 16])
        x, y = ds[0]
        arrays["x_fixed"] = x.numpy().astype(np.uint8)
        arrays["y_fixed"] = y.numpy().astype(np.int16)
    return arrays


def reference_training():
    with tempfile.TemporaryDirectory() as tmp:
        method = harness.run_reference_training(tmp, UNet3DRef, n_epochs=2, patience={'divide_lr': 1,
                                                                                      'early_stopping': 3})
        res = dict(method.results)
        res.pop('duration', None)
        res['state_dict_keys'] = list(method.model.state_dict().keys())
        return res


def oracle_unet3d():
    torch.manual_seed(42)
    m = UNet3DRef(1, 56)
    x, labels = synth_volume((16, 24, 16), 56, 1234, occupancy=0.06)
    x, labels = x.unsqueeze(0), labels.unsqueeze(0)
    m.train()
    logits = m(x)
    loss = torch.nn.functional.cross_entropy(logits, labels, ignore_index=-1)
    loss.backward()
    m.eval()
    with torch.no_grad():
        probs = m(x)
    idx = torch.nonzero(labels[0] >= 0)[:64]
    return {
        "loss": np.float64(loss.item()),
        "logits_sample": logits[0][:, idx[:, 0], idx[:, 1], idx[:, 2]].detach().numpy().T.astype(np.float32),
        "probs_sample": probs[0][:, idx[:, 0], idx[:, 1], idx[:, 2]].numpy().T.astype(np.float32),
        "sample_index": idx.numpy().astype(np.int32),
        "logits_mean_std": np.array([logits.mean().item(), logits.std().item()], np.float64),
        "grad_norms": np.array([p.grad.norm().item() for p in m.parameters()], np.float64),
    }


def cutting_cases():
    rng = np.random.RandomState(5)
    out = {}
    for case, (n, nf, sharp) in enumerate([(1500, 12, 3.0), (2500, 40, 1.0), (500, 1, 2.0), (64, 64, 3.0)]):
        s = synth_scores(n, 56, seed=case + 1, sharp=sharp).numpy()
        v = rng.randint(0, nf, size=n) * 13 + 5
        out["scores%d" % case] = s.astype(np.float32)
        out["vert%d" % case] = v.astype(np.int64)
        for th in (0, 5, 50, 100, 150):
            out["out%d_th%d" % (case, th)] = np.asarray(cutting_ref(s, v, None, th), np.int16)
    return out


def esi_cases():
    rng = np.random.RandomState(9)
    cases = []
    for n in (0, 10, 5000):
        yt = rng.randint(0, 8, size=n)
        yp = np.where(rng.rand(n) < 0.6, yt, rng.randint(0, 8, size=n))
        labels = [0, 1, 2, 3, 5, 7]
        tp, fp, fn = esi_counts_ref(yt, yp, labels)
        cases.append({"y_true": yt.tolist(), "y_pred": yp.tolist(), "labels": labels,
                      "tp": tp.tolist(), "fp": fp.tolist(), "fn": fn.tolist(),
                      "esi": esi_score_ref(yt, yp, labels)})
    return cases


if __name__ == "__main__":
    assert harness.reference_available(), "set UNETSULC_REFERENCE to a checkout of the reference"
    json.dump(plateau_traces(), open(os.path.join(HERE, "plateau_traces.json"), "w"))
    np.savez_compressed(os.path.join(HERE, "dataset_cases.npz"), **dataset_cases())
    json.dump(reference_training(), open(os.path.join(HERE, "reference_training.json"), "w"), indent=1)
    np.savez_compressed(os.path.join(HERE, "oracle_unet3d.npz"), **oracle_unet3d())
    np.savez_compressed(os.path.join(HERE, "cutting_cases.npz"), **cutting_cases())
    json.dump(esi_cases(), open(os.path.join(HERE, "esi_cases.json"), "w"))
    print("golden fixtures written to", HERE)
