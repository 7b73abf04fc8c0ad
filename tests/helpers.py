"""Shared test helpers: golden loading and oracle access (tests are the only oracle users)."""
import glob
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import coda_oracle  # noqa: E402
from coda_b200.synth import synth  # noqa: E402


def golden_names(prefix="traj_"):
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, prefix + "*.npz")))


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    g = {k: z[k] for k in z.files}
    g["ctor"] = {}
    for k, v in zip(g["ctor_keys"].tolist(), g["ctor_vals"].tolist()):
        g["ctor"][k] = bool(v) if k == "disable_diag_prior" else (int(v) if k == "prefilter_n" else float(v))
    if "final_dirichlets" not in g and "init_dirichlets" in g:
        g["final_dirichlets"] = final_dirichlets(g)
    return g


def final_dirichlets(g):
    """The posterior after the trajectory: a label of class t rewrites only dirichlets[:, t] (coda.py:316-317), and
    dir_row holds that column after every step, so a fixture need not store the whole H x C x C array twice."""
    d = g["init_dirichlets"].copy()
    for k, i in enumerate(g["idx"]):
        d[:, g["labels"][i]] = g["dir_row"][k]
    return d


def golden_slab(g):
    preds, labels = synth(int(g["H"]), int(g["N"]), int(g["C"]), int(g["data_seed"]), dense=bool(g["dense"]))
    assert np.array_equal(labels.numpy(), g["labels"])
    return preds, labels
