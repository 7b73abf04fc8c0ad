"""BASELINE.json configs[0] / north_star "main.py and the MLflow logging run unchanged", compared with what the
reference's driver (`main.py`, unmodified) logged when it ran on the reference's own `coda` package on CPU
(`tests/golden/cfg1_main_py.json`, made by `tests/golden/make_cfg1_golden.py` with the recording MLflow stand-in
`tests/stubs/mlflow`, since MLflow is not a dependency of this package).

The selection loop of main.py, written against the `coda` shim the way main.py imports it, runs on the GPU and must
reproduce the logged trajectory.  The driver script itself is not part of this repository (reference sources are never
copied in); where $CODA_REFERENCE_MAIN or $CODA_REFERENCE_PATH/main.py names it, the driver also runs unchanged as a
subprocess against THIS package, and its MLflow calls are checked too.
"""
import argparse
import json
import os
import random
import sys

import numpy as np
import pytest
import torch

from helpers import GOLDEN, ROOT

pytestmark = pytest.mark.gpu

sys.path.insert(0, GOLDEN)


def _main_py():
    ref = os.environ.get("CODA_REFERENCE_PATH")
    cands = [os.environ.get("CODA_REFERENCE_MAIN"), ref and os.path.join(ref, "main.py")]
    for c in cands:
        if c and os.path.exists(c):
            return c
    return None


def _run(tmp_path, extra_env=None, iters=None):
    import make_cfg1_golden as mk
    main_py = _main_py()
    if main_py is None:
        pytest.skip("the reference driver main.py is not available (set CODA_REFERENCE_MAIN)")
    gpath = os.path.join(GOLDEN, "cfg1_main_py.json")
    if not os.path.exists(gpath):
        pytest.skip("cfg1 golden not generated")
    g = json.load(open(gpath))
    iters = iters or g["iters"]
    d = str(tmp_path)
    mk.write_task(d)
    log = os.path.join(d, "mlflow.jsonl")
    # PYTHONSAFEPATH keeps the script's directory (the reference checkout, with ITS coda package) off sys.path:
    # `from coda import CODA` resolves to this repository's shim
    r = mk.run_main(main_py, d, iters, log, [ROOT, os.path.join(ROOT, "tests", "stubs")], extra_env=extra_env, safe_path=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    out = mk.parse_log(log)
    return g, out, r.stdout


def _compare(g, out, stdout, iters):
    assert "device is cuda" in stdout and "Loaded preds of shape torch.Size([80, 10000, 10])" in stdout
    # MLflow plumbing of main.py:132-164: experiment run + nested seed run, parameters, per-step metrics
    assert out["runs"] == g["runs"] == [["cifar10_5592-coda", False], ["cifar10_5592-coda-0", True]]
    assert out["params"]["method"] == "coda" and out["params"]["task"] == "cifar10_5592"
    assert ["seed", 0] in out["seed_params"] and "stochastic" in [k for k, _ in out["seed_params"]]
    return _compare_trajectory(g, out, iters)


def _compare_trajectory(g, out, iters):
    assert len(out["regret"]) == len(out["cumulative_regret"]) == len(out["chosen_idx"]) == iters
    # the selection trajectory (main.py:91-103): items, revealed classes, predicted best model, regret.  Free-running
    # index parity is ill-conditioned where the reference's own top candidates are within fp32 noise (SURVEY.md 8c-3):
    # the trajectories must be identical up to the first such step, and there our pick must be epsilon-optimal under
    # the REFERENCE's scores (golden["top"]: the reference's top candidates of every step along its trajectory).
    ref_idx = g["chosen_idx"][:iters]
    same = 0
    while same < iters and out["chosen_idx"][same] == ref_idx[same]:
        same += 1
    assert out["true_class"][:same] == g["true_class"][:same]
    assert out["best_model"][:same] == g["best_model"][:same]
    np.testing.assert_allclose(out["regret"][:same], g["regret"][:same], atol=1e-7)
    np.testing.assert_allclose(out["cumulative_regret"][:same], g["cumulative_regret"][:same], atol=1e-6)
    if same < iters:
        assert "top" in g, "golden has no reference scores to judge the divergence at step %d" % same
        top = dict((int(i), float(v)) for i, v in g["top"][same])
        best = max(top.values())
        ours = out["chosen_idx"][same]
        assert ours in top and top[ours] >= best - 5e-6, (same, ours, g["top"][same][:4])
        assert top[ref_idx[same]] >= best - 5e-6
    return same


def test_reference_main_py_runs_unchanged_on_one_gpu(tmp_path):
    g, out, stdout = _run(tmp_path)
    keep = os.environ.get("CODA_B200_KEEP_MAIN_LOG")
    if keep:
        with open(keep, "w") as f:
            f.write(stdout[-6000:])
            f.write("\n--- mlflow stub log (parsed) ---\n" + json.dumps(out)[:4000] + "\n")
    same = _compare(g, out, stdout, g["iters"])
    if keep:
        with open(keep, "a") as f:
            f.write("identical to the reference's CPU run of the same driver for the first %d of %d steps\n" % (same, g["iters"]))


def test_reference_main_py_runs_unchanged_on_all_gpus(tmp_path):
    """Same driver, same command line; CODA_B200_GPUS in the environment makes the selector shard the slab over the
    GPUs of the box from inside the one process main.py starts (SURVEY.md 8e process model)."""
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    g, out, stdout = _run(tmp_path, extra_env={"CODA_B200_GPUS": str(min(n, 8))}, iters=10)
    _compare(g, out, stdout, 10)


def test_main_py_selection_loop_through_the_shim_matches_the_reference(tmp_path, capsys):
    """main.py:55-105 for --method coda --seeds 1 (seed_all, true losses, the four calls per step, regret
    bookkeeping) against the `coda` shim, on the task file main.py read; needs no reference checkout."""
    import make_cfg1_golden as mk
    from coda import CODA
    from coda.datasets import Dataset
    from coda.options import LOSS_FNS
    from coda.oracle import Oracle
    g = json.load(open(os.path.join(GOLDEN, "cfg1_main_py.json")))
    mk.write_task(str(tmp_path))
    args = argparse.Namespace(**g["params"])
    dataset = Dataset(str(tmp_path / (args.task + ".pt")), device=torch.device("cuda:0"))
    assert "Loaded preds of shape torch.Size([80, 10000, 10])" in capsys.readouterr().out
    oracle = Oracle(dataset, loss_fn=LOSS_FNS[args.loss])
    random.seed(0); np.random.seed(0); torch.manual_seed(0); torch.cuda.manual_seed_all(0)
    true_losses = oracle.true_losses(dataset.preds)
    best_loss = min(true_losses)
    selector = CODA.from_args(dataset, args)
    selector.get_best_model_prediction()
    out = {"regret": [], "cumulative_regret": [], "chosen_idx": [], "true_class": [], "best_model": []}
    cumulative = 0
    for _ in range(args.iters):
        chosen_idx, selection_prob = selector.get_next_item_to_label()
        true_class = oracle(chosen_idx)
        selector.add_label(chosen_idx, true_class, selection_prob)
        best = selector.get_best_model_prediction()
        regret = true_losses[best] - best_loss
        cumulative += regret
        out["regret"].append(float(regret)); out["cumulative_regret"].append(float(cumulative))
        out["chosen_idx"].append(int(chosen_idx)); out["true_class"].append(int(true_class))
        out["best_model"].append(int(best))
    same = _compare_trajectory(g, out, args.iters)
    if same == args.iters:
        assert ["stochastic", selector.stochastic] in g["seed_params"]
