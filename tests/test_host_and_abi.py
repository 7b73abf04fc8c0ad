"""CPU-only tests: the C-ABI library loads and exports every declared symbol, host-side logic."""
import ctypes
import os
import random
import re

import numpy as np
import pytest
import torch

from helpers import ROOT


def test_library_exports_every_declared_symbol():
    from coda_b200 import _native as nat
    lib = nat.load()
    hdr = open(os.path.join(ROOT, "include", "coda_b200.h")).read()
    declared = set(re.findall(r"\b(coda_b200_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/coda_b200.h but not exported"
    assert declared == set(nat.SIGNATURES), declared ^ set(nat.SIGNATURES)
    assert lib.coda_b200_version() == nat.VERSION == 202
    raw = ctypes.CDLL(nat.lib_path())
    assert raw.coda_b200_version() == 202


def test_no_gpu_means_loud_failure():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from coda_b200 import CODA, TensorDataset, _native as nat
    with pytest.raises(nat.NativeError, match="no CUDA device"):
        nat.require_device()
    with pytest.raises(RuntimeError, match="no CPU path"):
        CODA(TensorDataset(torch.rand(2, 8, 3).softmax(-1)))


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "coda_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "coda_oracle" not in src and "oracle/" not in src, f
    for f in os.listdir(os.path.join(ROOT, "coda")):
        if f.endswith(".py"):
            assert "coda_oracle" not in open(os.path.join(ROOT, "coda", f)).read()


def test_merge_rule_and_tie_choice():
    from coda_b200.dist import IDX_NONE, choose_among_ties, merge_records
    recs = [(0.5, 10, 3, 0.7, 2), (0.5, 4, 1, 0.7, 9), (float("-inf"), IDX_NONE, 0, 0.1, 1)]
    assert merge_records(recs) == (0.5, 4, 4, 0.7, 2)
    # random.choice(list) and random.choice(range(len)) consume the RNG identically (coda.py:308)
    ties = [41, 7, 19]
    random.seed(3)
    a = choose_among_ties(ties, random)
    s1 = random.getstate()
    random.seed(3)
    b = sorted(ties)[random.choice([0, 1, 2])]
    assert a == b and s1 == random.getstate()


def test_unlabeled_view_semantics():
    from coda_b200.selector import _Unlabeled
    seen = []
    u = _Unlabeled(0, 10, seen.append)
    u.remove(3)
    assert len(u) == 9 and 3 not in u and 4 in u and list(u)[:4] == [0, 1, 2, 4] and seen == [3]
    with pytest.raises(ValueError):
        u.remove(3)
    with pytest.raises(ValueError):
        u.remove(10)


def test_synth_is_shard_invariant_and_argmax_clean():
    from coda_b200.synth import shard_range, synth
    full, y = synth(6, 1000, 5, seed=3)
    parts = [synth(6, 1000, 5, seed=3, n_lo=lo, n_hi=hi)[0] for lo, hi in (shard_range(1000, r, 3) for r in range(3))]
    assert torch.equal(torch.cat(parts, 1), full)
    assert torch.allclose(full.sum(-1), torch.ones(6, 1000), atol=1e-5)
    top2 = full.topk(2, -1).values
    assert float((top2[..., 0] - top2[..., 1]).min()) > 0


def test_coda_shim_exports_reference_names():
    import coda
    from coda.base import ModelSelector
    from coda.baselines import IID, ActiveTesting, ModelPicker, Uncertainty, VMA  # noqa: F401  (main.py:10)
    from coda.options import LOSS_FNS
    assert issubclass(coda.CODA, ModelSelector) and "acc" in LOSS_FNS
    with pytest.raises(NotImplementedError):
        IID(None, None)


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from coda_b200.dist import TorchComm, merge_records
    comm = TorchComm()
    # 1. arg-max exchange: every rank contributes one record, all ranks merge to the same global record
    rec = torch.tensor([[0.25, 7, 2, 0.5, 3], [0.25, 5, 1, 0.4, 8]][rank], dtype=torch.float64)
    allr = comm.allgather(rec)
    merged = merge_records([tuple(r.tolist()) for r in allr])
    # 2. construction: SUM all-reduce of the soft-confusion sums (coda.py:42), int64 fixed point
    jvec = torch.tensor([3, 1, 4, 1, 5], dtype=torch.int64) if rank == 1 else torch.zeros(5, dtype=torch.int64)
    comm.allreduce_sum_(jvec)
    # 3. marginals: exact int64 sums
    pis = torch.tensor([2 ** 40 + rank, 5], dtype=torch.int64)
    comm.allreduce_sum_(pis)
    mn = torch.tensor([100 + rank], dtype=torch.int64)
    comm.allreduce_min_(mn)
    q.put((rank, merged, jvec.tolist(), pis.tolist(), int(mn)))
    dist.destroy_process_group()


def test_sharded_exchanges_world2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + random.randint(0, 2000)
    ps = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in ps]
    out = sorted(q.get(timeout=120) for _ in ps)
    [p.join(60) for p in ps]
    for rank, merged, jvec, pis, mn in out:
        assert merged == (0.25, 5, 3, 0.5, 3)
        assert jvec == [3, 1, 4, 1, 5]
        assert pis == [2 ** 41 + 1, 10] and mn == 100


def test_sharded_file_dataset_reads_only_its_range(tmp_path):
    from coda_b200 import ShardedFileDataset
    from coda_b200.synth import shard_range, synth
    preds, labels = synth(5, 333, 4, seed=2)
    f = str(tmp_path / "task.pt")
    torch.save(preds.half(), f)                      # the loader forces fp32 like coda/datasets.py:14
    torch.save(labels, f.replace(".pt", "_labels.pt"))
    parts = []
    for r in range(3):
        ds = ShardedFileDataset(f, "cpu", rank=r, world=3)
        lo, hi = shard_range(333, r, 3)
        assert (ds.n_offset, ds.n_global, ds.preds.shape[1]) == (lo, 333, hi - lo)
        assert ds.preds.dtype == torch.float32 and ds.preds.is_contiguous() and torch.equal(ds.labels, labels)
        parts.append(ds.preds)
    assert torch.equal(torch.cat(parts, 1), preds.half().float())


def test_ctypes_signatures_match_header_arity():
    """Every declaration in include/coda_b200.h and its ctypes binding take the same number of arguments."""
    from coda_b200 import _native as nat
    hdr = open(os.path.join(ROOT, "include", "coda_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    for name, (_res, args) in nat.SIGNATURES.items():
        m = re.search(r"\b" + name + r"\s*\(([^;]*?)\)\s*;", hdr, flags=re.S)
        assert m, name
        params = m.group(1).strip()
        n = 0 if params in ("", "void") else params.count(",") + 1
        assert n == len(args), (name, n, len(args))


# Stands in for the reference's main.py where no checkout is given: the same imports from `coda`, and the calls main.py
# makes before its loop (main.py:114-118, 57-67), reading --task / --data-dir from the same command line.
_MAIN_PY_STAND_IN = """
import argparse, os
import mlflow  # noqa: F401
import torch
from coda import CODA
from coda.baselines import IID, ActiveTesting, VMA, ModelPicker, Uncertainty  # noqa: F401
from coda.datasets import Dataset
from coda.options import LOSS_FNS
from coda.oracle import Oracle
cli = argparse.ArgumentParser()
cli.add_argument("--task")
cli.add_argument("--data-dir")
a, _ = cli.parse_known_args()
ds = Dataset(os.path.join(a.data_dir, a.task + ".pt"), device=torch.device("cuda" if torch.cuda.is_available() else "cpu"))
print("Best possible loss is", min(Oracle(ds, loss_fn=LOSS_FNS["acc"]).true_losses(ds.preds)))
CODA.from_args(ds, argparse.Namespace(prefilter_n=0, alpha=0.9, learning_rate=0.01, multiplier=2.0, no_diag_prior=False,
                                      q="eig"))
"""


def test_reference_main_py_resolves_to_this_package(tmp_path):
    """INTEGRATION.md section 1, as far as a machine without a GPU can check it: the reference's driver, run with this
    repository first on PYTHONPATH, imports OUR coda package, loads the task through our Dataset / Oracle / LOSS_FNS and
    reaches CODA.from_args -- where the missing GPU is reported loudly instead of falling back to a CPU path.  The
    driver is the unmodified main.py of the checkout CODA_REFERENCE_PATH names, else a stand-in making the same calls."""
    import subprocess
    import sys
    if torch.cuda.is_available():
        pytest.skip("GPU present: main.py would run to completion")
    ref = os.environ.get("CODA_REFERENCE_PATH")
    main_py = os.path.join(ref, "main.py") if ref else ""
    if not os.path.exists(main_py):
        main_py = str(tmp_path / "main.py")
        with open(main_py, "w") as f:
            f.write(_MAIN_PY_STAND_IN)
    from coda_b200.synth import synth
    preds, labels = synth(6, 200, 4, seed=1)
    torch.save(preds, str(tmp_path / "toy.pt"))
    torch.save(labels, str(tmp_path / "toy_labels.pt"))
    stubs = tmp_path / "stubs"
    (stubs / "mlflow").mkdir(parents=True)
    (stubs / "mlflow" / "__init__.py").write_text("def set_tracking_uri(*a, **k):\n    pass\n")   # main.py:17 runs at import
    # PYTHONSAFEPATH: keep the script's own directory (the reference checkout) off sys.path[0] so `coda` is ours
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, str(stubs)]), PYTHONSAFEPATH="1")
    r = subprocess.run([sys.executable, main_py, "--task", "toy", "--data-dir", str(tmp_path),
                        "--method", "coda", "--seeds", "1", "--iters", "2", "--no-mlflow"],
                       capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=300)
    out = r.stdout + r.stderr
    best_loss = (preds.argmax(-1) != labels[None]).float().mean(1).min()
    assert "Loaded preds of shape torch.Size([6, 200, 4])" in out          # our Dataset (coda/datasets.py contract)
    assert f"Best possible loss is {best_loss!s}" in out, out[-2000:]        # our Oracle.true_losses + LOSS_FNS['acc']
    assert r.returncode != 0 and "no CPU path" in out, out[-2000:]          # our CODA: loud, no fallback


def test_merge_rule_is_shard_count_invariant_property():
    """hypothesis: merging per-shard arg-max records in any grouping / order gives the global record (max value,
    lowest index on equal values, counts summed) -- what makes the selected item independent of the shard count."""
    from hypothesis import given, settings, strategies as st
    from coda_b200.dist import IDX_NONE, merge_records

    vals = st.sampled_from([0.0, 0.125, 0.25, 0.25, 0.5])          # few distinct values -> many exact ties

    @settings(max_examples=200, deadline=None)
    @given(st.lists(st.tuples(vals, st.booleans()), min_size=1, max_size=40), st.integers(1, 8), st.randoms())
    def check(items, nshards, rnd):
        # item i: value v, candidate flag a (set A = candidates, set B = all)
        def rec(idxs):
            va, ia, ca, vb, ib = float("-inf"), IDX_NONE, 0, float("-inf"), IDX_NONE
            for i in idxs:
                v, a = items[i]
                if v > vb or (v == vb and i < ib):
                    vb, ib = v, i
                if a:
                    ca += 1
                    if v > va or (v == va and i < ia):
                        va, ia = v, i
            return (va, ia, ca, vb, ib)
        whole = rec(range(len(items)))
        bounds = sorted(rnd.sample(range(len(items) + 1), min(nshards - 1, len(items) + 1)))
        cuts = [0] + bounds + [len(items)]
        shards = [rec(range(cuts[k], cuts[k + 1])) for k in range(len(cuts) - 1)]
        rnd.shuffle(shards)
        assert merge_records(shards) == whole
        half = len(shards) // 2                                       # tree merge == flat merge
        assert merge_records([merge_records(shards[:half] or [shards[0]]), merge_records(shards[half:])]) == \
            merge_records((shards[:half] or [shards[0]]) + shards[half:])
    check()


def test_shard_ranges_partition_the_item_axis_property():
    from hypothesis import given, settings, strategies as st
    from coda_b200.synth import shard_range

    @settings(max_examples=200, deadline=None)
    @given(st.integers(0, 10 ** 7), st.integers(1, 64))
    def check(n, world):
        r = [shard_range(n, k, world) for k in range(world)]
        assert r[0][0] == 0 and r[-1][1] == n
        assert all(r[k][1] == r[k + 1][0] for k in range(world - 1))
        sizes = [hi - lo for lo, hi in r]
        assert max(sizes) - min(sizes) <= 1
    check()


def test_baseline_selectors_resolve_to_the_reference_when_pointed_at_it(tmp_path):
    """coda/baselines is out of scope (SURVEY section 2); with CODA_REFERENCE_PATH set the shim serves the classes of
    that checkout so `main.py --method iid|uncertainty|...` keeps working next to our CODA.  A stand-in checkout with
    the reference's layout (one module per selector under coda/baselines) is enough to check the resolution."""
    import subprocess
    import sys
    base = tmp_path / "coda" / "baselines"
    base.mkdir(parents=True)
    for cls, mod in (("IID", "iid"), ("ActiveTesting", "activetesting"), ("VMA", "vma"), ("ModelPicker", "modelpicker"),
                     ("Uncertainty", "uncertainty")):
        (base / (mod + ".py")).write_text(f"class {cls}:\n    def __init__(self, dataset, loss_fn):\n"
                                          f"        self.dataset, self.loss_fn = dataset, loss_fn\n")
    code = (
        "import inspect\n"
        "from coda.baselines import IID, ActiveTesting, VMA, ModelPicker, Uncertainty\n"
        "from coda.options import LOSS_FNS\n"
        "s = Uncertainty('task', LOSS_FNS['acc'])\n"
        "print('OK', IID.__module__, inspect.getfile(VMA), s.dataset, s.loss_fn is LOSS_FNS['acc'])\n")
    env = dict(os.environ, PYTHONPATH=ROOT, CODA_REFERENCE_PATH=str(tmp_path))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0 and f"OK coda.baselines.iid {base / 'vma.py'} task True" in r.stdout, \
        r.stdout + r.stderr[-1500:]


def test_best2_merge_matches_a_flat_scan_property():
    """hypothesis: the (value, lowest index, runner-up value) records of csrc/common.cuh (host mirror dist.merge_best2)
    merged over any partition equal one flat scan -- the runner-up is what lets the host-free loop flag an isclose tie."""
    from hypothesis import given, settings, strategies as st
    from coda_b200.dist import IDX_NONE, merge_best2

    vals = st.sampled_from([0.0, 0.125, 0.25, 0.25, 0.5, 0.5])

    @settings(max_examples=300, deadline=None)
    @given(st.lists(vals, min_size=1, max_size=30), st.integers(1, 6), st.randoms())
    def check(items, nshards, rnd):
        def flat(idxs):
            idxs = list(idxs)
            if not idxs:
                return (float("-inf"), IDX_NONE, float("-inf"))
            best = max(idxs, key=lambda i: (items[i], -i))
            rest = [items[i] for i in idxs if i != best]
            return (items[best], best, max(rest) if rest else float("-inf"))
        whole = flat(range(len(items)))
        bounds = sorted(rnd.sample(range(len(items) + 1), min(nshards - 1, len(items) + 1)))
        cuts = [0] + bounds + [len(items)]
        shards = [flat(range(cuts[k], cuts[k + 1])) for k in range(len(cuts) - 1)]
        rnd.shuffle(shards)
        assert merge_best2(shards) == whole
    check()


def test_compact_slab_densify_and_generator():
    from coda_b200 import CompactSlab
    from coda_b200.synth import shard_range, synth_compact
    ids, probs, labels = synth_compact(9, 500, 40, 4, seed=2)
    slab = CompactSlab(ids, probs, 40)
    dense = slab.densify()
    assert dense.shape == (9, 500, 40) and torch.allclose(dense.sum(-1), torch.ones(9, 500), atol=1e-5)
    assert float(dense.min()) >= 0 and torch.equal(dense.argmax(-1), ids[..., 0].long())
    assert bool((probs[..., :-1] >= probs[..., 1:]).all())                       # descending scores
    assert bool((dense.gather(2, ids.long()) == probs).all())                    # listed classes carry their scores
    rest = dense.sum(-1) - probs.sum(-1)
    assert bool((rest > 0).all())                                                 # some mass is always spread
    # shard invariance of the generator and N-range views
    parts = [synth_compact(9, 500, 40, 4, seed=2, n_lo=lo, n_hi=hi) for lo, hi in (shard_range(500, r, 3) for r in range(3))]
    assert torch.equal(torch.cat([p[0] for p in parts], 1), ids) and torch.equal(torch.cat([p[1] for p in parts], 1), probs)
    v = slab.narrow_items(100, 200)
    assert v.shape == (9, 100, 40) and torch.equal(v.densify(), dense[:, 100:200])
    with pytest.raises(TypeError):
        CompactSlab(ids.long(), probs, 40)
