"""fp16 prediction slabs: kept fp16 on the device, every result bit-identical to the run on the fp32 upcast.

Every GPU comparison is exact (torch.equal / np.array_equal) between a selector on ``p16`` and one on ``p16.float()``
built in the same process.  The CPU tier covers the loaders' ``keep_fp16`` rule and the shadow sizing.
"""
import argparse
import os
import random

import numpy as np
import pytest
import torch

from helpers import golden_slab, load_golden

gpu = pytest.mark.gpu
GOLDENS = ["traj_small_h32_n3000_c10", "traj_nodiag_h10_n400_c6", "traj_dense_h16_n500_c12", "traj_c100_h24_n400_c100",
           "traj_h256_h256_n1500_c100"]


def _sel(preds, labels=None, **kw):
    from coda_b200 import CODA, TensorDataset
    dev = torch.device("cuda:0")
    return CODA(TensorDataset(preds.to(dev), None if labels is None else labels.to(dev)), **kw)


def _pair(p16, labels=None, **kw):
    """Selectors on the fp16 slab and on its fp32 upcast (same values)."""
    p16 = p16.to("cuda:0")
    a = _sel(p16, labels, **kw)
    b = _sel(p16.float(), labels, **kw)
    assert a.engine.preds.dtype == torch.float16 and b.engine.preds.dtype == torch.float32
    return a, b


def _eq(x, y, what):
    assert x.dtype == y.dtype and x.shape == y.shape, what
    assert torch.equal(x.cpu(), y.cpu()), what


def _same_state(a, b, where=""):
    _eq(a.dirichlets, b.dirichlets, f"dirichlets {where}")
    _eq(a.pi_hat, b.pi_hat, f"pi_hat {where}")
    _eq(a.pi_hat_xi, b.pi_hat_xi, f"pi_hat_xi {where}")
    _eq(a.get_pbest(), b.get_pbest(), f"pbest {where}")
    assert int(a.get_best_model_prediction()) == int(b.get_best_model_prediction()), where


def _api_lockstep(a, b, labels, steps):
    """Free-running API loop on both selectors; the python RNG is replayed so a tie draws the same item on both."""
    labels = labels.cpu()
    for k in range(steps):
        st = random.getstate()
        ia, qa = a.get_next_item_to_label()
        random.setstate(st)
        ib, qb = b.get_next_item_to_label()
        assert (ia, np.float32(qa)) == (ib, np.float32(qb)), f"step {k}"
        _eq(a.eig, b.eig, f"eig step {k}")
        a.add_label(ia, int(labels[ia]), qa)
        b.add_label(ib, int(labels[ib]), qb)
        _same_state(a, b, f"step {k}")
    assert a.labeled_idxs == b.labeled_idxs


def _half_slab(name):
    g = load_golden(name)
    preds, labels = golden_slab(g)
    return preds.half(), labels, g


# ---------------------------------------------------------------------------------------------- 1. API path
@gpu
@pytest.mark.parametrize("mode", ["incremental", "recompute", "recompute_all"])
@pytest.mark.parametrize("name", GOLDENS)
def test_api_loop_fp16_equals_fp32_upcast(name, mode):
    p16, labels, g = _half_slab(name)
    random.seed(0)
    a, b = _pair(p16, labels, mode=mode, **g["ctor"])
    _same_state(a, b, "construction")
    assert torch.equal(a.engine.hard.cpu(), b.engine.hard.cpu())
    _api_lockstep(a, b, labels, 30)
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------- 2. host-free loop
@gpu
@pytest.mark.parametrize("graph", ["1", "0"])
def test_run_steps_fp16_equals_fp32_upcast(graph, monkeypatch):
    monkeypatch.setenv("CODA_B200_GRAPH", graph)
    p16, labels, _g = _half_slab("traj_c100_h24_n400_c100")
    a, b = _pair(p16, labels)
    for k in (1, 20, 19):
        a.run_steps(k, labels)
        b.run_steps(k, labels)
    for x, y in zip(a.history(), b.history()):
        assert np.array_equal(x, y)
    assert len(a.history()[0]) == 40
    _same_state(a, b, "after run_steps")
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------- 3. shards
@gpu
@pytest.mark.parametrize("shards", [2, 3])
def test_fp16_shards_equal_one_fp32_shard(shards):
    from coda_b200.synth import synth
    preds, labels = synth(24, 1001, 100, seed=5)          # odd N: item-range views with odd offsets
    p16 = preds.half().to("cuda:0")
    a = _sel(p16, labels, shards=shards, gpus=1)
    b = _sel(p16.float(), labels, shards=1)
    assert len(a.engines) == shards and all(e.preds.dtype == torch.float16 for e in a.engines)
    a.run_steps(25, labels)
    b.run_steps(25, labels)
    for x, y in zip(a.history(), b.history()):
        assert np.array_equal(x, y)
    _same_state(a, b, "sharded")
    a.close(); b.close()


@gpu
def test_fp16_two_gpus_equal_one_fp32_shard():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from coda_b200.synth import synth
    preds, labels = synth(24, 1001, 100, seed=5)
    p16 = preds.half().to("cuda:0")
    a = _sel(p16, labels, gpus=2)
    b = _sel(p16.float(), labels, gpus=1)
    assert all(e.preds.dtype == torch.float16 for e in a.engines)
    a.run_steps(25, labels)
    b.run_steps(25, labels)
    for x, y in zip(a.history(), b.history()):
        assert np.array_equal(x, y)
    _same_state(a, b, "2 GPUs")
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------- 4. kernel coverage
@gpu
@pytest.mark.parametrize("pi_full", ["simt", "tc"])
def test_marginal_pass_variants(pi_full, monkeypatch):
    monkeypatch.setenv("CODA_B200_PI_FULL", pi_full)
    p16, labels, _g = _half_slab("traj_h256_h256_n1500_c100")
    a, b = _pair(p16, labels, mode="recompute_all")
    assert a.engine._pi_tc == b.engine._pi_tc == (pi_full == "tc")
    _api_lockstep(a, b, labels, 6)
    a.close(); b.close()


@gpu
@pytest.mark.parametrize("H,N,C", [(12, 600, 150), (20, 701, 18), (9, 333, 10)])
def test_generic_and_non_tensor_core_shapes(H, N, C):
    """C = 150: the generic confusion / pass kernels (C > 128); C = 18 and C = 10 fail pi_full_tc_ok."""
    from coda_b200 import _native as nat
    from coda_b200.synth import synth
    preds, labels = synth(H, N, C, seed=H + C)
    p16 = preds.half()
    lib = nat.load()
    assert bool(lib.coda_b200_pi_full_tc_ok_f16(H, N, C, N * C)) == bool(lib.coda_b200_pi_full_tc_ok(H, N, C, N * C))
    for mode in ("incremental", "recompute_all"):
        random.seed(1)
        a, b = _pair(p16, labels, mode=mode)
        assert a.engine._pi_tc == b.engine._pi_tc == (16 <= C <= 128 and C % 4 == 0)
        _api_lockstep(a, b, labels, 8)
        a.close(); b.close()


@gpu
@pytest.mark.parametrize("shadow", ["off", "partial", "full"])
def test_rank1_refresh_with_and_without_shadow(shadow, monkeypatch):
    if shadow == "off":
        monkeypatch.setenv("CODA_B200_SHADOW", "0")
    elif shadow == "partial":
        monkeypatch.setenv("CODA_B200_SHADOW_MODELS", "5")
    p16, labels, _g = _half_slab("traj_c100_h24_n400_c100")
    a, b = _pair(p16, labels)
    want = {"off": 0, "partial": 5, "full": 24}[shadow]
    assert a.engine.n_shadow == b.engine.n_shadow == want
    if want:
        assert a.engine.shadow.dtype == torch.float16 and b.engine.shadow.dtype == torch.float32
        assert a.engine.shadow_cs % 8 == 0
    a.run_steps(30, labels)
    b.run_steps(30, labels)
    for x, y in zip(a.history(), b.history()):
        assert np.array_equal(x, y)
    _same_state(a, b, shadow)
    a.close(); b.close()


@gpu
@pytest.mark.parametrize("r1", ["v1d", "v4", "tma"])
def test_rank1_opt_in_variants(r1, monkeypatch):
    """v1d has an fp16 instantiation with the same bits; v4 / tma read fp32 words and refuse a 16-bit slab."""
    from coda_b200._native import NativeError
    monkeypatch.setenv("CODA_B200_R1", r1)
    p16, labels, _g = _half_slab("traj_c100_h24_n400_c100")
    if r1 != "v1d":
        with pytest.raises(NativeError, match="not available for a 16-bit slab"):
            _sel(p16, labels).run_steps(2, labels)
        return
    a, b = _pair(p16, labels)
    a.run_steps(10, labels)
    b.run_steps(10, labels)
    _same_state(a, b, r1)
    a.close(); b.close()


@gpu
@pytest.mark.parametrize("lo", [0, 1, 77])
def test_item_range_view_of_a_larger_fp16_slab(lo):
    """model stride != N * C, and (odd lo) an item offset that is not 16-byte aligned in fp16."""
    from coda_b200 import CODA, TensorDataset
    from coda_b200.synth import synth
    preds, labels = synth(24, 1200, 100, seed=9)
    big16 = preds.half().to("cuda:0")
    big32 = big16.float()
    hi = lo + 901
    lab = labels[lo:hi].to("cuda:0")
    a = CODA(TensorDataset(big16[:, lo:hi], lab))
    b = CODA(TensorDataset(big32[:, lo:hi], lab))
    assert a.engine.model_stride == 1200 * 100
    assert a.engine._pi_tc == b.engine._pi_tc
    _api_lockstep(a, b, lab, 10)
    a.close(); b.close()


@gpu
def test_fp16_shadow_twice_the_models_for_the_same_memory(monkeypatch):
    """Both engines are shown the same free memory (10 fp32 slots, nothing reserved): the fp16 shadow takes 20 slots."""
    from coda_b200.synth import synth
    preds, labels = synth(64, 1000, 100, seed=3)
    p16 = preds.half().to("cuda:0")
    p32 = p16.float()
    real = torch.cuda.mem_get_info
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda dev=None: (10 * 1000 * 100 * 4, real(dev)[1]))
    monkeypatch.setenv("CODA_B200_SHADOW_RESERVE_GB", "0")
    b = _sel(p32, labels, mode="recompute")
    a = _sel(p16, labels, mode="recompute")
    assert b.engine.n_shadow == 10 and b.engine.shadow.dtype == torch.float32
    assert a.engine.n_shadow == 20 and a.engine.shadow.dtype == torch.float16
    assert a.engine.shadow.numel() * 2 == b.engine.shadow.numel() * 4
    monkeypatch.setattr(torch.cuda, "mem_get_info", real)
    a.run_steps(10, labels)
    b.run_steps(10, labels)
    _same_state(a, b, "shadows of different width")
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------- 5. guards
@gpu
@pytest.mark.parametrize("bad", ["nan", "inf", "negative"])
def test_bad_values_raise_the_same_errors(bad):
    from coda_b200.synth import synth
    preds, _ = synth(8, 300, 10, seed=2)
    p16 = preds.half()
    p16[3, 17, 4] = {"nan": float("nan"), "inf": float("inf"), "negative": -0.25}[bad]
    errs = []
    for p in (p16, p16.float()):
        with pytest.raises((RuntimeError, ValueError)) as ei:
            _sel(p)
        errs.append((type(ei.value), str(ei.value)))
    assert errs[0] == errs[1]


@gpu
def test_bf16_slab_raises_type_error():
    from coda_b200.synth import synth
    preds, _ = synth(8, 300, 10, seed=2)
    with pytest.raises(TypeError):
        _sel(preds.bfloat16())


# ---------------------------------------------------------------------------------------------- 6. checkpoint
@gpu
@pytest.mark.parametrize("first", ["fp16", "fp32"])
def test_state_dict_crosses_element_types(first):
    p16, labels, g = _half_slab("traj_c100_h24_n400_c100")
    p16 = p16.to("cuda:0")
    slabs = {"fp16": p16, "fp32": p16.float()}
    second = "fp32" if first == "fp16" else "fp16"
    random.seed(0)
    ref = _sel(slabs[second], labels, **g["ctor"])            # uninterrupted run on the other element type
    random.seed(0)
    x = _sel(slabs[first], labels, **g["ctor"])
    _api_lockstep(x, ref, labels, 8)
    sd = x.state_dict()
    x.close()
    y = _sel(slabs[second], labels, **g["ctor"])
    y.load_state_dict(sd)
    _same_state(y, ref, "resumed")
    _api_lockstep(y, ref, labels, 8)
    y.close(); ref.close()


# ---------------------------------------------------------------------------------------------- 7. drop-in
def _main_py_loop(path, iters=8):
    from coda import CODA
    from coda.datasets import Dataset
    from coda.options import LOSS_FNS
    from coda.oracle import Oracle
    args = argparse.Namespace(prefilter_n=0, alpha=0.9, learning_rate=0.01, multiplier=2.0, no_diag_prior=False, q="eig",
                              iters=iters)
    dataset = Dataset(path, device=torch.device("cuda:0"))                              # main.py:114
    oracle = Oracle(dataset, loss_fn=LOSS_FNS["acc"])                                   # main.py:117-118
    random.seed(0); np.random.seed(0); torch.manual_seed(0)                             # main.py:19-26
    true_losses = oracle.true_losses(dataset.preds)                                     # main.py:57
    best_loss = min(true_losses)
    selector = CODA.from_args(dataset, args)                                            # main.py:67
    regrets = [float(true_losses[selector.get_best_model_prediction()] - best_loss)]   # main.py:83-84
    for _ in range(args.iters):                                                         # main.py:89-103
        chosen_idx, selection_prob = selector.get_next_item_to_label()
        true_class = oracle(chosen_idx)
        selector.add_label(chosen_idx, true_class, selection_prob)
        regrets.append(float(true_losses[selector.get_best_model_prediction()] - best_loss))
    out = dict(dtype=dataset.preds.dtype, regrets=regrets, idx=list(selector.labeled_idxs),
               pbest=selector.get_pbest().cpu())
    selector.close()
    return out


@gpu
def test_main_py_loop_through_the_coda_shim_on_an_fp16_file(tmp_path, monkeypatch):
    from coda_b200.synth import synth
    preds, labels = synth(16, 1500, 8, seed=23)
    torch.save(preds.half(), str(tmp_path / "toy.pt"))
    torch.save(labels, str(tmp_path / "toy_labels.pt"))
    monkeypatch.delenv("CODA_B200_KEEP_FP16", raising=False)
    up = _main_py_loop(str(tmp_path / "toy.pt"))
    monkeypatch.setenv("CODA_B200_KEEP_FP16", "1")
    kept = _main_py_loop(str(tmp_path / "toy.pt"))
    assert up["dtype"] == torch.float32 and kept["dtype"] == torch.float16
    assert kept["regrets"] == up["regrets"] and kept["idx"] == up["idx"]
    assert torch.equal(kept["pbest"], up["pbest"])


# ---------------------------------------------------------------------------------------------- 8. CPU tier
def _save(tmp_path, dtype):
    t = (torch.arange(4 * 6 * 3, dtype=torch.float32).reshape(4, 6, 3) / 100).to(dtype)
    p = str(tmp_path / f"s_{str(dtype).split('.')[-1]}.pt")
    torch.save(t, p)
    return p, t


@pytest.mark.parametrize("dtype,kept", [(torch.float16, torch.float16), (torch.float32, torch.float32),
                                        (torch.bfloat16, torch.float32)])
def test_loaders_keep_fp16(tmp_path, monkeypatch, dtype, kept):
    from coda_b200.datasets import Dataset, ShardedFileDataset
    monkeypatch.delenv("CODA_B200_KEEP_FP16", raising=False)
    p, t = _save(tmp_path, dtype)
    d = Dataset(p, "cpu", keep_fp16=True)
    assert d.preds.dtype == kept and torch.equal(d.preds.float(), t.float())
    s = ShardedFileDataset(p, "cpu", rank=1, world=2, keep_fp16=True)
    assert s.preds.dtype == kept and torch.equal(s.preds.float(), t[:, 3:6].float())
    # the default is unchanged: everything becomes fp32
    assert Dataset(p, "cpu").preds.dtype == torch.float32
    assert ShardedFileDataset(p, "cpu", rank=0, world=2).preds.dtype == torch.float32


def test_keep_fp16_environment_sets_the_default(tmp_path, monkeypatch):
    from coda_b200.datasets import Dataset, ShardedFileDataset
    p, _t = _save(tmp_path, torch.float16)
    monkeypatch.setenv("CODA_B200_KEEP_FP16", "1")
    assert Dataset(p, "cpu").preds.dtype == torch.float16
    assert ShardedFileDataset(p, "cpu").preds.dtype == torch.float16
    assert Dataset(p, "cpu", keep_fp16=False).preds.dtype == torch.float32
    monkeypatch.setenv("CODA_B200_KEEP_FP16", "0")
    assert Dataset(p, "cpu").preds.dtype == torch.float32


def test_shadow_sizing_by_element_size():
    from coda_b200.engine import shadow_slots
    for N in (1000, 1001, 1007):
        cs32, cs16 = (N + 3) // 4 * 4, (N + 7) // 8 * 8
        spare = 10 * cs32 * 100 * 4
        assert shadow_slots(spare, 256, N, 100, 4) == (10, cs32)
        s16, cs = shadow_slots(spare, 256, N, 100, 2)
        assert cs == cs16 and s16 == spare // (cs16 * 100 * 2)
        assert s16 == 20 if N % 8 == 0 else s16 in (19, 20)   # the fp16 column stride rounds to 8 items, not 4
    assert shadow_slots(10 ** 12, 7, 100, 10, 2)[0] == 7
    assert shadow_slots(-5, 7, 100, 10, 2)[0] == 0


def test_f16_entry_points_are_declared():
    hdr = open(os.path.join(os.path.dirname(__file__), "..", "include", "coda_b200.h")).read()
    from coda_b200._native import SIGNATURES
    for name in ("scan_slab", "confusion_sorted", "confusion_accum", "pi_full", "pi_full_tc_ok", "pi_full_tc",
                 "shadow_build", "pi_rank1"):
        f16 = f"coda_b200_{name}_f16"
        assert f16 + "(" in hdr and f16 in SIGNATURES
        # the fp16 twin takes the same arguments as the fp32 entry point
        assert SIGNATURES[f16] == SIGNATURES[f"coda_b200_{name}"]
