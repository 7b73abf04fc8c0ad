"""Pin the CPU oracle (oracle/coda_oracle.py) against outputs of the reference itself
(tests/golden/*.npz, produced by tests/golden/make_golden.py in the build container)."""
import random

import numpy as np
import pytest
import torch

from helpers import coda_oracle, golden_names, golden_slab, load_golden, GOLDEN


@pytest.fixture(autouse=True)
def golden_thread_count():
    """The reference ran with 8 torch threads when it wrote the goldens.  torch splits a CPU reduction by thread count,
    and another split sums in another order: the fp32 quadrature behind every EIG moves by ~1e-6 with it.  The replay
    uses the same split, so the tolerances below measure the oracle and not the core count of the host."""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


def test_quadrature_known_answers():
    z = np.load(f"{GOLDEN}/quadrature_kat.npz")
    got = coda_oracle.pbest_rows(torch.from_numpy(z["alpha"]), torch.from_numpy(z["beta"]))
    np.testing.assert_allclose(got.numpy(), z["pbest"], rtol=2e-6, atol=1e-9)
    assert np.array_equal(coda_oracle.quad_grid().numpy(), z["grid"])   # trap T1: same fp32 grid bits
    np.testing.assert_allclose(got.sum(-1).numpy(), 1.0, atol=1e-5)


@pytest.mark.parametrize("name", golden_names())
def test_trajectory_matches_reference(name):
    g = load_golden(name)
    if int(g["N"]) > 5000 or int(g["H"]) * int(g["N"]) * int(g["C"]) > 2e7:
        pytest.skip("large golden is for the GPU parity test; oracle replay would take minutes")
    preds, labels = golden_slab(g)
    random.seed(0)
    sel = coda_oracle.OracleSelector(preds, **g["ctor"])
    np.testing.assert_allclose(sel.dirichlets.numpy(), g["init_dirichlets"], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(sel.pi_hat.numpy(), g["init_pi_hat"], rtol=1e-6)
    np.testing.assert_allclose(sel.pi_hat_xi.numpy(), g["init_pi_hat_xi"], rtol=1e-5, atol=1e-8)
    assert int(sel.get_best_model_prediction()) == int(g["init_best_model"])
    np.testing.assert_allclose(sel.get_pbest().numpy(), g["init_pbest"], rtol=1e-5, atol=1e-8)
    for k in range(int(g["steps"])):
        idx, q = sel.get_next_item_to_label()
        ref_eig = g["eig"][k]
        cand = np.asarray(sel.last_cand)
        assert len(cand) == int(g["n_cand"][k])
        assert np.all(np.isfinite(ref_eig[cand])) and np.isnan(np.delete(ref_eig, cand)).all()
        # same arithmetic order as the reference => agreement to fp32 rounding noise
        np.testing.assert_allclose(sel.last_q.numpy(), ref_eig[cand], atol=2e-6)
        assert idx == int(g["idx"][k]), (k, idx, int(g["idx"][k]))
        assert abs(q - float(g["q"][k])) < 2e-6
        t = int(labels[idx])
        sel.add_label(idx, t, q)
        assert int(sel.get_best_model_prediction()) == int(g["best_model"][k])
        np.testing.assert_allclose(sel.get_pbest().numpy()[0], g["pbest"][k], rtol=1e-5, atol=1e-8)
        np.testing.assert_allclose(sel.pi_hat.numpy(), g["pi_hat"][k], rtol=1e-6)
        np.testing.assert_array_equal(sel.dirichlets[:, t].numpy(), g["dir_row"][k])  # update is one fp32 add
    np.testing.assert_allclose(sel.dirichlets.numpy(), g["final_dirichlets"], rtol=1e-6, atol=1e-7)
    assert sel.step == int(g["steps"]) + 1
    assert int(sel.stochastic) == int(g["stochastic"])


def test_error_behaviour_matches_reference():
    """coda.py:297 NotImplementedError(q); coda.py:323 list.remove ValueError; util.py:20-25 RuntimeError."""
    g = load_golden("traj_tiny_h8_n300_c5")
    preds, labels = golden_slab(g)
    sel = coda_oracle.OracleSelector(preds, q="bogus")
    with pytest.raises(NotImplementedError):
        sel.get_next_item_to_label()
    sel = coda_oracle.OracleSelector(preds)
    sel.add_label(3, 1, 0.0)
    with pytest.raises(ValueError):
        sel.add_label(3, 1, 0.0)
    bad = torch.tensor([[float("nan"), 1.0]])
    with pytest.raises(RuntimeError, match="NUMERIC ERROR"):
        coda_oracle.pbest_rows(bad, torch.ones(1, 2))


def _rng_words():
    return np.array(random.getstate()[1], dtype=np.uint32)


@pytest.mark.parametrize("q", ["iid", "uncertainty"])
def test_oracle_ablation_acquisitions_vs_live_reference(q):
    """The ablation acquisitions against what the reference itself did on the same slab and seed
    (tests/golden/acquisitions.npz, made by tests/golden/make_golden.py): same picks, same scores, same RNG
    consumption, same best model after every label."""
    from coda_b200.synth import synth
    g = np.load(f"{GOLDEN}/acquisitions.npz")
    preds, labels = synth(12, 500, 6, seed=17)
    random.seed(4)
    o = coda_oracle.OracleSelector(preds, q=q)
    for k in range(4):
        io, qo = o.get_next_item_to_label()
        assert io == int(g[f"{q}_idx"][k]) and abs(qo - float(g[f"{q}_q"][k])) < 1e-7
        assert np.array_equal(_rng_words(), g[f"{q}_rng"][k])
        o.add_label(io, int(labels[io]), qo)
        assert int(o.get_best_model_prediction()) == int(g[f"{q}_best_model"][k])


def test_oracle_prefilter_subsample_vs_live_reference():
    """coda.py:221-223 (--prefilter-n): random.sample over the candidate list, then the tie rule on the subsample --
    checked against what the reference itself did (same RNG consumption, same pick)."""
    from coda_b200.synth import synth
    g = np.load(f"{GOLDEN}/acquisitions.npz")
    preds, labels = synth(10, 600, 6, seed=8)
    random.seed(5)
    o = coda_oracle.OracleSelector(preds, prefilter_n=50)
    io, qo = o.get_next_item_to_label()
    assert io == int(g["prefilter_idx"]) and abs(qo - float(g["prefilter_q"])) < 2e-6
    assert np.array_equal(_rng_words(), g["prefilter_rng"])
    assert o.stochastic and bool(g["prefilter_stochastic"])
