"""Generate golden fixtures by RUNNING THE REFERENCE (CPU, fp32) in the build container.

    python tests/golden/make_golden.py            # needs /root/reference; writes tests/golden/*.npz

The reference has no tests or golden vectors of its own (SURVEY.md 8c), so the pins are
outputs of the unmodified ``/root/reference/coda/coda.py`` on seeded synthetic slabs
(``coda_b200.synth``).  ``/root/reference`` does not exist on the GPU box; only the small
``.npz`` files travel.  ``matplotlib`` is not installed here and ``coda/util.py:2`` imports
it, so an empty stub module is put on ``sys.modules`` first (nothing on the path uses it).

Each fixture stores the synthetic-task parameters (the slab is regenerated from them), the
reference's initial state, and a free-running K-step trajectory: per step the candidate
EIG vector, chosen index, q, the posterior after the label, pi_hat and P(best).
"""
import os
import random
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
from helpers import final_dirichlets  # noqa: E402

REF = os.environ.get("CODA_REFERENCE_PATH", "/root/reference")


def import_reference():
    for name in ("matplotlib", "matplotlib.pyplot"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.path.insert(0, REF)
    # our repo also has a package called ``coda``; make sure the reference's wins here
    for k in [k for k in sys.modules if k == "coda" or k.startswith("coda.")]:
        del sys.modules[k]
    import coda.coda as ref_coda
    assert ref_coda.__file__.startswith(REF), ref_coda.__file__
    import tqdm
    ref_coda.tqdm = lambda it, *a, **k: it          # silence the progress bar only
    return ref_coda


class _DS:
    def __init__(self, preds, labels):
        self.preds, self.labels, self.device = preds, labels, preds.device


def seed_all(seed):
    """main.py:19-26"""
    random.seed(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)


def run_case(ref_coda, name, H, N, C, data_seed, steps, dense=False, ctor=None, save_eig=True, slim=False, drop=()):
    from coda_b200.synth import synth
    ctor = ctor or {}
    preds, labels = synth(H, N, C, data_seed, dense=dense)
    seed_all(0)
    sel = ref_coda.CODA(_DS(preds, labels), **ctor)
    out = {
        "H": H, "N": N, "C": C, "data_seed": data_seed, "dense": int(dense), "steps": steps,
        "ctor_keys": np.array(list(ctor.keys()), dtype="U32"),
        "ctor_vals": np.array([float(v) for v in ctor.values()], dtype=np.float64),
        "init_dirichlets": sel.dirichlets.numpy().copy(),
        "init_pi_hat": sel.pi_hat.numpy().copy(),
        "init_pi_hat_xi": sel.pi_hat_xi.numpy().copy(),
        "labels": labels.numpy(),
    }
    best0 = sel.get_best_model_prediction()
    out["init_pbest"] = sel.get_pbest().numpy().copy()
    out["init_best_model"] = int(best0)
    idxs, qs, bests, pbests, pis, eigs, cands, ntie, dirs, xi_rows = [], [], [], [], [], [], [], [], [], []
    for k in range(steps):
        # replicate get_next_item_to_label but keep the full EIG vector (coda.py:283-313)
        st = random.getstate()
        q_vals, cand = sel.eig_batched()
        best = q_vals.max()
        ties = torch.isclose(q_vals, best, rtol=1e-8)
        ntie.append(int(ties.sum()))
        # coda.py:306-313 applied to the vector we already have ...
        loc = random.choice(torch.nonzero(ties, as_tuple=True)[0].tolist()) if ties.sum() > 1 \
            else torch.argmax(q_vals).item()
        if ties.sum() > 1:
            sel.stochastic = True
        idx, q = cand[loc], q_vals[loc].item()
        if N <= 5000:
            # ... and cross-checked against the reference's own call (same RNG state => same pick)
            st_after = random.getstate()
            random.setstate(st)
            idx2, q2 = sel.get_next_item_to_label()
            assert (idx2, q2) == (idx, q) and random.getstate() == st_after
        if save_eig:
            full = np.full((N,), np.nan, dtype=np.float32)
            full[np.asarray(cand)] = q_vals.numpy()
            eigs.append(full)
        cands.append(len(cand))
        t = int(labels[idx])
        sel.add_label(idx, t, q)
        b = sel.get_best_model_prediction()
        idxs.append(idx); qs.append(q); bests.append(int(b))
        pbests.append(sel.get_pbest().numpy().copy()[0])
        pis.append(sel.pi_hat.numpy().copy())
        dirs.append(sel.dirichlets[:, t].numpy().copy())
        xi_rows.append(sel.pi_hat_xi[:64].numpy().copy())
    out.update(idx=np.array(idxs), q=np.array(qs, dtype=np.float64), best_model=np.array(bests),
               pbest=np.stack(pbests), pi_hat=np.stack(pis), n_cand=np.array(cands), n_ties=np.array(ntie),
               dir_row=np.stack(dirs), xi_head=np.stack(xi_rows),
               final_dirichlets=sel.dirichlets.numpy().copy(), stochastic=int(sel.stochastic))
    if save_eig:
        out["eig"] = np.stack(eigs)
    if slim:     # H*C*C-sized arrays make a multi-megabyte fixture: keep the per-step rows only
        for k in ("init_dirichlets", "final_dirichlets", "init_pi_hat_xi"):
            out.pop(k)
        out["xi_head"] = out["xi_head"][:, :8]
    elif np.array_equal(final_dirichlets(out), out["final_dirichlets"]):
        out.pop("final_dirichlets")          # tests/helpers.py rebuilds it from init_dirichlets and dir_row
    for k in drop:
        out.pop(k)
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print(name, "idx", idxs, "ties", ntie, "->", path, os.path.getsize(path) // 1024, "KiB")


def unit_vectors(ref_coda):
    """Known-answer vectors for the quadrature alone (coda.py:77-119) on hand-made Betas."""
    g = torch.Generator().manual_seed(123)
    a = torch.rand((7, 5), generator=g) * 6 + 0.05
    b = torch.rand((7, 5), generator=g) * 6 + 0.05
    a[0] = torch.tensor([0.02, 0.5, 1.0, 30.0, 200.0]); b[0] = torch.tensor([0.02, 3.0, 1.0, 2.0, 40.0])
    out = ref_coda.compute_pbest_beta_batched(a.view(7, 1, 1, 5), b.view(7, 1, 1, 5)).view(7, 5)
    x = torch.linspace(1e-6, 1 - 1e-6, 256)
    np.savez_compressed(os.path.join(HERE, "quadrature_kat.npz"), alpha=a.numpy(), beta=b.numpy(),
                        pbest=out.numpy(), grid=x.numpy())
    print("quadrature_kat", out[0])


def _rng_state():
    version, words, gauss = random.getstate()
    assert version == 3 and gauss is None
    return np.array(words, dtype=np.uint32)


def acquisitions(ref_coda):
    """The ablation acquisitions q='iid' / 'uncertainty' (coda.py:287-295) and the --prefilter-n subsample
    (coda.py:221-223): per step the pick, its score, the Python RNG state right after the pick (what random.choice /
    random.sample consumed) and the best model after the label."""
    from coda_b200.synth import synth
    out = {}
    preds, labels = synth(12, 500, 6, seed=17)
    for q in ("iid", "uncertainty"):
        random.seed(4)
        sel = ref_coda.CODA(_DS(preds, labels), q=q)
        idx, qs, states, bests = [], [], [], []
        for _ in range(4):
            i, v = sel.get_next_item_to_label()
            states.append(_rng_state())
            sel.add_label(i, int(labels[i]), v)
            idx.append(i); qs.append(v); bests.append(int(sel.get_best_model_prediction()))
        out.update({f"{q}_idx": np.array(idx), f"{q}_q": np.array(qs, dtype=np.float64),
                    f"{q}_rng": np.stack(states), f"{q}_best_model": np.array(bests)})
    preds, labels = synth(10, 600, 6, seed=8)
    random.seed(5)
    sel = ref_coda.CODA(_DS(preds, labels), prefilter_n=50)
    i, v = sel.get_next_item_to_label()
    out.update(prefilter_idx=np.array(i), prefilter_q=np.array(v, dtype=np.float64), prefilter_rng=_rng_state(),
               prefilter_stochastic=np.array(int(sel.stochastic)))
    path = os.path.join(HERE, "acquisitions.npz")
    np.savez_compressed(path, **out)
    print("acquisitions", {k: v.tolist() for k, v in out.items() if not k.endswith("_rng")}, "->", path)


if __name__ == "__main__":
    ref = import_reference()
    unit_vectors(ref)
    which = sys.argv[1:] or ["tiny", "small", "c100", "dense", "nodiag", "acq"]
    if "tiny" in which:
        run_case(ref, "traj_tiny_h8_n300_c5", 8, 300, 5, 1, steps=6)
    if "small" in which:
        run_case(ref, "traj_small_h32_n3000_c10", 32, 3000, 10, 0, steps=8)
    if "c100" in which:
        run_case(ref, "traj_c100_h24_n400_c100", 24, 400, 100, 2, steps=3)
    if "dense" in which:
        run_case(ref, "traj_dense_h16_n500_c12", 16, 500, 12, 3, steps=4, dense=True)
    if "nodiag" in which:
        run_case(ref, "traj_nodiag_h10_n400_c6", 10, 400, 6, 4, steps=4,
                 ctor=dict(disable_diag_prior=1, alpha=0.8, learning_rate=0.05, multiplier=1.5))
    if "h256" in which:   # full-width tensor-core tile (Hp = 256, C = 100): ~6 min per step on 8 cores
        run_case(ref, "traj_h256_h256_n1500_c100", 256, 1500, 100, 5, steps=2, slim=True)
    if "cfg2" in which:   # ~270 s/step on 8 cores: a few steps only; no test reads the 2 MB initial pi_hat_xi
        run_case(ref, "traj_cfg2_h64_n50000_c10", 64, 50000, 10, 0, steps=3, drop=("init_pi_hat_xi",))
    if "acq" in which:
        acquisitions(ref)
