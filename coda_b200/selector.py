"""``CODA`` -- host-side mirror of the reference selector (coda/coda.py:171-346) over the sm_100a kernels.

Same constructor, same three ``ModelSelector`` calls, same attributes callers read
(``stochastic``, ``unlabeled_idxs``, ``pi_hat``, ``pi_hat_xi``, ``dirichlets``, ``labeled_idxs``,
``labels``, ``q_vals``, ``step``, ``H/N/C``, ``device``), same error types.  The arithmetic is in
``libcoda_b200.so``; there is no CPU route -- a CPU ``dataset.preds`` raises.

Sharding (SURVEY.md 8e), chosen at construction:
  * one process per GPU (torchrun + ``torch.distributed`` initialised): this process owns one shard;
  * ONE process, several GPUs (``main.py`` unchanged): ``gpus=`` / ``CODA_B200_GPUS`` (default: every visible GPU once the
    slab is >= 4 GiB) splits ``dataset.preds`` along N -- shard 0 reads the caller's tensor in place, the others get
    peer copies -- and this object drives all shards, each on its own stream;
  * ``shards=`` > number of GPUs puts several shards on one GPU (the 1-GPU test tier exercises the exchange that way).
"""
from __future__ import annotations

import os
import random

import numpy as np
import torch

from .base import ModelSelector
from .dist import InProcessGroup, ProcessGroup, SoloGroup, choose_among_ties, default_comm
from .engine import TIE_CAP, build_engines
from .synth import shard_range


class _Unlabeled:
    """List-like view of the unlabeled item indices (coda.py:200, 323; demo/app.py:188 calls ``remove``).
    The reference keeps a Python list and pays O(N) per removal; this keeps a removed-set and a device mask."""

    def __init__(self, n_lo: int, n_hi: int, on_remove):
        self._lo, self._hi = n_lo, n_hi
        self._removed = set()
        self._on_remove = on_remove

    def remove(self, idx):
        idx = int(idx)
        if not (self._lo <= idx < self._hi) or idx in self._removed:
            raise ValueError("list.remove(x): x not in list")             # coda.py:323 behaviour
        self._removed.add(idx)
        self._on_remove(idx)

    def __contains__(self, idx):
        return self._lo <= int(idx) < self._hi and int(idx) not in self._removed

    def __len__(self):
        return self._hi - self._lo - len(self._removed)

    def __iter__(self):
        rem = self._removed
        return (i for i in range(self._lo, self._hi) if i not in rem)

    def __getitem__(self, k):
        return list(self)[k]


def _auto_gpus(preds) -> int:
    env = os.environ.get("CODA_B200_GPUS")
    if env:
        return max(1, int(env))
    # bytes of the slab: a dense fp16 slab counts 2 per score (the compact form reports its own float count)
    esize = 2 if getattr(preds, "dtype", None) == torch.float16 else 4
    if preds.numel() * esize < (4 << 30):
        return 1
    return max(1, torch.cuda.device_count())


class CODA(ModelSelector):
    def __init__(self, dataset, prefilter_n=0, alpha=0.9, learning_rate=0.01, multiplier=2.0,
                 disable_diag_prior=False, q="eig", *, mode="incremental", comm=None, gpus=None, shards=None):
        self.dataset = dataset
        preds = dataset.preds
        self.device = preds.device
        self.prefilter_n = prefilter_n
        self.disable_diag_prior = disable_diag_prior
        self.q = q
        self.prior_strength = 1 - alpha                     # coda.py:189
        self.update_strength = learning_rate                # coda.py:190
        comm = comm or default_comm()
        n_offset = int(getattr(dataset, "n_offset", 0))
        n_global = int(getattr(dataset, "n_global", preds.shape[1]))
        kw = dict(alpha=alpha, learning_rate=learning_rate, multiplier=multiplier,
                  uniform_prior=bool(disable_diag_prior), mode=mode, n_global=n_global)
        if comm.world > 1:                                  # one process per GPU: this is one shard of the task
            self.group = ProcessGroup(comm)
            layout = [(preds, n_offset)]
        else:
            nshards = int(shards) if shards else (int(gpus) if gpus else _auto_gpus(preds))
            ngpus = int(gpus) if gpus else min(nshards, max(1, torch.cuda.device_count()))
            nshards = max(1, min(nshards, preds.shape[1]))
            if nshards == 1:
                self.group = SoloGroup()
                layout = [(preds, n_offset)]
            else:
                self.group = InProcessGroup(nshards)
                layout = self._split(preds, nshards, ngpus)
        self.engines = build_engines(layout, self.group, **kw)
        self.engine = self.engines[0]
        self.H, self.C = self.engine.H, self.engine.C
        self.N = n_global                                   # callers see the whole task (coda.py:183)
        self.labeled_idxs, self.labels = [], []
        self.unlabeled_idxs = _Unlabeled(0, n_global, self._mark_labeled)
        self.q_vals = []
        self.stochastic = False
        self.step = 0
        self.last_report = None
        self._hist_seen = 0                                 # device-loop steps already mirrored into the host lists
        self._labels_dev = None
        self._loop_dirty = False

    @staticmethod
    def _split(preds, nshards, ngpus):
        """N-range shards of a slab that lives on one device: shards on the home device are VIEWS of the caller's
        tensor (the kernels take the model stride), the others are contiguous copies on their device."""
        n = preds.shape[1]
        home = preds.device.index
        devs = [home] + [d for d in range(torch.cuda.device_count()) if d != home]
        devs = devs[:max(1, ngpus)]
        out = []
        for r in range(nshards):
            lo, hi = shard_range(n, r, nshards)
            d = devs[r * len(devs) // nshards]              # consecutive shards share a device when shards > GPUs
            if isinstance(preds, torch.Tensor):
                view = preds[:, lo:hi]
                if d != home:
                    view = view.to(torch.device("cuda", d)).contiguous()
            else:                                           # CompactSlab
                view = preds.narrow_items(lo, hi)
                if d != home:
                    view = view.to(torch.device("cuda", d))
            out.append((view, lo))
        for d in devs:                                      # the peer copies ran on the current streams; the shards use their own
            torch.cuda.synchronize(d)
        return out

    @classmethod
    def from_args(cls, dataset, args):
        """coda.py:205-213"""
        return cls(dataset, prefilter_n=args.prefilter_n, alpha=args.alpha, learning_rate=args.learning_rate,
                   multiplier=args.multiplier, disable_diag_prior=args.no_diag_prior, q=args.q)

    # -- plumbing over the shards -----------------------------------------------------------------
    def _sync(self):
        for e in self.engines:
            e.sync()

    def _mark_labeled(self, idx):
        for e in self.engines:
            e.mark_labeled(idx)

    def _home(self, t):
        return t if t.device == self.device else t.to(self.device)

    def _cat(self, name):
        """Per-item vector ``name`` over all items, on the dataset's device (cold paths).  With one process per GPU it
        would need a host all-gather of N-sized vectors: not offered there -- use the single-process front end."""
        if self.group.world > 1 and len(self.engines) == 1:
            raise NotImplementedError("this acquisition variant needs all items in one process: build CODA with "
                                      "gpus=... (one process driving all GPUs) instead of one process per GPU")
        self._sync()
        if len(self.engines) == 1:
            return getattr(self.engine, name)
        return torch.cat([self._home(getattr(e, name)) for e in self.engines], 0)

    # -- attributes the reference exposes as tensors ---------------------------------------
    @property
    def dirichlets(self):
        self._sync()
        return self.engine.D

    @property
    def pi_hat(self):
        self._sync()
        return self.engine.pi_hat

    @property
    def pi_hat_xi(self):
        parts = [e.pi_hat_xi() for e in self.engines]
        self._sync()
        return parts[0] if len(parts) == 1 else torch.cat([self._home(p) for p in parts], 0)

    @property
    def eig(self):
        """Per-item expected information gain of the last scoring pass (this process's shards, item order)."""
        self._sync()
        return self.engine.eig if len(self.engines) == 1 else torch.cat([self._home(e.eig) for e in self.engines], 0)

    # -- acquisition -------------------------------------------------------------------------
    def _fetch_report(self):
        for e in self.engines:
            e.report()                                      # enqueue on every shard before anyone waits
        rep = self.engine.fetch()
        self.last_report = rep
        self.engine.check_flags(flags=rep["flags"])
        return rep

    def get_next_item_to_label(self):
        """coda.py:283-313.  Returns (global item index: int, q: float)."""
        if self.q in ("iid", "uncertainty"):
            return self._select_ablation()                  # coda.py:287-295
        if self.q != "eig":
            raise NotImplementedError(self.q)               # coda.py:297
        rep = self._fetch_report()
        if self.prefilter_n:
            return self._select_prefiltered()
        if rep["n_ties"] == 0:
            raise RuntimeError("no unlabeled items left to select from")
        if rep["n_ties"] > 1:                               # coda.py:308-311
            self.stochastic = True
            if rep["n_ties"] <= len(rep["tie_idx"]):
                ties = rep["tie_idx"]
                idx = choose_among_ties(ties, random)
                q = float(rep["tie_val"][int(np.nonzero(ties == idx)[0][0])])
            else:
                idx, q = self._select_many_ties(rep)
            return idx, q
        return int(rep["tie_idx"][0]), float(rep["tie_val"][0])   # == arg-max, first index wins (coda.py:309)

    @staticmethod
    def _candidate_mask(labeled, disagree):
        m = (labeled == 0) & (disagree != 0)
        if not bool(m.any()):
            m = labeled == 0                                # coda.py:239 `or self.unlabeled_idxs`
        return m

    def _select_ablation(self):
        """coda.py:287-295: the two ablation acquisitions of the paper (random / ensemble-entropy sampling) followed by
        the same tie rule (coda.py:306-313).  Cold path over ``ens`` = sum_h preds from the slab scan."""
        if self.prefilter_n:
            raise NotImplementedError(f"q={self.q!r} together with prefilter_n")
        mask = self._candidate_mask(self._cat("labeled"), self._cat("disagree"))
        n = int(mask.sum())
        if n == 0:
            raise RuntimeError("no unlabeled items left to select from")
        if self.q == "iid":
            qv = torch.full((self.N,), np.float32(1.0 / n).item(), dtype=torch.float32, device=self.device)
        else:
            if getattr(self, "_ens_entropy", None) is None:      # non-adaptive: computed once (uncertainty.py:6-11)
                if self.engine.ens is None:
                    raise RuntimeError("q='uncertainty' needs the ensemble sums (CODA_B200_ENS=0 disables them)")
                mean = self._cat("ens") / float(self.H)
                self._ens_entropy = -(mean * torch.log(mean + 1e-8)).sum(-1)
            qv = self._ens_entropy
        best = qv[mask].max()
        ties = torch.isclose(qv, best, rtol=1e-8) & mask        # coda.py:307
        nt = int(ties.sum())
        if nt > 1:                                              # coda.py:308-311
            idx = random.choice(torch.nonzero(ties, as_tuple=True)[0].tolist())
            self.stochastic = True
        else:
            idx = int(torch.nonzero(ties, as_tuple=True)[0][0])
        return idx, float(qv[idx])

    def _select_many_ties(self, rep):
        """More than TIE_CAP isclose-ties: evaluate the tie rule on the full vector (cold path)."""
        eig = self._cat("eig").cpu().numpy()
        cand = np.nonzero(self._candidate_mask(self._cat("labeled"), self._cat("disagree")).cpu().numpy())[0]
        qv = eig[cand]
        best = np.float32(rep["best_val"])
        tol = np.float32(1e-8) + np.abs(np.float32(1e-8) * best)
        ties = cand[(qv == best) | (np.abs(qv - best) <= tol)]
        idx = choose_among_ties(ties, random)
        return int(idx), float(eig[idx])

    def _select_prefiltered(self):
        """coda.py:221-223: random subsample of the candidates (``--prefilter-n``), then coda.py:306-313
        on the subsample in sample order.  Cold ablation path; uses the EIG vector the kernels produced."""
        labeled, disagree = self._cat("labeled"), self._cat("disagree")
        m = (labeled == 0) & (disagree != 0)
        ids = torch.nonzero(m, as_tuple=True)[0].tolist()
        if self.prefilter_n and len(ids) > self.prefilter_n:
            ids = random.sample(ids, self.prefilter_n)
            self.stochastic = True
        if not ids:
            ids = torch.nonzero(labeled == 0, as_tuple=True)[0].tolist()
        qv = self._cat("eig")[torch.tensor(ids, device=self.device)]
        best = qv.max()
        ties = torch.isclose(qv, best, rtol=1e-8)
        if int(ties.sum()) > 1:
            loc = random.choice(torch.nonzero(ties, as_tuple=True)[0].tolist())
            self.stochastic = True
        else:
            loc = int(torch.argmax(qv))
        return ids[loc], float(qv[loc])

    # -- posterior update --------------------------------------------------------------------
    def add_label(self, idx, true_class, selection_prob):
        """coda.py:315-323"""
        idx, true_class = int(idx), int(true_class)
        if self._loop_dirty:
            self.history()                                  # a device loop ran: bring the host-side lists up to date first
        if not (0 <= true_class < self.C):
            raise IndexError(f"index {true_class} is out of bounds for dimension 1 with size {self.C}")
        if idx not in self.unlabeled_idxs:
            raise ValueError("list.remove(x): x not in list")
        eager = self.q == "eig" and not self.prefilter_n    # the next call will want the scores: enqueue them now
        for e in self.engines:                              # phases in lock-step over the shards (see Engine.label_stage)
            e.label_stage(idx, true_class)
        if eager and all(e.api_graph_wanted() for e in self.engines):
            for e in self.engines:
                e.api_capture()
        for e in self.engines:
            e.label_run(eager)
        self.labeled_idxs.append(idx)
        self.labels.append(true_class)
        self.q_vals.append(selection_prob)
        self.unlabeled_idxs._removed.add(idx)               # the label kernels already set the device mask

    def get_pbest(self):
        """coda.py:325-332 -> (1, H) float32 tensor on the device."""
        out = self.engine.pbest()
        if self.engine.stream is not None:
            self.engine.sync()
        return out

    def get_best_model_prediction(self):
        """coda.py:334-346 -> a fresh 0-d LongTensor like torch.argmax (trap T10); bumps ``step``."""
        self.step += 1
        with self.engine._on():
            out = self.engine.best_model[0].clone()
        if self.engine.stream is not None:
            self.engine.sync()
        return out

    # -- host-free loop (SURVEY.md 8f rank 2) ----------------------------------------------------
    def run_steps(self, k, labels):
        """``k`` acquisition steps with the oracle's labels resident on the device(s): main.py:89-94 without a host
        round trip (arg-max pick, first index on equal values; a step where the reference would have drawn from
        ``random.choice`` because of an isclose tie is flagged in ``history()``).  ``labels``: int64 tensor of all N
        labels.  Returns nothing; read ``history()`` / ``get_pbest()`` afterwards."""
        cache = getattr(self, "_labels_dev", None)
        if cache is None or cache[0] is not labels:
            per_dev = {}
            for e in self.engines:
                if e.dev not in per_dev:
                    per_dev[e.dev] = labels.to(e.dev, torch.int64).contiguous()
            for d in per_dev:
                torch.cuda.synchronize(d)
            self._labels_dev = cache = (labels, per_dev)
        per_dev = cache[1]
        if k <= 0:
            return
        self._loop_dirty = True
        # phases in lock-step over the shards: nobody waits on the host for a peer that has not been enqueued
        for e in self.engines:
            e.loop_prepare(per_dev[e.dev])
        if not all(e.loop_ready() for e in self.engines):
            for e in self.engines:
                e.loop_eager()
            k -= 1
            for e in self.engines:
                e.loop_capture()
        for _ in range(k):
            for e in self.engines:
                e.loop_replay(1)

    def history(self):
        """(idx, q, tie) arrays of the device-loop steps so far (the last HIST_CAP of them); also mirrors them into the
        host-side bookkeeping the API path keeps (``labeled_idxs``, ``labels``, ``q_vals``, ``unlabeled_idxs``)."""
        self._sync()
        e = self.engine
        with e._on():
            n = int(e.step_ctr.item())
            idx = e.hist_idx[:n].cpu().numpy()
            q = e.hist_q[:n].cpu().numpy()
            tie = e.hist_tie[:n].cpu().numpy()
            e.check_flags(sync=True)
        if n > self._hist_seen and self._labels_dev is not None:
            lab = self._labels_dev[0]
            new = idx[self._hist_seen:n]
            cls = lab[torch.as_tensor(new, device=lab.device)].cpu().tolist() if len(new) else []
            for i, qq, t in zip(new.tolist(), q[self._hist_seen:n].tolist(), cls):
                self.labeled_idxs.append(int(i)); self.labels.append(int(t)); self.q_vals.append(float(qq))
                self.unlabeled_idxs._removed.add(int(i))
            self._hist_seen = n
        self._loop_dirty = False
        return idx, q, tie

    # -- checkpoint / resume (SURVEY.md 8f rank 4; the reference restarts a killed seed from step 0) ------
    def state_dict(self):
        self._sync()
        sd = {"version": 1, "H": self.H, "N": self.N, "C": self.C, "mode": self.engine.mode,
              "labeled_idxs": list(self.labeled_idxs), "labels": list(self.labels), "q_vals": list(self.q_vals),
              "removed": sorted(self.unlabeled_idxs._removed), "stochastic": self.stochastic, "step": self.step,
              "python_random_state": random.getstate(), "shards": []}
        for e in self.engines:
            with e._on():
                sd["shards"].append({"n_offset": e.n_offset, "N": e.N,
                                     **{k: v.detach().cpu().clone() for k, v in e.state_tensors().items()}})
        return sd

    def load_state_dict(self, sd, restore_rng=True):
        """Resume a selector built on the same slab: bit-exact continuation (same picks, same posterior bits).
        The state may have been saved with a different shard count (this process must hold all its items)."""
        if (sd["H"], sd["N"], sd["C"]) != (self.H, self.N, self.C):
            raise ValueError("state_dict belongs to a different task shape")
        self._sync()
        order = sorted(sd["shards"], key=lambda s: s["n_offset"])
        U = torch.cat([s["U"] for s in order], 0)
        labeled = torch.cat([s["labeled"] for s in order], 0)
        base = order[0]["n_offset"]
        for e in self.engines:
            with e._on():
                lo, hi = e.n_offset - base, e.n_offset - base + e.N
                if lo < 0 or hi > U.shape[0]:
                    raise ValueError("state_dict does not cover this shard's items")
                e.D.copy_(order[0]["D"].to(e.dev))
                e.U.copy_(U[lo:hi].to(e.dev))
                e.labeled.copy_(labeled[lo:hi].to(e.dev))
                e.step_ctr.copy_(order[0]["step_ctr"].to(e.dev))
                e.pisum.zero_()
                e._call("coda_b200_pi_reduce", e.U.data_ptr(), e.N, e.C, e.fx_shift, None, e.pisum.data_ptr(),
                        e.flags.data_ptr(), e._s())
                e._tables(0, e.C)
                e.cache_valid, e.scored, e.reported, e.pending = False, False, False, False
                e.graphs.clear()
        for e in self.engines:
            e.construct_mixture()
        self._sync()
        self.labeled_idxs, self.labels, self.q_vals = list(sd["labeled_idxs"]), list(sd["labels"]), list(sd["q_vals"])
        self.unlabeled_idxs._removed = set(sd["removed"])
        self.stochastic, self.step = bool(sd["stochastic"]), int(sd["step"])
        if restore_rng:
            random.setstate(sd["python_random_state"])

    def close(self):
        """Free the device memory of every shard now (a selector is otherwise kept alive by reference cycles until gc)."""
        for e in self.engines:
            e.close()
        self._labels_dev = None
        self.dataset = None
