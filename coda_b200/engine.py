"""Device-side state and kernel sequencing for one shard of the CODA acquisition path.

PyTorch is used for device memory, streams, CUDA graphs and the construction-time all-reduce -- the arithmetic of
the hot path and the per-step exchanges between shards are in the C-ABI library (``include/coda_b200.h``).

Modes (what is kept between steps; results are the same):
  ``incremental``   the normalised P(best | hypothetical) row of every row is cached; a label of
                    class t only invalidates the rows of class t (coda.py:317 touches row t only)
                    and the marginal refresh is the rank-1 column update of coda.py:319.
  ``recompute``     every step recomputes all rows from the tables (no row cache).
  ``recompute_all`` additionally rebuilds all class tables and re-runs the full slab pass of
                    ``update_pi_hat`` every step -- the reference's literal per-step work.

One acquisition step on the device (host-free loop, ``run_steps``; everything below is ONE CUDA graph):

    step_select   merge block records, exchange with the peers, arg-max, label lookup, D[h][t][p_h] += lr, gather list
    ---- fork ----  side stream: beta_tables(class t) -> pair_rows(class t)        main: pi_rank1 (marginal refresh)
    step_mixture  exchange the marginal sums, pi_hat, P(best), H_before, argmax         (needs PB[t] from the side)
    ---- join ----
    template_gains + gain_eig   the scoring pass for the NEXT selection -> block records
"""
from __future__ import annotations

import contextlib
import math
import os

import numpy as np
import torch

from . import _native as nat

_CONST_SLOTS = {}          # device index -> set of constant-memory term-table slots in use (csrc/slab.cu c_terms_bank)
_CONST_TERMS = 3584


def _acquire_const_slot(dev_index, H):
    per = (2 * H + 63) // 64 * 64
    used = _CONST_SLOTS.setdefault(dev_index, set())
    for s in range(_CONST_TERMS // per):
        if s not in used:
            used.add(s)
            return s
    return -1                  # every slot of this device is taken: the shared-memory copy of the list is used


def _release_const_slot(dev_index, slot):
    if slot is not None and slot >= 0:
        _CONST_SLOTS.get(dev_index, set()).discard(slot)


TIE_CAP = 256
REP_WORDS = 12 + TIE_CAP + TIE_CAP // 2     # [flags | record (8) | tie hdr (2) | pad | tie idx | tie val]
MODES = ("incremental", "recompute", "recompute_all")
TABLE_BATCH_BYTES = 512 << 20
HIST_CAP = 1 << 16


def _ptr(t):
    return t.data_ptr() if t is not None else None


def shadow_slots(spare_bytes, H, N, C, esize):
    """(model slots, column stride in elements) of a class-major shadow of ``esize``-byte elements in ``spare_bytes``:
    every (slot, class) column starts 16-byte aligned, so an fp16 shadow fits twice the models of an fp32 one."""
    per16 = 16 // esize
    cs = (N + per16 - 1) // per16 * per16
    return int(min(H, max(0, spare_bytes // (cs * C * esize)))), cs


class Engine:
    rep_words = REP_WORDS

    def __init__(self, preds: torch.Tensor, *, alpha: float, learning_rate: float, multiplier: float,
                 uniform_prior: bool, hyp_w: float = 1.0, mode: str = "incremental", n_offset: int = 0,
                 n_global: int | None = None, world: int = 1, own_stream: bool = False):
        from .datasets import CompactSlab
        if mode not in MODES:
            raise ValueError(f"mode must be one of {MODES}")
        self.compact = preds if isinstance(preds, CompactSlab) else None
        if not ((isinstance(preds, torch.Tensor) or self.compact is not None) and preds.is_cuda):
            raise RuntimeError("coda_b200: dataset.preds must live on a CUDA (sm_100a) device; "
                               "there is no CPU path in this package")
        H, N, Cc = (int(s) for s in preds.shape)
        if N < 1:
            raise ValueError("coda_b200: empty shard (fewer items than shards?)")
        if self.compact is not None:
            if mode == "recompute_all":
                raise NotImplementedError("coda_b200: mode='recompute_all' is not offered for a compact slab")
            self.K = self.compact.K
        else:
            if preds.dtype not in (torch.float32, torch.float16) or preds.dim() != 3:
                raise TypeError("coda_b200: preds must be a float32 or float16 (H, N, C) tensor (coda/datasets.py:14)")
            if not (preds.stride(2) == 1 and preds.stride(1) == Cc and (H == 1 or preds.stride(0) >= N * Cc)):
                raise ValueError("coda_b200: preds must be (H, N, C) with contiguous items (an N-range view of a "
                                 "contiguous slab is fine)")
        self.lib = nat.load()
        self.preds = preds
        # an fp16 slab stays fp16 on the device: the `_f16` entry points convert on load and give the bits of the fp32
        # run on preds.float(); every buffer derived from it (ensemble sums, U, D, ...) is fp32 as before
        self.f16 = self.compact is None and preds.dtype == torch.float16
        self.esize = 2 if self.f16 else 4                     # bytes per slab element
        self.dev = preds.device
        with torch.cuda.device(self.dev):
            nat.require_device()
            # sector gathers of the rank-1 refresh: ask for 64-byte L2 fills (the default 128 doubles their DRAM
            # traffic; streaming kernels measured the same at 64 and 128).  A per-device limit.
            nat.check(self.lib.coda_b200_set_l2_fetch_granularity(int(os.environ.get("CODA_B200_L2_FETCH", "64"))), "l2_fetch")
        self.H, self.N, self.C = H, N, Cc
        if self.compact is not None:
            self.model_stride = int(self.compact.ids.stride(0)) if H > 1 else N * self.K     # elements of ids / probs
        else:
            self.model_stride = int(preds.stride(0)) if H > 1 else N * Cc
        self.Hp = (H + 31) // 32 * 32
        self.W = self.Hp // 32
        self.P = 256
        self.T = Cc * (1 + H)
        self.mode = mode
        self.world = int(world)
        self.n_offset = int(n_offset)
        self.n_global = int(n_global if n_global is not None else N)
        self.lr = float(learning_rate)
        self.hyp_w = float(hyp_w)
        self.prior_strength = 1 - alpha                       # coda.py:189
        self.multiplier = float(multiplier)
        self.uniform_prior = bool(uniform_prior)
        if H > 1024:
            raise NotImplementedError("coda_b200: H > 1024 models is not supported yet")
        if Cc > 4096:
            raise NotImplementedError("coda_b200: C > 4096 classes is not supported yet")
        self.fx_shift = max(8, min(40, 62 - math.ceil(math.log2(self.n_global + 1))))
        self.counters = {"launches": 0}
        # CODA_B200_OVERLAP=0: class-t table / row refresh on the main stream instead of a side stream
        self.overlap = os.environ.get("CODA_B200_OVERLAP", "1") != "0"
        self.use_graph = os.environ.get("CODA_B200_GRAPH", "1") != "0"
        self.profile, self.profile_only = None, None
        self.xchg = None                                      # set by the group (dist.py) before the first exchange
        self._mailbox = None
        self._pi_tc, self._pi_scratch = None, None           # tensor-core marginal pass: decided on first use
        self.cidx = None                                      # compact slab: inverted index (see _build_compact_index)
        self.stream = torch.cuda.Stream(device=self.dev) if own_stream else None
        self.side = torch.cuda.Stream(device=self.dev)
        self.ev_fork, self.ev_join, self.ev_tables = torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event()
        self.graphs = {}
        self.labels_ptr = None
        # a private slot of the device's constant-memory term table (several selectors / shards may share a device)
        self.const_slot = _acquire_const_slot(self.dev.index, H) if os.environ.get("CODA_B200_R1_CONST", "1") != "0" else -1
        with self._on():
            self._alloc_static()

    # ------------------------------------------------------------------------------ utils
    @contextlib.contextmanager
    def _on(self):
        """Run the body with this shard's device current and, if it owns one, its stream current."""
        with torch.cuda.device(self.dev):
            if self.stream is not None:
                with torch.cuda.stream(self.stream):
                    yield
            else:
                yield

    def _cur(self):
        return torch.cuda.current_stream(self.dev)

    def _s(self):
        return self._cur().cuda_stream

    def sync(self):
        (self.stream or torch.cuda.current_stream(self.dev)).synchronize()

    def _call(self, name, *args, n=1):
        prof = self.profile
        if prof is not None and (self.profile_only is None or name in self.profile_only):
            st = self._cur()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            rc = getattr(self.lib, name)(*args)
            e1.record(st)
            prof.setdefault(name, []).append((e0, e1))
        else:
            rc = getattr(self.lib, name)(*args)
        nat.check(rc, name)
        self.counters["launches"] += n

    def start_profile(self, only=None):
        """Bracket every C-ABI launch (or just ``only``) with CUDA events on the launching stream (eager steps only)."""
        self.profile, self.profile_only = {}, (set(only) if only else None)

    def stop_profile(self):
        """-> {entry point: (launches, total ms, max ms)}; synchronises."""
        torch.cuda.synchronize(self.dev)
        out = {}
        for k, v in (self.profile or {}).items():
            ts = [a.elapsed_time(b) for a, b in v]
            out[k] = (len(ts), float(sum(ts)), float(max(ts)))
        self.profile = None
        return out

    def _z(self, shape, dtype):
        return torch.zeros(shape, dtype=dtype, device=self.dev)

    def _e(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.dev)

    # --------------------------------------------------------------------------- buffers
    def _alloc_static(self):
        H, N, C, Hp, P = self.H, self.N, self.C, self.Hp, self.P
        self.hard = self._e((N, H), torch.int16)              # uint16 bit patterns
        self.pseudo = self._e((N,), torch.int32)
        self.disagree = self._e((N,), torch.uint8)
        self.labeled = self._z((N,), torch.uint8)
        # soft-confusion sums (coda.py:42), int64 fixed point; the compact slab adds one "every column" term per row
        self.conf_buf = self._z((H * C * C + H * C,), torch.int64)
        self.conf_fx = self.conf_buf[: H * C * C].view(H, C, C)
        self.conf_rest = self.conf_buf[H * C * C:].view(H, C) if self.compact is not None else None
        self.D = self._e((H, C, C), torch.float32)
        # 16 bytes of slack behind U: the bulk-TMA marginal refresh rounds the last tile's copy up to 16 bytes
        self.U = self._e((N * C + 4,), torch.float32)[: N * C].view(N, C)
        self.pisum = self._z((C,), torch.int64)               # THIS shard's column sums (summed over shards in step_mixture)
        self.grid = torch.linspace(1e-6, 1 - 1e-6, P).to(self.dev)   # coda.py:86, built on the host (trap T1)
        self.dL = self._e((C, H, P), torch.float32)
        self.G0T = self._z((C, P, Hp), torch.float32)
        self.G1T = self._z((C, P, Hp), torch.float32)
        self.PB = self._z((C, Hp), torch.float32)
        # bf16 limb tables in tensor-core operand order (pairs_tc.cu); SIMT kernel (pairs.cu) when Hp > 256
        self.use_tc = Hp <= 256 and os.environ.get("CODA_B200_TC", "1") != "0"
        self.dLb = self._z((C, Hp // 32, 3, 256 * 32), torch.bfloat16) if self.use_tc else None
        self.Gb = self._z((C, 16, 4, Hp * 16), torch.bfloat16) if self.use_tc else None
        self.pi_hat = self._z((C,), torch.float32)
        self.m0 = self._z((Hp,), torch.float32)
        self.hb = self._z((1,), torch.float32)
        self.best_model = self._z((1,), torch.int64)
        self.eig = self._e((N,), torch.float32)
        self.nblocks = int(self.lib.coda_b200_eig_blocks(N, H, C))
        self.partials = self._z((self.nblocks, nat.REC_WORDS), torch.int64)
        # report block: one D2H copy per API step.  [flags | record (8) | tie hdr (2) | pad | tie idx | tie val]
        self.rep = self._z((REP_WORDS,), torch.int64)
        self.flags = self.rep[0:1].view(torch.int32)[0:1]
        self.bestrec = self.rep[1:9]
        self.tie_hdr = self.rep[9:11]
        self.tie_idx = self.rep[12:12 + TIE_CAP]
        self.tie_val = self.rep[12 + TIE_CAP:].view(torch.float32)[:TIE_CAP]
        self.rep_all = self._z((self.world, REP_WORDS), torch.int64)
        self.rep_host = torch.zeros((self.world, REP_WORDS), dtype=torch.int64).pin_memory()
        self.sel = self._z((2,), torch.int64)
        # staging ring for host-chosen (idx, class) records: a slot is rewritten only after its copy has executed
        self.sel_ring = torch.zeros((8, 2), dtype=torch.int64).pin_memory()
        self.sel_events = [None] * 8
        self.sel_pos = 0
        self.jvec = self._z((H,), torch.int32)
        self.terms = self._z((2 + 8 * H + 2,), torch.int64).view(torch.int32)[: 2 + 8 * H]   # 8-byte aligned
        self.step_ctr = self._z((1,), torch.int64)
        self.hist_idx = self._z((HIST_CAP,), torch.int64)
        self.hist_q = self._z((HIST_CAP,), torch.float32)
        self.hist_tie = self._z((HIST_CAP,), torch.int32)
        # ensemble sums E[n][c] (N*C floats) feed pi_rank1's majority shortcut; CODA_B200_ENS=0 disables it
        self.ens = self._e((N, C), torch.float32) if (os.environ.get("CODA_B200_ENS", "1") != "0" or self.compact is not None) else None
        cls_per_batch = max(1, min(C, TABLE_BATCH_BYTES // max(1, self.lib.coda_b200_tables_scratch_bytes(H, 1))))
        self.table_batch = int(cls_per_batch)
        self.scratch = self._e((int(self.lib.coda_b200_tables_scratch_bytes(H, self.table_batch)),), torch.uint8)

    def _make_step_struct(self):
        st = nat.StepStruct()
        st.H, st.C, st.N, st.n_offset, st.fx_shift, st.lr = self.H, self.C, self.N, self.n_offset, self.fx_shift, self.lr
        st.hard, st.labeled, st.D, st.jvec, st.sel = _ptr(self.hard), _ptr(self.labeled), _ptr(self.D), _ptr(self.jvec), _ptr(self.sel)
        st.terms = _ptr(self.terms)
        st.slot_of_model = _ptr(self.slot_of_model)
        st.shadow_off = ((self.shadow.data_ptr() - self._slab_ptr()) // self.esize) if self.shadow is not None else 0
        st.shadow_col_stride = self.shadow_cs
        st.model_stride = self.model_stride
        st.have_ens = 1 if self.ens is not None else 0
        st.compact_k = self.K if self.compact is not None else 0
        st.pisum_fx, st.PB, st.pi_hat, st.m0 = _ptr(self.pisum), _ptr(self.PB), _ptr(self.pi_hat), _ptr(self.m0)
        st.h_before, st.best_model = _ptr(self.hb), _ptr(self.best_model)
        st.partials, st.nblocks, st.eig, st.bestrec = _ptr(self.partials), self.nblocks, _ptr(self.eig), _ptr(self.bestrec)
        st.labels_global = None
        st.hist_idx, st.hist_q, st.hist_tie, st.hist_cap = _ptr(self.hist_idx), _ptr(self.hist_q), _ptr(self.hist_tie), HIST_CAP
        st.step_ctr = _ptr(self.step_ctr)
        st.flags = _ptr(self.flags)
        self.st = st

    def _slab_fn(self, name):
        """C entry point of a pass over the dense slab, for its element type."""
        return name + "_f16" if self.f16 else name

    def _slab_ptr(self):
        return self.preds.data_ptr() if self.compact is None else 0

    def _x(self):
        return self.xchg if (self.xchg is not None and self.world > 1) else None

    # ---------------------------------------------------------------------- construction
    # phases: scan -> [group: sum conf_fx over shards] -> posterior -> mixture (exchange) -> finish (host sync)
    def construct_scan(self):
        with self._on():
            H, N, C, s = self.H, self.N, self.C, self._s()
            if self.compact is not None:
                cs = self.compact
                self._call("coda_b200_scan_compact", _ptr(cs.ids), _ptr(cs.probs), self.model_stride, H, N, C, self.K,
                           _ptr(self.hard), _ptr(self.pseudo), _ptr(self.disagree), _ptr(self.ens), _ptr(self.flags), s)
                self._call("coda_b200_confusion_compact", _ptr(cs.ids), _ptr(cs.probs), self.model_stride,
                           _ptr(self.pseudo), H, N, C, self.K, self.fx_shift, _ptr(self.conf_fx), _ptr(self.conf_rest), s)
                self._build_compact_index()
                return
            self._call(self._slab_fn("coda_b200_scan_slab"), _ptr(self.preds), self.model_stride, H, N, C, _ptr(self.hard),
                       _ptr(self.pseudo), _ptr(self.disagree), _ptr(self.ens), _ptr(self.flags), s)
            if C <= 128:
                order = torch.argsort(self.pseudo).to(torch.int32)      # init-time plumbing: any grouping by label will do
                self._call(self._slab_fn("coda_b200_confusion_sorted"), _ptr(self.preds), self.model_stride, _ptr(self.pseudo),
                           _ptr(order), H, N, C, self.fx_shift, _ptr(self.conf_fx), s)
                del order
            else:
                self._call(self._slab_fn("coda_b200_confusion_accum"), _ptr(self.preds), self.model_stride, _ptr(self.pseudo), H, N, C,
                           self.fx_shift, _ptr(self.conf_fx), s)

    def construct_posterior(self):
        with self._on():
            H, C, s = self.H, self.C, self._s()
            self._call("coda_b200_init_dirichlets", _ptr(self.conf_fx), _ptr(self.conf_rest), H, C, self.fx_shift,
                       self.prior_strength, self.multiplier, int(self.uniform_prior), _ptr(self.D), s)
            self.conf_fx = self.conf_rest = self.conf_buf = None    # H*C*C int64, only needed once
            self._marginals_full()
            self._build_rows()
            self._build_shadow()
            self._make_step_struct()
            self._tables(0, C)
            self.cache_valid = False     # incremental mode: P(best | hypothetical) rows are cached once scored
            self.pending = False         # a side-stream refresh the next scoring pass has to join
            self.scored = False          # block records (`partials`) are current
            self.reported = False        # the report block in rep_host is (being) produced for the current state

    def construct_mixture(self):
        with self._on():
            self._mixture()

    def construct_finish(self):
        with self._on():
            self.check_flags(sync=True)

    def _build_compact_index(self):
        """Inverted index of the compact slab (csrc/compact.cu): per (model, class) the items whose top-K list holds the
        class.  With it the rank-1 marginal refresh reads H short lists (N K / C entries each) instead of the whole slab
        every step.  Same bytes as the slab (8 per entry): skipped when they do not fit (``CODA_B200_COMPACT_INDEX=0``
        forces the slab scan)."""
        self.cidx = None
        if os.environ.get("CODA_B200_COMPACT_INDEX", "1") == "0":
            return
        H, N, C, K, s = self.H, self.N, self.C, self.K, self._s()
        need = 8 * H * N * K + 16 * (H * C + 1) + 12 * N
        free, _total = torch.cuda.mem_get_info(self.dev)
        # leave room for what construction allocates after this point: U, the row cache (bounded by 4 * N * C * Hp bytes
        # only in the worst case; a quarter of free memory is kept back instead)
        if need > 0.5 * free:
            return
        cs = self.compact
        counts = self._z((H * C,), torch.int64)
        self._call("coda_b200_compact_index_count", _ptr(cs.ids), self.model_stride, H, N, C, K, _ptr(counts), s)
        off = self._z((H * C + 1,), torch.int64)
        torch.cumsum(counts, 0, out=off[1:])                          # construction-time plumbing
        cursor = off[:-1].clone()
        ent = self._e((H * N * K,), torch.int64)                      # {item u32, float bits} pairs
        rest = self._e((N,), torch.float32)
        self._call("coda_b200_compact_index_fill", _ptr(cs.ids), _ptr(cs.probs), self.model_stride, H, N, C, K,
                   _ptr(cursor), _ptr(ent), _ptr(rest), s, n=2)
        del counts, cursor
        self.cidx = dict(off=off, ent=ent, rest=rest, delta=self._z((N,), torch.int64))

    def _marginals_full(self):
        """coda.py:226-233 as one streaming pass; leaves THIS shard's column sums in ``pisum``."""
        H, N, C, s = self.H, self.N, self.C, self._s()
        if self.compact is not None:
            cs = self.compact
            dt = self._e((H, C, C), torch.float32)                  # D transposed + row sums: construction-time scratch
            rs = self._e((H, C), torch.float32)
            self._call("coda_b200_pi_full_compact", _ptr(cs.ids), _ptr(cs.probs), self.model_stride, _ptr(self.D), H, N, C,
                       self.K, _ptr(dt), _ptr(rs), _ptr(self.U), s, n=3)
            del dt, rs
        else:
            self._pi_full()
        self._call("coda_b200_pi_reduce", _ptr(self.U), N, C, self.fx_shift, None, _ptr(self.pisum),
                   _ptr(self.flags), s)

    def _pi_full(self):
        """coda.py:227-229 over the dense slab: the tcgen05 kernel when the shape allows it (pi_tc.cu), else fp32 SIMT.
        ``CODA_B200_PI_FULL=simt`` forces the SIMT kernel."""
        H, N, C, s = self.H, self.N, self.C, self._s()
        if self._pi_tc is None:
            want = os.environ.get("CODA_B200_PI_FULL", "tc") != "simt"
            # the same views qualify for both element types: an element offset that is a multiple of 4
            ok = getattr(self.lib, self._slab_fn("coda_b200_pi_full_tc_ok"))
            self._pi_tc = bool(want and ok(H, N, C, self.model_stride) and self.preds.data_ptr() % (4 * self.esize) == 0)
            if self._pi_tc:
                self._pi_scratch = self._e((int(self.lib.coda_b200_pi_full_tc_scratch_bytes(H, C)),), torch.uint8)
        if self._pi_tc:
            self._call(self._slab_fn("coda_b200_pi_full_tc"), _ptr(self.preds), self.model_stride, _ptr(self.D), H, N, C, _ptr(self.U),
                       _ptr(self._pi_scratch), _ptr(self.flags), s, n=2)
        else:
            self._call(self._slab_fn("coda_b200_pi_full"), _ptr(self.preds), self.model_stride, _ptr(self.D), H, N, C, _ptr(self.U), s)

    def _build_rows(self):
        H, N, C, W, T, s = self.H, self.N, self.C, self.W, self.T, self._s()
        ent_cnt = self._e((N,), torch.int32)
        heavy_cnt = self._e((N,), torch.int32)
        cls_heavy = self._z((C,), torch.int32)
        self._call("coda_b200_pair_count", _ptr(self.hard), H, N, C, _ptr(ent_cnt), _ptr(heavy_cnt), _ptr(cls_heavy), s)
        heavy = cls_heavy.cpu().numpy().astype(np.int64)        # host sync (construction only)
        n_ent = int(ent_cnt.sum(dtype=torch.int64).item())
        self.n_heavy = int(heavy.sum())
        self.n_entries = n_ent
        self.max_entries = int(ent_cnt.max().item())
        per_cls = 1 + H + heavy
        cls_base = np.zeros(C + 1, dtype=np.int64)
        np.cumsum(per_cls, out=cls_base[1:])
        self.npairs = int(cls_base[-1])                         # == T + n_heavy
        if self.npairs >= 2 ** 31 or n_ent >= 2 ** 31:
            raise NotImplementedError("coda_b200: more than 2^31 rows in one shard")
        self.ent_off = self._z((N + 1,), torch.int32)
        self.heavy_off = self._z((N + 1,), torch.int32)
        torch.cumsum(ent_cnt, 0, out=self.ent_off[1:])          # init-time plumbing
        torch.cumsum(heavy_cnt, 0, out=self.heavy_off[1:])
        del ent_cnt, heavy_cnt
        self.cls_base_host = cls_base
        self.cls_base = torch.from_numpy(cls_base).to(self.dev)
        # tiles of <= 32 (SIMT) or <= 128 (tcgen05) same-class work-list positions
        def make_tiles(width):
            nt = (per_cls + width - 1) // width
            tile_off = np.zeros(C + 1, dtype=np.int64)
            np.cumsum(nt, out=tile_off[1:])
            cls_of_tile = np.repeat(np.arange(C, dtype=np.int64), nt)
            k_in_cls = np.arange(int(tile_off[-1]), dtype=np.int64) - tile_off[cls_of_tile]
            start = cls_base[cls_of_tile] + width * k_in_cls
            cnt = np.minimum(width, per_cls[cls_of_tile] - width * k_in_cls)
            tiles = np.stack([cls_of_tile, start, cnt, np.zeros_like(cnt)], axis=1).astype(np.int32)
            return tile_off, int(nt.max()), torch.from_numpy(tiles).to(self.dev)
        width = 128 if self.use_tc else 32
        tile_off, self.max_cls_tiles, self.tiles = make_tiles(width)
        self.tile_off_host = tile_off
        self.tile_off = torch.from_numpy(tile_off).to(self.dev)
        self.ntiles = int(tile_off[-1])
        self.ent_row = self._e((max(1, n_ent),), torch.int32)
        self.ent_cls = self._e((max(1, n_ent),), torch.int16)
        self.zmask = self._e((self.npairs, W), torch.int32)
        self.row_of = self._e((self.npairs,), torch.int32)
        self.row_cls = self._e((max(1, self.n_heavy),), torch.int16)
        cursor = self._z((C,), torch.int32)
        self._call("coda_b200_pair_fill", _ptr(self.hard), H, N, C, _ptr(self.ent_off), _ptr(self.heavy_off),
                   _ptr(self.cls_base), _ptr(cursor), _ptr(self.ent_row), _ptr(self.ent_cls), _ptr(self.zmask),
                   _ptr(self.row_of), _ptr(self.row_cls), s, n=2)
        # ELL copy of the entry lists when the longest one fits four entries per lane of an 8-lane group
        self.ell_row, self.ell_cls, self.ell_k = None, None, 0
        if 0 < self.max_entries <= 32 and C <= 128:
            self.ell_k = (self.max_entries + 3) // 4 * 4
            self.ell_row = self._e((N, self.ell_k), torch.int32)
            self.ell_cls = self._e((N, self.ell_k), torch.int16)
            self._call("coda_b200_ell_build", _ptr(self.ent_off), _ptr(self.ent_row), _ptr(self.ent_cls), N, self.ell_k,
                       _ptr(self.ell_row), _ptr(self.ell_cls), s)
        self.gain = self._z((self.npairs,), torch.float32)      # information gain of every row (templates first)
        # CODA_B200_FUSED_SCORE=1: one kernel computes the row gains and assembles the per-item EIG (measured slower
        # than the streaming row-gain kernel followed by the 8-lane assembly)
        self.fused_score = os.environ.get("CODA_B200_FUSED_SCORE", "0") == "1"
        self.ph_cache = None
        if self.mode == "incremental":
            need = self.npairs * self.Hp * 4
            free, _total = torch.cuda.mem_get_info(self.dev)
            if need + (2 << 30) > free + torch.cuda.memory_reserved(self.dev) - torch.cuda.memory_allocated(self.dev):
                # the row cache does not fit next to the slab: fall back to recomputing the rows every step
                import warnings
                warnings.warn(f"coda_b200: row cache of {need / 2 ** 30:.1f} GiB does not fit "
                              f"({free / 2 ** 30:.1f} GiB free); falling back to mode='recompute'")
                self.mode = "recompute"
            else:
                self.ph_cache = self._e((self.npairs, self.Hp), torch.float32)

    def _build_shadow(self):
        """Class-major shadow copy of as many models as spare HBM allows (least accurate first), in the slab's element
        type: an fp16 shadow holds twice the models in the same memory."""
        self.shadow, self.slot_of_model, self.n_shadow, self.shadow_cs = None, None, 0, 0
        if self.mode == "recompute_all" or os.environ.get("CODA_B200_SHADOW", "1") == "0" or self.compact is not None:
            return
        H, N, C = self.H, self.N, self.C
        torch.cuda.synchronize(self.dev)
        torch.cuda.empty_cache()
        free, _total = torch.cuda.mem_get_info(self.dev)
        reserve = int(float(os.environ.get("CODA_B200_SHADOW_RESERVE_GB", "8")) * 2 ** 30)
        S, cs = shadow_slots(free - reserve, H, N, C, self.esize)
        cap = os.environ.get("CODA_B200_SHADOW_MODELS")
        if cap is not None:
            S = min(S, int(cap))
        if S <= 0:
            return
        # disagreement of every model with the ensemble pseudo-label: the models that will need gathers most often
        dis = torch.zeros(H, dtype=torch.int64, device=self.dev)
        step = max(1, (64 << 20) // max(1, H))
        for n0 in range(0, N, step):
            blk = self.hard[n0:n0 + step].to(torch.int32) & 0xFFFF
            dis += (blk != self.pseudo[n0:n0 + step, None]).sum(0)
        order = torch.argsort(dis, descending=True, stable=True)[:S].to(torch.int32)
        slot = torch.full((H,), -1, dtype=torch.int32, device=self.dev)
        slot[order.long()] = torch.arange(S, dtype=torch.int32, device=self.dev)
        self.shadow = self._e((S, C, cs), self.preds.dtype)
        self._call(self._slab_fn("coda_b200_shadow_build"), _ptr(self.preds), self.model_stride, H, N, C, _ptr(order), S, cs,
                   _ptr(self.shadow), self._s())
        self.slot_of_model, self.n_shadow, self.shadow_cs = slot, S, cs

    # ------------------------------------------------------------------------ step pieces (enqueue only)
    def _tables(self, lo, hi, sel=False):
        H, C, s = self.H, self.C, self._s()
        if sel:
            self._call("coda_b200_beta_tables", _ptr(self.D), _ptr(self.grid), H, C, self.P, self.hyp_w, 0, 1,
                       _ptr(self.sel), _ptr(self.scratch), _ptr(self.dL), _ptr(self.G0T), _ptr(self.G1T),
                       _ptr(self.PB), _ptr(self.dLb), _ptr(self.Gb), _ptr(self.flags), s, n=3)
            return
        for b0 in range(lo, hi, self.table_batch):
            b1 = min(hi, b0 + self.table_batch)
            self._call("coda_b200_beta_tables", _ptr(self.D), _ptr(self.grid), H, C, self.P, self.hyp_w, b0, b1, None,
                       _ptr(self.scratch), _ptr(self.dL), _ptr(self.G0T), _ptr(self.G1T), _ptr(self.PB),
                       _ptr(self.dLb), _ptr(self.Gb), _ptr(self.flags), s, n=3)

    def _mixture(self):
        self._call("coda_b200_step_mixture", self.st, self._x(), self._s())

    def _pair_rows(self, tile_lo, tile_hi, gains=True, sel=False):
        tail = (_ptr(self.PB), _ptr(self.m0) if gains else None, _ptr(self.pi_hat) if gains else None, self.H,
                _ptr(self.ph_cache), _ptr(self.gain) if gains else None, _ptr(self.sel) if sel else None,
                _ptr(self.tile_off) if sel else None, _ptr(self.flags), self._s())
        if self.use_tc:
            self._call("coda_b200_pair_rows_tc", _ptr(self.tiles), int(tile_lo), int(tile_hi), _ptr(self.zmask),
                       _ptr(self.row_of), _ptr(self.dLb), _ptr(self.Gb), *tail)
        else:
            self._call("coda_b200_pair_rows", _ptr(self.tiles), int(tile_lo), int(tile_hi), _ptr(self.zmask),
                       _ptr(self.row_of), _ptr(self.dL), _ptr(self.G0T), _ptr(self.G1T), *tail)

    def _score(self):
        """coda.py:235-281 + the per-block arg-max of coda.py:306/309 -> ``partials``."""
        if self.scored:
            return
        if self.mode == "incremental":
            if not self.cache_valid:
                self._pair_rows(0, self.ntiles, gains=False)    # fill the row cache once
                self.cache_valid = True
            if self.pending:
                self._cur().wait_event(self.ev_join)            # the class-t rows of the side stream
                self.pending = False
            if self.fused_score:
                self._call("coda_b200_template_gains", _ptr(self.ph_cache), self.H, self.C, _ptr(self.PB), _ptr(self.m0),
                           _ptr(self.pi_hat), _ptr(self.gain), self._s())
            else:                                               # template rows + heavy rows in one stream
                self._call("coda_b200_row_gains", _ptr(self.ph_cache), _ptr(self.row_cls), self.n_heavy, self.H, self.C,
                           _ptr(self.PB), _ptr(self.m0), _ptr(self.pi_hat), _ptr(self.gain), self._s())
        else:
            if self.pending:
                self._cur().wait_event(self.ev_join)
                self.pending = False
            self._pair_rows(0, self.ntiles)
        self._call("coda_b200_gain_eig", _ptr(self.U), self.N, self.C, self.H, _ptr(self.ent_off), _ptr(self.heavy_off),
                   _ptr(self.ent_row), _ptr(self.ent_cls), _ptr(self.ph_cache) if self.fused_score else None,
                   _ptr(self.gain), _ptr(self.PB), _ptr(self.m0), _ptr(self.pi_hat), _ptr(self.labeled),
                   _ptr(self.disagree), self.n_offset, self.max_entries, _ptr(self.ell_row), _ptr(self.ell_cls),
                   self.ell_k, _ptr(self.eig), _ptr(self.partials), _ptr(self.flags), self._s())
        self.scored = True

    def _post_label(self):
        """coda.py:317-319 after ``sel`` / ``jvec`` / D / the gather list are in place (step_select or step_label):
        marginal refresh + the tables that depend on the new D.  incremental / recompute: the class-t tables (and the
        cached rows of the class-t work list) only need the new D, so they are rebuilt on a side stream while the main
        stream does the HBM-bound marginal refresh; the mixture waits for the tables, the next scoring pass for the rows."""
        H, N, C, s = self.H, self.N, self.C, self._s()
        self.scored = False
        self.reported = False
        if self.mode == "recompute_all":
            self._pi_full()
            self._call("coda_b200_pi_reduce", _ptr(self.U), N, C, self.fx_shift, None, _ptr(self.pisum), _ptr(self.flags), s)
            self._tables(0, C)
            self._mixture()
            return
        main = self._cur()
        refresh_rows = self.mode == "incremental" and self.cache_valid
        fork = self.overlap
        if fork:
            self.ev_fork.record(main)
            self.side.wait_event(self.ev_fork)
            ctx = torch.cuda.stream(self.side)
        else:
            ctx = contextlib.nullcontext()
        with ctx:
            self._tables(0, 1, sel=True)
            if fork:
                self.ev_tables.record(self.side)
            if refresh_rows:     # cached rows of the class-t work list (no gains: m0 / pi_hat are not final yet)
                self._pair_rows(0, self.max_cls_tiles, gains=False, sel=True)
            if fork:
                self.ev_join.record(self.side)
        if self.compact is not None and self.cidx is not None:
            ix = self.cidx
            self._call("coda_b200_pi_rank1_index", _ptr(ix["off"]), _ptr(ix["ent"]), _ptr(ix["rest"]), _ptr(self.jvec), H, N, C,
                       _ptr(self.sel), self.lr, self.fx_shift, _ptr(self.terms), _ptr(ix["delta"]), _ptr(self.U),
                       _ptr(self.pisum), _ptr(self.flags), s, n=2)
        elif self.compact is not None:
            cs = self.compact
            self._call("coda_b200_pi_rank1_compact", _ptr(cs.ids), _ptr(cs.probs), self.model_stride, _ptr(self.ens), H, N,
                       C, self.K, _ptr(self.sel), self.lr, self.fx_shift, _ptr(self.terms), _ptr(self.U),
                       _ptr(self.pisum), _ptr(self.flags), s)
        else:
            self._call(self._slab_fn("coda_b200_pi_rank1"), _ptr(self.preds), _ptr(self.ens), H, N, C, _ptr(self.sel), self.lr,
                       self.fx_shift, _ptr(self.terms), _ptr(self.U), _ptr(self.pisum), _ptr(self.flags),
                       4 if fork else 8, self.const_slot, s)
        if fork:
            main.wait_event(self.ev_tables)     # the mixture needs PB[t]; the rows are awaited by the scoring pass
            self.pending = True
        self._mixture()

    # ------------------------------------------------------------------------ host-free loop
    def _bind_labels(self, labels_dev):
        if labels_dev.data_ptr() != self.labels_ptr:
            if labels_dev.dtype != torch.int64 or labels_dev.device != self.dev or labels_dev.numel() < self.n_global:
                raise ValueError("labels_dev must be an int64 tensor of all n_global labels on this shard's device")
            self.st.labels_global = labels_dev.data_ptr()
            self.labels_ptr = labels_dev.data_ptr()
            self._labels_keep = labels_dev
            self.graphs.pop("loop", None)

    def _loop_body(self):
        """select -> posterior update -> scoring pass for the next selection (one graph)."""
        self._call("coda_b200_step_select", self.st, self._x(), self._s())
        self._post_label()
        self._score()

    def device_step(self, labels_dev: torch.Tensor, step: int | None = None, hist_idx=None, hist_q=None):
        """One acquisition step with no host round trip: pick the arg-max (first index on equal values, coda.py:309;
        an isclose tie that the reference would break with random.choice is recorded in ``hist_tie``), look the label
        up on the device (coda/oracle.py:23-24), update the posterior, score the next selection.  Eager launches; see
        ``run_steps`` for the CUDA-graph loop.  ``hist_idx`` / ``hist_q``: optional caller-owned history (slot = step)."""
        with self._on():
            self._bind_labels(labels_dev)
            if step is not None:
                self.step_ctr.fill_(int(step))
            self._score()
            self._loop_body()
            if hist_idx is not None and step is not None:
                hist_idx[step] = self.hist_idx[int(step) % HIST_CAP]
                if hist_q is not None:
                    hist_q[step] = self.hist_q[int(step) % HIST_CAP]

    # The graph loop in phases, so that a front end driving several shards from one thread never blocks on a shard
    # whose peers have not been enqueued yet: prepare (no exchange inside) -> one eager step -> capture -> replays.
    def loop_prepare(self, labels_dev: torch.Tensor):
        with self._on():
            self._bind_labels(labels_dev)
            self._score()

    def loop_ready(self) -> bool:
        return (not self.use_graph) or self.graphs.get("loop") is not None

    def loop_eager(self):
        with self._on():
            self._loop_body()

    def _try_capture(self, key, body):
        """Capture `body` as graph `key`; a failed capture (driver / allocator state) falls back to eager launches."""
        try:
            g, n = self._capture(body)
        except Exception as e:      # nothing was executed during the capture: the device state is still the pre-capture one
            import warnings
            warnings.warn(f"coda_b200: CUDA graph capture failed ({type(e).__name__}: {e}); continuing with eager launches")
            self.use_graph = False
            self.pending, self.scored, self.reported = False, False, False
            torch.cuda.synchronize(self.dev)
            return None, 0
        self.graphs[key] = g
        return g, n

    def loop_capture(self):
        with self._on():
            _g, self.launches_per_step = self._try_capture("loop", self._loop_body)

    def loop_replay(self, k: int = 1):
        with self._on():
            g = self.graphs.get("loop")
            for _ in range(k):
                if g is None:
                    self._loop_body()
                else:
                    g.replay()
            if g is not None:
                self.counters["launches"] += k * self.launches_per_step

    def run_steps(self, k: int, labels_dev: torch.Tensor):
        """``k`` acquisition steps as ``k`` replays of one captured CUDA graph (SURVEY.md 8f rank 2; replaces the
        host loop of main.py:89-94 for offline runs).  History: ``hist_idx/hist_q/hist_tie[step_ctr % HIST_CAP]``."""
        if k <= 0:
            return
        self.loop_prepare(labels_dev)
        if not self.loop_ready():
            self.loop_eager()                                   # warm-up (module loading, attributes) outside capture
            k -= 1
            self.loop_capture()
        self.loop_replay(k)

    def _capture(self, body):
        torch.cuda.synchronize(self.dev)
        g = torch.cuda.CUDAGraph()
        cap_stream = self.stream or torch.cuda.Stream(device=self.dev)
        before = self.counters["launches"]
        if self.pending:                                        # join eager side-stream work before the capture starts
            self._cur().wait_event(self.ev_join)
            self.pending = False
        self.scored = False
        with torch.cuda.graph(g, stream=cap_stream, capture_error_mode="relaxed"):
            body()
            if self.pending:                                    # every forked stream has to rejoin inside the capture
                self._cur().wait_event(self.ev_join)
                self.pending = False
        launches = self.counters["launches"] - before
        self.counters["launches"] = before
        torch.cuda.synchronize(self.dev)
        return g, launches

    # ------------------------------------------------------------------------ API path
    def _report(self):
        """coda.py:306-309: global record + isclose tie list of every shard -> pinned host block (enqueue only)."""
        self._score()
        N, s = self.N, self._s()
        self._call("coda_b200_step_merge", self.st, self._x(), s)
        self._call("coda_b200_ties", _ptr(self.eig), N, _ptr(self.labeled), _ptr(self.disagree), self.n_offset,
                   _ptr(self.bestrec), TIE_CAP, _ptr(self.tie_hdr), _ptr(self.tie_idx), _ptr(self.tie_val), s, n=2)
        self._call("coda_b200_report_gather", _ptr(self.rep), REP_WORDS, _ptr(self.rep_all), self._x(), _ptr(self.flags), s)
        self.rep_host.copy_(self.rep_all, non_blocking=True)
        self.reported = True

    def report(self):
        with self._on():
            if not self.reported:
                self._report()

    def _api_body(self):
        self._call("coda_b200_step_label", self.st, self._x(), self._s())
        self._post_label()
        self._report()

    # add_label in phases (a front end driving several shards calls each phase on every shard before the next, so
    # that nothing blocks the host -- a graph capture synchronises the device -- while a peer's kernels are missing):
    #   label_stage    stage the host-chosen (idx, class) record: pinned ring slot -> device, no exchange inside
    #   api_capture    (once, after two eager steps) capture label + refresh + scoring pass + report as one graph
    #   label_run      replay the graph, or enqueue the same kernels one by one
    def label_stage(self, idx_global: int, true_class: int):
        with self._on():
            k = self.sel_pos
            self.sel_pos = (k + 1) % len(self.sel_events)
            if self.sel_events[k] is not None:
                self.sel_events[k].synchronize()                # the copy that last used this slot has executed
            loc = idx_global - self.n_offset
            self.sel_ring[k, 0] = loc if 0 <= loc < self.N else -1
            self.sel_ring[k, 1] = true_class
            self.sel.copy_(self.sel_ring[k], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self._cur())
            self.sel_events[k] = ev

    def api_graph_wanted(self) -> bool:
        return (self.use_graph and self.graphs.get("api") is None and self.graphs.get("api_warm", 0) >= 2
                and (self.cache_valid or self.mode != "incremental"))

    def api_capture(self):
        with self._on():
            _g, self.launches_per_api_step = self._try_capture("api", self._api_body)

    def label_run(self, eager_report: bool = True):
        with self._on():
            if not eager_report:
                self._call("coda_b200_step_label", self.st, self._x(), self._s())
                self._post_label()
                return
            g = self.graphs.get("api") if self.use_graph else None
            if g is not None:
                if self.pending:
                    self._cur().wait_event(self.ev_join)
                    self.pending = False
                g.replay()
                self.counters["launches"] += self.launches_per_api_step
                self.scored, self.reported = True, True
                return
            self.graphs["api_warm"] = self.graphs.get("api_warm", 0) + 1
            self._api_body()

    def label(self, idx_global: int, true_class: int, eager_report: bool = True):
        """coda.py:316-319 for a host-chosen (idx, class): stage the record, posterior update, marginal refresh and --
        so that the next get_next_item_to_label only has to wait -- the next scoring pass + report.  Enqueue only."""
        self.label_stage(idx_global, true_class)
        if eager_report and self.api_graph_wanted():
            self.api_capture()
        self.label_run(eager_report)

    def fetch(self):
        """Wait for the report block and decode it.  Returns a dict of host values."""
        with self._on():
            if not self.reported:
                self._report()
            self._cur().synchronize()
        allr = self.rep_host.numpy()                            # (world, REP_WORDS)
        r0 = allr[0]
        flags = 0
        for r in allr:
            flags |= int(r[0:1].view(np.int32)[0])
        use_a = int(r0[3]) > 0                                  # the record is the merged (global) one on every shard
        bits = int(r0[1] if use_a else r0[4])
        best_val = float(np.array([bits & 0xFFFFFFFF], dtype=np.uint32).view(np.float32)[0])
        n_ties = int(sum(int(r[9]) for r in allr))
        idxs, vals = [], []
        for r in allr:
            k = min(int(r[9]), TIE_CAP)
            idxs.append(r[12:12 + k])
            vals.append(r[12 + TIE_CAP:].view(np.float32)[:k])
        return dict(flags=flags, use_a=use_a, n_cand=int(r0[3]), best_val=best_val,
                    best_idx=int(r0[2] if use_a else r0[5]), n_ties=n_ties,
                    tie_min=int(min(int(r[10]) for r in allr)), tie_idx=np.concatenate(idxs).copy(),
                    tie_val=np.concatenate(vals).copy())

    def check_flags(self, sync=False, flags=None):
        if flags is None:
            flags = int(self.flags.item()) if sync else 0
        if not flags:
            return
        if flags & nat.FLAG_ROWSUM_WARN:                        # util.py:37-39 prints a warning and carries on
            print("[WARN] Pbest(beta) normalized rows not normalised")
            self.flags.bitwise_and_(~nat.FLAG_ROWSUM_WARN)
            flags &= ~nat.FLAG_ROWSUM_WARN
            if not flags:
                return
        if flags & nat.FLAG_PIPELINE_TIMEOUT:
            raise RuntimeError("coda_b200: the tensor-core marginal pass (k_pi_full_tc) stopped; its result is invalid")
        if flags & nat.FLAG_XCHG_TIMEOUT:
            raise RuntimeError("coda_b200: a shard did not arrive at an exchange within 2 s (peer crashed or not launched)")
        if flags & nat.FLAG_NO_CANDIDATE:
            raise RuntimeError("no unlabeled items left to select from")
        if flags & nat.FLAG_NEGATIVE_PROB:
            raise RuntimeError("Pbest(beta) normalized has negatives")                 # util.py:33-35
        if flags & nat.FLAG_RANGE_INPUT and not flags & nat.FLAG_NONFINITE_INPUT:
            raise ValueError("coda_b200: dataset.preds must hold post-softmax scores in [0, 1] (coda/datasets.py:6)")
        names = [v for k, v in nat.FLAG_NAMES.items() if flags & k]
        raise RuntimeError(f"[NUMERIC ERROR] {', '.join(names)} has bad values (NaN/Inf)")   # util.py:20-25

    def mark_labeled(self, idx_global: int):
        loc = idx_global - self.n_offset
        with self._on():
            if 0 <= loc < self.N:
                self.labeled[loc] = 1
            self.scored = False
            self.reported = False

    # ------------------------------------------------------------------------- read-outs
    def pbest(self) -> torch.Tensor:
        with self._on():
            return self.m0[: self.H].clone().view(1, self.H)    # coda.py:329 -> (1, H)

    def pi_hat_xi(self) -> torch.Tensor:
        with self._on():
            xi = torch.empty_like(self.U)
            scratch = torch.zeros_like(self.pisum)
            self._call("coda_b200_pi_reduce", _ptr(self.U), self.N, self.C, self.fx_shift, _ptr(xi), _ptr(scratch),
                       _ptr(self.flags), self._s())
            return xi

    # ------------------------------------------------------------------------- checkpoint
    def state_tensors(self):
        """Everything a resumed run cannot rebuild from the slab alone (SURVEY.md 8f rank 4): the posterior, the
        un-normalised marginals they imply, the label mask and the device step counter."""
        return {"D": self.D, "U": self.U, "labeled": self.labeled, "pisum": self.pisum, "step_ctr": self.step_ctr}

    def __del__(self):
        try:
            _release_const_slot(self.dev.index, getattr(self, "const_slot", -1))
        except Exception:
            pass

    def close(self):
        """Release the graphs, the mailbox and every device buffer of this shard (the object is unusable afterwards)."""
        self.graphs.clear()
        _release_const_slot(self.dev.index, self.const_slot)
        self.const_slot = -1
        if self._mailbox is not None:
            self._mailbox.close()
            self._mailbox = None
        for k, v in list(self.__dict__.items()):
            if isinstance(v, torch.Tensor) or k in ("preds", "compact", "st", "xchg", "_labels_keep", "cidx"):
                setattr(self, k, None)


def build_engines(shards, group, **kw):
    """Construct the shards of one task in lock-step (``shards``: list of (preds, n_offset) on this process).
    Phase order matters once peers spin on each other: every shard enqueues its mixture before any host sync."""
    n_global = kw.pop("n_global")
    own = len(shards) > 1
    engines = [Engine(p, n_offset=off, n_global=n_global, world=group.world, own_stream=own, **kw) for p, off in shards]
    for e in engines:
        e.construct_scan()
    group.attach(engines)
    group.allreduce_sum_([e.conf_buf for e in engines])         # coda.py:42 sums over ALL items
    for e in engines:
        e.construct_posterior()
    for e in engines:
        e.construct_mixture()
    for e in engines:
        e.construct_finish()
    return engines
