#!/usr/bin/env python
"""bench.py -- acquisition steps/sec of the CODA hot path on B200 (BASELINE.json metric).

    python bench.py --gpus 1 --steps 50 --warmup 5                 # our arm, one JSON line
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W  # N-axis sharded over N GPUs
    python bench.py --impl reference --steps 2 --warmup 1          # reference algorithm on the host cores
    python bench.py --steps 50 --warmup 5 --dump-outputs DIR       # + what the timed loop computed, as DIR/*.npy

One step = get_next_item_to_label() -> oracle(idx) -> add_label() -> get_best_model_prediction()
(reference main.py:91-94).  Workload: synthetic M=256, N=1e6, C=100 (BASELINE.json configs[2]),
strong scaling: the N axis is split over the ranks.

  value  steps/s of the host-free device loop (labels resident in HBM; pick = arg-max, first index on equal values),
         CUDA-event timed, max over ranks;
  e2e    steps/s through the public ``coda_b200.CODA`` API with a HOST oracle: per step a pinned
         H2D copy of {idx, class} and a D2H read of the selection report and the best-model index;
  roofline  the dominant kernel of the timed region, CUDA events on the launching stream;
  cpu_baseline  the oracle (CPU restatement of coda/coda.py) on a bounded sample, extrapolated.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "cfg3": dict(H=256, N=1_000_000, C=100),     # BASELINE.json configs[2] / configs[3]
    "cfg2": dict(H=64, N=50_000, C=10),          # BASELINE.json configs[1] (parity config)
    "mini": dict(H=32, N=20_000, C=10),          # smoke-sized
    # BASELINE.json configs[4]: 16.4 TB as dense fp32 -- runs from the compact top-K slab (98 GB over 8 GPUs); perf-only,
    # the reference cannot run it (coda.py:227 materialises a second slab)
    "cfg5": dict(H=1024, N=4_000_000, C=1000, K=4, compact=True),
    "cfg5mini": dict(H=1024, N=131_072, C=1000, K=4, compact=True),
    "cfg5shard": dict(H=1024, N=500_000, C=1000, K=4, compact=True),     # what one of the 8 GPUs of cfg5 holds
}
METRIC = "acquisition steps/sec (M=256,N=1e6,C=100)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default="incremental", choices=["incremental", "recompute", "recompute_all"])
    ap.add_argument("--extra-modes", default="recompute", help="comma list of other modes to time briefly ('' = none)")
    ap.add_argument("--extra-steps", type=int, default=5)
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = same as --steps")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--dense", action="store_true", help="worst-case synthetic slab (wrong class uniform)")
    ap.add_argument("--no-dense-extra", dest="dense_extra", action="store_false",
                    help="skip the dense worst-case slab that the N=1 run reports under modes.dense_slab")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the device loop computed as DIR/<name>.npy (rank 0)")
    return ap.parse_args()


DUMP_ARRAY_BYTES = 16 << 20     # per array: with three item- or class-sized arrays a dump stays under 64 MB


def dump_outputs(out_dir, arrays):
    """Write every tensor as ``out_dir/<name>.npy``: floating point as float32 (float64 stays), integers as float64.
    Larger than DUMP_ARRAY_BYTES, an array is replaced by a fixed, seeded sample of its rows (all axes but the last
    flattened), and the row numbers go to ``<name>_rows.npy``: two builds given the same arguments sample the same
    rows, so their dumps compare element for element."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = torch.as_tensor(t)
        t = t.float() if t.is_floating_point() and t.dtype != torch.float64 else t.double()
        rows = t.reshape(-1, t.shape[-1]) if t.dim() > 1 else t.reshape(-1, 1)
        if rows.numel() * rows.element_size() > DUMP_ARRAY_BYTES:
            k = max(1, DUMP_ARRAY_BYTES // (rows.shape[1] * rows.element_size()))
            pick = np.sort(np.random.default_rng(0).choice(rows.shape[0], size=k, replace=False))
            np.save(os.path.join(out_dir, name + "_rows.npy"), pick.astype(np.float64))
            t = rows[torch.from_numpy(pick).to(rows.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clock / throttle-reason sampler running DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def count(self):
        try:
            with open(self.f.name) as f:
                return sum(1 for _ in f)
        except Exception:
            return 0

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().strip().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ---------------------------------------------------------------------------------------------------
_CPU_SEL = {}


def host_cores():
    """Cores this process may really use: min(scheduler affinity, cgroup CPU quota).  A GPU lease is often a
    cgroup-limited slice of a big host; sizing the thread pool from the affinity mask alone oversubscribes it."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:                                                   # cgroup v2
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, -(-int(quota) // int(period))))
    except Exception:
        try:                                               # cgroup v1
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0:
                n = min(n, max(1, -(-quota // period)))
        except Exception:
            pass
    return max(1, n)


def workload_string(args, wl, world):
    form = f", compact top-{wl['K']} slab" if wl.get("compact") else ""
    return (f"synthetic M={wl['H']} N={wl['N']} C={wl['C']} ({args.workload}{', dense' if args.dense else ''}{form}), "
            f"N-axis sharded over {world} GPU(s)")


class CpuReference:
    """Reference algorithm (oracle port of coda/coda.py) on the host cores: bounded samples, extrapolated.

    A full CPU step at cfg3 is ~days (6.55e12 quadrature cells), so one *sample* times the body of the EIG loop
    (coda.py:262-279) on a small batch of candidates of a 512-item sub-slab; `update_pi_hat`, `_prefilter` and
    `get_pbest` are timed once on the sub-slab.  Everything is scaled linearly to N items (the loop body is
    independent per item and equal-cost).  Every sample is bounded by WALL CLOCK: the batch size is calibrated
    from a 1-item probe so that a sample fits its time slice on whatever core budget this box grants."""

    N_SUB = 512

    def __init__(self, wl, seed, dense=False, threads=None):
        import torch
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import coda_oracle
        from coda_b200.synth import synth
        self.torch, self.ora = torch, coda_oracle
        self.cores = threads or host_cores()
        torch.set_num_threads(self.cores)        # torchrun pins OMP_NUM_THREADS=1; the reference uses what it is given
        self.H, self.N, self.C = wl["H"], wl["N"], wl["C"]
        self.n_sub = min(self.N, self.N_SUB)
        t0 = time.perf_counter()
        preds, _ = synth(self.H, self.N, self.C, seed, n_lo=0, n_hi=self.n_sub, dense=dense)
        self.sel = coda_oracle.OracleSelector(preds)
        t1 = time.perf_counter()
        self.cand = self.sel.candidates()
        self.t_pref = time.perf_counter() - t1
        t1 = time.perf_counter()
        coda_oracle.consensus_marginals(self.sel.dirichlets, self.sel.preds)
        self.t_pi = time.perf_counter() - t1
        t1 = time.perf_counter()
        self.sel.get_pbest()
        self.t_pb = time.perf_counter() - t1
        # probes with 1 and 3 items: the loop body costs a + b * items (a = the 255-iteration cdf loop and the other
        # per-chunk launches, coda.py:98-101, amortised by the reference over 100 items; b = per-item arithmetic)
        t1 = time.perf_counter()
        self.sel.eig_scores(self.cand[:1], chunk=1)
        p1 = time.perf_counter() - t1
        t1 = time.perf_counter()
        self.sel.eig_scores(self.cand[1:4], chunk=3)
        p3 = time.perf_counter() - t1
        self.s_per_item = max(1e-5, (p3 - p1) / 2)
        self.s_fixed = max(0.0, p1 - self.s_per_item)
        self.setup_s = time.perf_counter() - t0
        self.cursor = 4

    def sample(self, seconds):
        """Time one batch of the EIG loop sized to ~`seconds`; -> dict(step_seconds, items, cells_per_s, ...)."""
        chunk = self.ora.CHUNK
        bs = int(max(1, min(chunk, (0.8 * seconds - self.s_fixed) / self.s_per_item, len(self.cand))))
        if self.cursor + bs > len(self.cand):
            self.cursor = 0
        ids = self.cand[self.cursor:self.cursor + bs]
        self.cursor += bs
        t0 = time.perf_counter()
        self.sel.eig_scores(ids, chunk=bs)
        dt = time.perf_counter() - t0
        per_item = (dt - self.s_fixed) / len(ids) if dt > 2 * self.s_fixed else dt / len(ids)
        self.s_per_item = max(1e-6, per_item)
        chunk_s = dt if len(ids) == chunk else self.s_fixed + per_item * chunk     # one 100-item chunk as the reference runs it
        frac_cand = len(self.cand) / self.n_sub
        step_s = chunk_s * (self.N * frac_cand / chunk) + (self.t_pi + self.t_pref) * (self.N / self.n_sub) + 2 * self.t_pb
        cells = len(ids) * self.C * self.H * self.ora.QUAD_NODES
        return dict(step_seconds=step_s, items=len(ids), seconds=dt, cells_per_s=cells / dt)

    def describe(self, samples):
        items = sum(s["items"] for s in samples)
        secs = sum(s["seconds"] for s in samples)
        cps = sum(s["cells_per_s"] * s["seconds"] for s in samples) / max(secs, 1e-9)
        return (f"extrapolated: {len(samples)} sample(s), {items} items of the EIG loop body (coda.py:262-279) in {secs:.1f}s "
                f"({cps:.3g} cells/s; per-chunk overhead {self.s_fixed * 1e3:.0f} ms amortised over 100 items as the reference does) "
                f"+ update_pi_hat + prefilter + get_pbest timed once on a {self.n_sub}-item sub-slab, "
                f"scaled linearly to N={self.N}; {self.cores} torch threads (cgroup-aware)")


def cpu_baseline(wl, seconds, seed, dense=False):
    """`cpu_baseline` leg of the GPU arm (rank 0, N=1): a few wall-clock-bounded samples, ~`seconds` in total."""
    key = (wl["H"], wl["N"], wl["C"], seed, dense)
    if key not in _CPU_SEL:
        _CPU_SEL[key] = CpuReference(wl, seed, dense)
    ref = _CPU_SEL[key]
    n = 3
    samples = [ref.sample(seconds / n) for _ in range(n)]
    step_s = statistics.mean(s["step_seconds"] for s in samples)
    return dict(value=1.0 / step_s, unit="steps/s", cores=ref.cores, kind="port", sample=ref.describe(samples))


REFERENCE_BUDGET_S = 75.0     # wall-clock budget of all timed + warm-up samples of `--impl reference`


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port; the Python reference cannot travel to
    the GPU box) on this box's host cores.  Rank 0 only.  Whole run: set-up (~10-30 s) + <= REFERENCE_BUDGET_S."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    t_start = time.perf_counter()
    ref = CpuReference(wl, args.seed, args.dense)
    n = max(1, args.warmup + args.steps)
    per = max(0.05, min(args.cpu_seconds, REFERENCE_BUDGET_S / n))
    deadline = t_start + ref.setup_s + REFERENCE_BUDGET_S
    vals = []
    for i in range(n):
        # never start a sample that cannot finish before the deadline: shrink it, and if nothing is left reuse the
        # running estimate (the loop body is equal-cost per item, so a skipped sample changes nothing but noise)
        left = deadline - time.perf_counter()
        if left < ref.s_per_item and vals:
            r = dict(vals[-1], items=0, seconds=0.0)
        else:
            r = ref.sample(min(per, max(left, ref.s_per_item)))
        if i >= args.warmup:
            vals.append(r)
    step_s = statistics.mean(v["step_seconds"] for v in vals)
    v = 1.0 / step_s
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "steps/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(args, wl, world), "mode": "reference-cpu"},
        "cpu_baseline": {"value": v, "unit": "steps/s", "cores": ref.cores, "kind": "port",
                         "sample": ref.describe([x for x in vals if x["items"]] or vals)},
        "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.perf_counter() - t_start,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
HOT = {   # C-ABI entry point -> kernel name printed in the roofline line
    "coda_b200_row_gains": "k_row_gains", "coda_b200_gain_eig": "k_eig_assemble_g8", "coda_b200_pi_rank1_compact": "k_pi_rank1_compact", "coda_b200_pi_rank1_index": "k_r1i_scatter+k_r1i_rows", "coda_b200_pi_rank1": "k_pi_rank1", "coda_b200_pair_rows_tc": "k_pair_rows_tc",
    "coda_b200_pair_rows": "k_pair_rows", "coda_b200_pi_full": "k_pi_full", "coda_b200_template_gains": "k_template_gains",
    "coda_b200_beta_tables": "k_beta_nodes+k_beta_combine+k_pb_normalize", "coda_b200_step_select": "k_step_select",
    "coda_b200_step_mixture": "k_step_mixture",
}


def gathered_models(eng):
    """Models in the rank-1 gather list of the last step (two terms per model with the majority shortcut)."""
    try:
        nt, tp = (int(x) for x in eng.terms[:2].tolist())
        return max(1, nt // 2 if tp >= 0 else nt)
    except Exception:
        return eng.H


def algorithmic_bytes(eng):
    """Algorithmic bytes per launch, per shard (DESIGN.md section 4)."""
    H, N, C, Hp = eng.H, eng.N, eng.C, eng.Hp
    ent, heavy = eng.n_entries, eng.n_heavy
    lists = 6 * N * eng.ell_k if eng.ell_row is not None else 6 * ent + 8 * N
    return {
        # the cached row of every heavy (item, class) + its class id; writes one gain per row
        "coda_b200_row_gains": 4 * eng.npairs * Hp + 2 * heavy + 4 * eng.npairs,
        # U rows + entry lists + one gain per entry + candidate masks; writes eig
        "coda_b200_gain_eig": ((4 * heavy * Hp) if getattr(eng, "fused_score", False) else 0) + 4 * N * C + lists + 4 * ent
                              + 2 * N + 4 * N,
        # one 24-byte entry per gathered model and item (the models that disagree with the majority on the labeled item;
        # read from the gather list of the last step) + the U row pass + the ensemble column
        "coda_b200_pi_rank1_compact": 6 * getattr(eng, "K", 4) * gathered_models(eng) * N + 4 * N * C + 8 * N,
        # inverted index: H lists of ~N K / C entries (8 B) + rest sums + the int64 scatter target (read, cleared) + the U row pass
        "coda_b200_pi_rank1_index": 8 * H * N * getattr(eng, "K", 4) // max(1, C) + 4 * N + 16 * N + 4 * N * C + 4 * N,
        # one float per (model, item) + the U row pass (read all, write one column) + the ensemble column
        "coda_b200_pi_rank1": 4 * H * N + 4 * N * C + 4 * N + 4 * N,
        "coda_b200_pi_full": 4 * H * N * C + 4 * N * C,
        "coda_b200_template_gains": 4 * eng.T * Hp + 4 * eng.T,
    }


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    # stdout carries exactly one JSON line: park the real stdout and point fd 1 at stderr while libraries
    # (NCCL's version banner, torch warnings) may write
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    from coda_b200 import CODA, SyntheticDataset
    from coda_b200.dist import LocalComm, TorchComm

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with: python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ...")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"      # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
        comm = TorchComm()
    else:
        comm = LocalComm()
    wl = WORKLOADS[args.workload]
    H, N, C = wl["H"], wl["N"], wl["C"]
    if args.steps + args.warmup + 64 >= N:
        raise SystemExit("bench: steps + warmup must stay below the number of items")
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak, peak_src = (peaks["hbm_gbs"], "measured") if "hbm_gbs" in peaks else (6650.0, "fallback")
    tf_peak = peaks.get("bf16_tflops_sustained", 1400.0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def dataset(dense):
        t = time.time()
        if wl.get("compact"):
            from coda_b200 import SyntheticCompactDataset
            ds = SyntheticCompactDataset(H, N, C, K=wl["K"], seed=args.seed, device=dev, rank=rank, world=world)
        else:
            ds = SyntheticDataset(H, N, C, seed=args.seed, device=dev, dense=dense, rank=rank, world=world)
        torch.cuda.synchronize()
        return ds, ds.labels.to(dev), ds.labels_host.numpy(), time.time() - t

    def make(ds, mode):
        random.seed(0)
        t = time.time()
        s = CODA(ds, mode=mode, comm=comm)
        torch.cuda.synchronize()
        return s, time.time() - t

    def graph_loop(sel, labels_dev, warm, steps):
        """`value`: host-free loop, one CUDA-graph replay per step, exchanges inside the kernels."""
        eng = sel.engine
        sel.run_steps(max(warm, 2), labels_dev)            # warm-up (>= 2: the first step is eager, then the capture)
        barrier()
        launches0 = eng.counters["launches"]
        wait0 = eng._mailbox.epoch[4:8].clone() if eng._mailbox is not None else None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        sel.run_steps(steps, labels_dev)
        e1.record()
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1))
        eng.check_flags(sync=True)
        if wait0 is not None:    # time the step kernels spent waiting for the peers' contributions (latency + skew), this rank
            w = (eng._mailbox.epoch[4:8] - wait0).cpu().tolist()
            graph_loop.exchange = {"argmax_record_ms_per_step": w[0] / 1e6 / steps, "marginal_sums_ms_per_step": w[1] / 1e6 / steps}
        return ms, eng.counters["launches"] - launches0

    def eager_profile(sel, labels_dev, steps):
        """Per-kernel CUDA-event times over a few eager steps (same kernels, launched one by one; not part of `value`)."""
        eng = sel.engine
        eng.loop_prepare(labels_dev)
        barrier()
        eng.start_profile()
        for _ in range(steps):
            eng.loop_eager()
        prof = eng.stop_profile()
        barrier()
        return prof

    def api_loop(sel, labels_host, warm, steps):
        """main.py:91-94 with a host oracle; every step copies {idx, class} H2D from pinned memory and reads
        the selection report + best model back."""
        best_host = torch.zeros(1, dtype=torch.int64).pin_memory()
        picks = []

        def one():
            idx, q = sel.get_next_item_to_label()
            t = int(labels_host[idx])                          # oracle(idx), host-resident labels
            sel.add_label(idx, t, q)
            b = sel.get_best_model_prediction()
            best_host.copy_(b.view(1), non_blocking=True)
            torch.cuda.current_stream().synchronize()
            picks.append((idx, int(best_host[0])))
        for _ in range(warm):
            one()
        barrier()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            one()
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = max_over_ranks(max(e0.elapsed_time(e1), wall * 1e3))
        return ms, picks

    def kernel_table(prof):
        return {k.replace("coda_b200_", ""): {"avg_ms": v[1] / max(1, v[0]), "max_ms": v[2], "launches_per_step": v[0] / max(1, prof_steps)}
                for k, v in prof.items()}

    def roofline(eng, prof, ms_step, mode):
        if not prof:
            return None
        dom = max(prof, key=lambda k: prof[k][1])
        cnt, tot, mx = prof[dom]
        avg_ms = tot / max(1, cnt)
        alg = algorithmic_bytes(eng)
        base = {"kernel": HOT.get(dom, dom), "avg_launch_ms": avg_ms, "share_of_step": (tot / prof_steps) / ms_step,
                "peak_source": peak_src, "traffic": None}
        if dom in alg:
            ach = alg[dom] / (avg_ms * 1e-3) / 1e9
            base.update(bound="hbm", achieved=ach, peak=hbm_peak, unit="GB/s", frac=ach / hbm_peak,
                        algorithmic_bytes_per_launch=alg[dom])
        elif dom == "coda_b200_pair_rows_tc":
            # 9 bf16 MMAs of 128 x 256 x Hp (3 dL limbs) / 128 x Hp x 256 (2 tables x 3 cross terms) per 128-row tile
            tiles = eng.ntiles if mode != "incremental" else max(1, eng.ntiles // C)
            flops = 9 * 2 * 128 * 256 * eng.Hp * tiles
            ach = flops / (avg_ms * 1e-3) / 1e12
            base.update(bound="tensor", achieved=ach, peak=tf_peak, unit="TFLOP/s", frac=ach / tf_peak,
                        algorithmic_flops_per_launch=flops)
        else:
            base.update(bound="hbm", achieved=None, peak=hbm_peak, unit="GB/s", frac=None)
        try:    # measured DRAM traffic of the same kernel/config from the committed ncu capture (not measurable live)
            tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic_r2.json")))
            ent = tr.get(f"{args.workload}/{world}/{mode}", {}).get(base["kernel"])
            if ent:
                base["traffic"], base["traffic_source"] = ent, "profiles/r2_step_kernels_ncu.txt"
        except Exception:
            pass
        return base

    # ---- our arm -------------------------------------------------------------------------------------
    ds, labels_dev, labels_host, t_gen = dataset(args.dense)
    sel, t_init = make(ds, args.mode)
    eng = sel.engine
    sampler = ClockSampler(local_rank) if rank == 0 else None
    graph_loop.exchange = None
    ms, launches = graph_loop(sel, labels_dev, args.warmup, args.steps)
    exchange = graph_loop.exchange
    value = args.steps / (ms / 1e3)
    picks_dev = sel.history()[0][-(args.steps):].tolist()
    ties_dev = int(sel.history()[2].sum())
    if args.dump_outputs:
        if rank == 0:   # with several ranks, eig and pi_hat_xi are rank 0's shard of the item axis
            h_idx, h_q, h_tie = sel.history()
            dump_outputs(args.dump_outputs, {
                "history_idx": h_idx[-args.steps:], "history_q": h_q[-args.steps:], "history_tie": h_tie[-args.steps:],
                "best_model": eng.best_model[:1], "pbest": sel.get_pbest(),
                "pi_hat": sel.pi_hat, "dirichlets": sel.dirichlets, "eig": sel.eig, "pi_hat_xi": sel.pi_hat_xi})
        barrier()

    prof_steps = min(10, args.steps)
    prof = eager_profile(sel, labels_dev, prof_steps)
    roof = roofline(eng, prof, ms / args.steps, args.mode)

    e2e_steps = args.e2e_steps or min(args.steps, 200)
    ms_e2e, picks_api = api_loop(sel, labels_host, max(3, min(args.warmup, 5)), e2e_steps)
    # the clock sampler has been running since before the warm-up; a very short run may end before nvidia-smi has
    # produced samples, so keep the same load on (untimed) until a few exist
    t_wait = time.time()
    while True:
        more = torch.tensor([1 if (sampler is not None and sampler.count() < 5 and time.time() - t_wait < 3.0) else 0],
                            device=dev)
        if world > 1:
            dist.broadcast(more, src=0)        # every rank runs the same number of extra steps
        if not int(more.item()):
            break
        sel.run_steps(20, labels_dev)
        torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else {}
    e2e = e2e_steps / (ms_e2e / 1e3)
    h2d = 16
    d2h = eng.rep_host.numel() * 8 + 8
    info = dict(pairs=eng.npairs, heavy=eng.n_heavy, ent=eng.n_entries, n_loc=eng.N, shadow=eng.n_shadow,
                tc=bool(eng.use_tc), mode=eng.mode)
    kernels = kernel_table(prof)

    def marginals_full(eng):
        """The construction / recompute_all pass (coda.py:227-229) on this shard: the tcgen05 kernel beside the fp32 SIMT
        kernel, CUDA events around one launch each (U is rewritten with the same values the steps maintained)."""
        if eng.compact is not None or not eng._pi_tc:
            return None
        out = {}
        for name, use_tc in (("k_pi_full_tc", True), ("k_pi_full", False)):
            eng._pi_tc = use_tc
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            with eng._on():
                st = eng._cur()
                a.record(st)
                eng._pi_full()
                b.record(st)
            torch.cuda.synchronize()
            t = a.elapsed_time(b)
            out[name] = {"ms": t, "slab_GB_per_s": 4.0 * eng.H * eng.N * eng.C / (t * 1e-3) / 1e9,
                         "fp32_equiv_TFLOP_per_s": 2.0 * eng.H * eng.N * eng.C * eng.C / (t * 1e-3) / 1e12}
        eng._pi_tc = True
        with eng._on():
            eng._pi_full()                                       # leave the tensor-core result in U, as construction did
        torch.cuda.synchronize()
        eng.check_flags(sync=True)
        return out
    marg = marginals_full(eng) if world == 1 else None

    extra = {}
    extra_list = [x for x in args.extra_modes.split(",") if x and x != args.mode]
    import gc
    for m in extra_list:                                        # other modes on the same slab, a few steps each
        sel.close()
        del sel, eng
        gc.collect()
        torch.cuda.empty_cache()
        sel, t_i = make(ds, m)
        eng = sel.engine
        ms_m, _ = graph_loop(sel, labels_dev, 2, args.extra_steps)
        prof_steps = min(3, args.extra_steps)
        pm = eager_profile(sel, labels_dev, prof_steps)
        extra[m] = {"value": args.extra_steps / (ms_m / 1e3), "unit": "steps/s", "ms_per_step": ms_m / args.extra_steps,
                    "init_s": t_i, "roofline": roofline(eng, pm, ms_m / args.extra_steps, m), "kernel_ms": kernel_table(pm)}
    if args.dense_extra and not args.dense and world == 1 and not wl.get("compact"):
        # SURVEY 8(d): the dense worst case (wrong class uniform over all C) beside the default slab
        sel.close()
        del sel, eng, ds, labels_dev
        gc.collect()
        torch.cuda.empty_cache()
        ds2, lab2, _lh2, _ = dataset(True)
        sel, t_i = make(ds2, args.mode)
        eng = sel.engine
        ms_d, _ = graph_loop(sel, lab2, 3, args.extra_steps * 2)
        prof_steps = min(3, args.extra_steps)
        pd = eager_profile(sel, lab2, prof_steps)
        extra["dense_slab"] = {"value": args.extra_steps * 2 / (ms_d / 1e3), "unit": "steps/s", "mode": eng.mode,
                               "ms_per_step": ms_d / (args.extra_steps * 2), "init_s": t_i,
                               "nnz_frac": eng.n_entries / max(1, eng.N) / C, "heavy_rows": eng.n_heavy,
                               "roofline": roofline(eng, pd, ms_d / (args.extra_steps * 2), eng.mode),
                               "kernel_ms": kernel_table(pd)}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not wl.get("compact"):   # rank 0, N=1 only (the reference arm covers N>1)
        cpu = cpu_baseline(wl, args.cpu_seconds, args.seed, args.dense)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": workload_string(args, wl, world),
                "mode": info["mode"], "l2": "per-step working set (row cache + U + slab gather) >> 126 MB L2; no flush needed",
                "loop": "CUDA graph, one replay per step; shards exchange through peer memory inside the step kernels",
                "tie_rule_value": "arg-max, first index (device loop); isclose ties in the timed run: %d" % ties_dev,
                "tie_rule_e2e": "random.choice (coda.py:308)",
                "rows": info["pairs"], "heavy_rows": info["heavy"], "tensor_core_rows": info["tc"],
                "entries_per_item": info["ent"] / max(1, info["n_loc"]), "nnz_frac": info["ent"] / max(1, info["n_loc"]) / C,
                "gen_s": t_gen, "init_s": t_init, "shadow_models": info["shadow"],
            },
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": "steps/s", "ms_per_step": ms_e2e / e2e_steps, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps},
            "gpu_launches": launches,
            "roofline": roof,
            "kernel_ms": kernels,
            "exchange_wait": exchange,
            "marginals_full": marg,
            "modes": extra,
            "cpu_baseline": cpu,
            "first_picks": {"device_loop": picks_dev[:8], "api": [p[0] for p in picks_api[:8]]},
        }
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
