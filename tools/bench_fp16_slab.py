"""fp16 slab against its fp32 upcast at cfg3 (synthetic 256 x 1e6 x 100) on one GPU, plus a capacity leg.

    python tools/bench_fp16_slab.py [--steps 500] [--reps 2] [--out DIR]

Both arms run on the SAME values (the fp16 slab and its exact fp32 upcast), so they follow the same trajectory and do
the same per-step work.  Arms alternate (fp16, fp32, fp16, fp32, ...) in one process; only the running arm's slab is
resident (each is rebuilt from the other, exactly, between arms), and every selector is closed before the next is built.
Per arm: CUDA-event times of the construction kernels, shadow model count, device memory in use, the rank-1 refresh time
per step (eager steps), host-free steps/s over ``--steps`` graph replays, and the final state, which must be equal
across arms.  Capacity leg: 256 x 2.5e6 x 100 as fp16 (its fp32 slab, 256 GB, does not fit one B200): build it, run
``--cap-steps`` steps, report memory and steps/s; if it does not fit, the largest N tried that does.
Prints one JSON document (and writes it to DIR/bench_fp16_slab.json with ``--out``).
"""
import argparse
import gc
import json
import os
import random
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from coda_b200 import CODA, TensorDataset  # noqa: E402
from coda_b200 import _native as nat  # noqa: E402
from coda_b200.engine import Engine  # noqa: E402
from coda_b200.synth import synth  # noqa: E402

CHUNK = 1 << 16          # items generated (fp32) and cast to fp16 at a time


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else q.stderr}


def half_slab(H, N, C, seed, dev):
    """fp16 slab of the synthetic task, built one item range at a time (the fp32 range is cast and dropped)."""
    p16 = torch.empty((H, N, C), dtype=torch.float16, device=dev)
    for lo in range(0, N, CHUNK):
        hi = min(N, lo + CHUNK)
        p, _ = synth(H, N, C, seed, device=dev, n_lo=lo, n_hi=hi)
        p16[:, lo:hi].copy_(p.half())
        del p
    _, labels = synth(H, N, C, seed, device=dev, want_preds=False)
    torch.cuda.synchronize()
    return p16, labels


def convert(src, dtype):
    """The other arm's slab from this one (exact both ways), one model at a time; `src` is released by the caller."""
    dst = torch.empty(src.shape, dtype=dtype, device=src.device)
    for h in range(src.shape[0]):
        dst[h].copy_(src[h])
    torch.cuda.synchronize()
    return dst


_orig_scan = Engine.construct_scan


def _profiled_scan(self):
    self.start_profile()          # bracket every construction launch with CUDA events (stopped in run_arm)
    _orig_scan(self)


def run_arm(slab, labels, steps, eager_steps):
    Engine.construct_scan = _profiled_scan
    try:
        random.seed(0)
        torch.cuda.synchronize()
        t0 = time.time()
        sel = CODA(TensorDataset(slab, labels), gpus=1)
        torch.cuda.synchronize()
        t_build = time.time() - t0
    finally:
        Engine.construct_scan = _orig_scan
    eng = sel.engine
    construction = {k: {"launches": n, "ms": round(ms, 3)} for k, (n, ms, _mx) in eng.stop_profile().items()}
    out = {"dtype": str(slab.dtype).split(".")[-1], "construct_s": round(t_build, 2), "construction_kernels": construction,
           "shadow_models": eng.n_shadow, "shadow_dtype": str(eng.shadow.dtype).split(".")[-1] if eng.shadow is not None
           else None, "mode": eng.mode,
           "mem_allocated_gb": round(torch.cuda.memory_allocated() / 1e9, 2)}
    free, total = torch.cuda.mem_get_info()
    out["device_mem_in_use_gb"] = round((total - free) / 1e9, 2)
    # rank-1 refresh: eager steps, events around that launch only
    r1 = eng._slab_fn("coda_b200_pi_rank1")
    eng.loop_prepare(labels)
    eng.start_profile(only={r1})
    for _ in range(eager_steps):
        eng.loop_eager()
    prof = eng.stop_profile()
    n, ms, _mx = prof[r1]
    out["pi_rank1_ms_per_step"] = round(ms / n, 4)
    # host-free loop: graph replays
    sel.run_steps(3, labels)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    sel.run_steps(steps, labels)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    out["steps"] = steps
    out["steps_per_s"] = round(steps / (ms / 1e3), 1)
    eng.check_flags(sync=True)
    idx, q, tie = sel.history()
    state = {"idx": torch.from_numpy(idx.copy()), "q": torch.from_numpy(q.copy()), "D": eng.D.cpu(),
             "U": eng.U.cpu(), "pi_hat": eng.pi_hat.cpu(), "pbest": sel.get_pbest().cpu()}
    sel.close()
    del sel, eng
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return out, state


def same(a, b):
    return all(torch.equal(a[k], b[k]) for k in a)


def capacity(H, N_list, C, seed, steps, dev):
    """The first N of `N_list` (tried in order) whose fp16 run fits one GPU: memory and steps/s."""
    tried = []
    for N in N_list:
        sel = p16 = labels = None
        try:
            p16, labels = half_slab(H, N, C, seed, dev)
            random.seed(0)
            sel = CODA(TensorDataset(p16, labels), gpus=1)
            free, total = torch.cuda.mem_get_info()
            rec = {"H": H, "N": N, "C": C, "slab_gb": round(p16.numel() * 2 / 1e9, 1), "mode": sel.engine.mode,
                   "shadow_models": sel.engine.n_shadow, "device_mem_in_use_gb": round((total - free) / 1e9, 2)}
            sel.run_steps(3, labels)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            sel.run_steps(steps, labels)
            e1.record()
            torch.cuda.synchronize()
            sel.engine.check_flags(sync=True)
            rec.update(steps=steps, steps_per_s=round(steps / (e0.elapsed_time(e1) / 1e3), 1), fits=True)
            tried.append(rec)
        except torch.OutOfMemoryError as e:
            tried.append({"H": H, "N": N, "C": C, "fits": False, "error": str(e).splitlines()[0][:200]})
        finally:
            if sel is not None:
                sel.close()
            sel = p16 = labels = None
            gc.collect()                  # a construction that ran out of memory leaves its buffers to the collector
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
        if tried[-1]["fits"]:
            break
    return tried


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--H", type=int, default=256)
    ap.add_argument("--N", type=int, default=1_000_000)
    ap.add_argument("--C", type=int, default=100)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--eager-steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--cap-N", type=int, nargs="*", default=[2_500_000, 2_000_000, 1_500_000])
    ap.add_argument("--cap-steps", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    nat.require_device()
    dev = torch.device("cuda:0")
    res = {"workload": f"synthetic H={args.H} N={args.N} C={args.C} seed={args.seed}", **gpu_info(), "arms": []}
    t0 = time.time()
    slab, labels = half_slab(args.H, args.N, args.C, args.seed, dev)
    res["generate_s"] = round(time.time() - t0, 1)
    first = {}
    for rep in range(args.reps):
        for kind in ("fp16", "fp32"):
            want = torch.float16 if kind == "fp16" else torch.float32
            if slab.dtype != want:
                other = convert(slab, want)
                del slab
                torch.cuda.empty_cache()
                slab = other
            out, state = run_arm(slab, labels, args.steps, args.eager_steps)
            out["rep"] = rep
            if "ref" not in first:
                first["ref"] = state
            out["final_state_equal_to_first_arm"] = same(state, first["ref"])
            res["arms"].append(out)
            print(json.dumps(out), flush=True)
    res["all_final_states_equal"] = all(a["final_state_equal_to_first_arm"] for a in res["arms"])
    del slab, labels, first
    torch.cuda.empty_cache()
    if args.cap_N:
        res["capacity"] = capacity(args.H, args.cap_N, args.C, args.seed, args.cap_steps, dev)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_fp16_slab.json"), "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
