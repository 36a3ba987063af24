"""Sampling without replacement (stochastic beam search) against the multinomial call it replaces, in one process on
one GPU.

The bench job: 1024 spectra x 128 candidates x 128 positions, bf16, bench weights (torch.manual_seed(0) model) and
inputs (make_spectra(1024, seed=1000)).  Two public calls alternate, three repetitions each after a warm-up, wall time
around a device synchronise (encode excluded):
  multinomial  multinomial_sequence_multi(..., n_candidates=128, per_memory_rng=True)
  sbs          sample_without_replacement(..., n_candidates=128)
Then one profiled call of each (mmt_profile_enable: per-kernel-class device time; for sbs the classes sbs_select,
beam_copy_pages and the decode step's kernels), and the mean number of distinct SMILES per spectrum of both calls on
the trained-like weights (tests/test_gpu_trained_weights.py) at temperature 1.0 and 0.7.  Prints the card name and
power limit with the results as JSON.
Usage: python profiles/sample_without_replacement_timing.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import multimodalspectraltransformer_b200 as M                      # noqa: E402
from multimodalspectraltransformer_b200 import synthetic             # noqa: E402
from multimodalspectraltransformer_b200.engine import engine_for     # noqa: E402

STOI = {"<PAD>": 0, "<UNK>": 1, "<EOS>": 2, "<SOS>": 3, "<MASK>": 4}
SBS_CLASSES = ("sbs_init", "sbs_select", "sbs_finish", "beam_copy_pages")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else None
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from test_gpu_candidate_streams import ITOS
    from test_gpu_trained_weights import trained_state_dict
    B, K, T = 1024, 128, 128
    cfg = M.default_config(device="cuda", precision="bf16", max_len=T)
    torch.manual_seed(0)
    model = M.MultimodalTransformer(cfg).eval()
    eng = engine_for(model, cfg)
    data = synthetic.make_spectra(B, seed=1000)
    memory, mask, *_ = M.run_model(model, data, cfg)
    calls = {
        "multinomial": lambda: M.multinomial_sequence_multi(model, memory, mask, STOI, cfg, n_candidates=K, per_memory_rng=True),
        "sbs": lambda: M.sample_without_replacement(model, STOI, memory, mask, cfg, n_candidates=K),
    }
    for fn in calls.values():          # warm-up: arena, graph capture
        fn()
    ms = {k: [] for k in calls}
    for _ in range(args.reps):
        for k, fn in calls.items():
            ms[k].append(round(timed(fn)[0], 2))
    prof = {}
    for k, fn in calls.items():
        eng.profile(True)
        fn()
        rep = eng.profile_report()
        eng.profile(False)
        total = sum(v["ms"] for v in rep.values())
        p = {"total_ms": round(total, 2)}
        if k == "sbs":
            for c in SBS_CLASSES:
                if c in rep:
                    p[c] = {"launches": rep[c]["launches"], "ms": round(rep[c]["ms"], 3)}
            p["decode_step_ms"] = round(sum(v["ms"] for c, v in rep.items() if c not in SBS_CLASSES), 2)
        p["classes"] = {c: {"launches": v["launches"], "ms": round(v["ms"], 3)} for c, v in sorted(rep.items(), key=lambda kv: -kv[1]["ms"])}
        prof[k] = p
    # distinct SMILES per spectrum, trained-like weights
    tm = M.MultimodalTransformer(cfg).eval()
    tm.load_state_dict({k: v.float() for k, v in trained_state_dict().items()})
    tmem, tmask, *_ = M.run_model(tm, data, cfg)
    distinct = {}
    for tau in (1.0, 0.7):
        cfg.temperature = tau
        row = {}
        for k, fn in (("multinomial", lambda: M.multinomial_sequence_multi(tm, tmem, tmask, STOI, cfg, n_candidates=K, per_memory_rng=True)[0]),
                      ("sbs", lambda: M.sample_without_replacement(tm, STOI, tmem, tmask, cfg, n_candidates=K)[0])):
            lists = M.distinct_smiles(fn(), ITOS, K)
            n = np.array([len(x) for x in lists])
            row[k] = {"mean": round(float(n.mean()), 2), "min": int(n.min()), "total": int(n.sum())}
        distinct[str(tau)] = row
    cfg.temperature = 1
    res = {"card": card(), "workload": f"{B} spectra x {K} candidates x {T} positions, bf16",
           "wall_ms": ms, "median_ms": {k: float(np.median(v)) for k, v in ms.items()},
           "profile": prof, "distinct_smiles_per_spectrum_trained_like": distinct}
    s = json.dumps(res, indent=1)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
