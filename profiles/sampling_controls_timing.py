"""Per-spectrum sampling controls against the plain decode, in one process on one GPU.

The bench job: 1024 spectra x 128 candidates x 128 positions, bf16, multinomial, one wave, bench weights
(torch.manual_seed(0) model) and inputs (make_spectra(1024, seed=1000), sampling seed 1234).  Four calls alternate, three
repetitions each, wall time around a device synchronise (encode excluded):
  plain    Engine.decode at temperature 1.0 (mmt_decode)
  neutral  mmt_decode_controlled with every column at 1.0, top-k and top-p off
  temps    mmt_decode_controlled with temperatures 0.7 / 1.0 / 1.3 by column
  topk_p   mmt_decode_controlled with top_k=20, top_p=0.95 in every column
Then one profiled call of plain and of topk_p (mmt_profile_enable: per-kernel-class device time, sample_tokens vs
sample_tokens_controlled).  Prints the card name and power limit with the results as JSON.
Usage: python profiles/sampling_controls_timing.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import multimodalspectraltransformer_b200 as M                      # noqa: E402
from multimodalspectraltransformer_b200 import synthetic             # noqa: E402
from multimodalspectraltransformer_b200.engine import engine_for     # noqa: E402
from multimodalspectraltransformer_b200.generate import _mask_to_bias  # noqa: E402


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
    B, K, T = 1024, 128, 128
    cfg = M.default_config(device="cuda", precision="bf16", max_len=T)
    torch.manual_seed(0)
    model = M.MultimodalTransformer(cfg).eval()
    eng = engine_for(model, cfg)
    memory, mask, *_ = M.run_model(model, synthetic.make_spectra(B, seed=1000), cfg)
    bias = _mask_to_bias(mask)
    kw = dict(n_cand=K, max_len=T, precision="bf16", seed=1234, offset=0)
    ones = np.ones(B, np.float32)
    calls = {
        "plain": lambda: eng.decode(memory, bias, temperature=1.0, sampling="multinomial", **kw),
        "neutral": lambda: eng.decode_controlled(memory, bias, temperature=ones, top_k=0, top_p=1.0, **kw),
        "temps": lambda: eng.decode_controlled(memory, bias, temperature=np.array([0.7, 1.0, 1.3], np.float32)[np.arange(B) % 3], **kw),
        "topk_p": lambda: eng.decode_controlled(memory, bias, temperature=1.0, top_k=20, top_p=0.95, **kw),
    }
    for fn in calls.values():          # warm-up: graph capture of each variant
        fn()
    ms = {k: [] for k in calls}
    outs = {}
    for _ in range(args.reps):
        for k, fn in calls.items():
            t, outs[k] = timed(fn)
            ms[k].append(round(t, 2))
    same_neutral = bool(torch.equal(outs["plain"][0], outs["neutral"][0]) and torch.equal(outs["plain"][1], outs["neutral"][1]))
    moved = float((outs["topk_p"][0] != outs["plain"][0]).any(0).float().mean())
    prof = {}
    for k in ("plain", "topk_p"):
        eng.profile(True)
        calls[k]()
        rep = eng.profile_report()
        eng.profile(False)
        prof[k] = {c: {"launches": v["launches"], "ms": round(v["ms"], 3)} for c, v in rep.items() if c.startswith("sample_tokens")}
        prof[k]["total_ms"] = round(sum(v["ms"] for v in rep.values()), 2)
    res = {"card": card(), "workload": f"{B} spectra x {K} candidates x {T} positions, bf16, multinomial, one wave",
           "wall_ms": ms, "median_ms": {k: float(np.median(v)) for k, v in ms.items()},
           "neutral_bit_identical_to_plain": same_neutral, "topk_p_sequences_differing_from_plain": round(moved, 4),
           "profile": prof}
    s = json.dumps(res, indent=1)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
