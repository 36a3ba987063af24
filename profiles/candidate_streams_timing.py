"""Candidate generation in both RNG modes, and distinct SMILES against the host post-processing.

    python profiles/candidate_streams_timing.py [--reps 3] [--out candidate_streams.json]

1. The 1024 spectra x 128 candidates x 128 positions multinomial call (bf16, the bench geometry) with the global mapping
   and with per_memory_rng=True, alternated in one process, each timed with a device synchronise around the call.
2. distinct_smiles against tensor_to_smiles_and_prob_2 on the same 131,072 candidates (the real output of the call),
   the host path timed on CUDA tensors as a caller hands them over.

The card's name and power limit are recorded beside the numbers.  Needs a GPU; there is no CPU path.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

STOI = {"<PAD>": 0, "<UNK>": 1, "<EOS>": 2, "<SOS>": 3, "<MASK>": 4}
ITOS = {str(i): c for i, c in enumerate(["<PAD>", "<UNK>", "<EOS>", "<SOS>", "<MASK>", "C", "c", "O", "N", "(", ")", "=",
                                          "1", "2", "3", "[", "]", "Cl", "l", "Br", "r", "F", "S", "#", "@", "H", "+", "-",
                                          "n", "o", "s", "/", "\\", "4", "5", "6", "P", "I", "B", "%", "Si", "Se", "."])}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import multimodalspectraltransformer_b200 as M
    from multimodalspectraltransformer_b200 import synthetic
    B, K = 1024, 128
    cfg = M.default_config(device="cuda", precision="bf16", max_len=128)
    torch.manual_seed(0)
    model = M.MultimodalTransformer(cfg).eval()
    memory, mask, *_ = M.run_model(model, synthetic.make_spectra(B, seed=3003), cfg)

    def call(per_memory):
        return M.multinomial_sequence_multi_2(model, memory, mask, STOI, cfg, n_candidates=K, per_memory_rng=per_memory)

    for pm in (False, True):      # warm-up: graph capture of both modes
        call(pm)
    times = {"global": [], "per_memory": []}
    for _ in range(args.reps):
        for pm in (False, True):
            torch.manual_seed(1)
            dt, res = timed(lambda: call(pm))
            times["per_memory" if pm else "global"].append(dt)
    tok, pr = res
    d_times, h_times = [], []
    M.distinct_smiles(tok, ITOS, K, token_prob=pr)        # warm-up: itos upload
    for _ in range(args.reps):
        dt, got = timed(lambda: M.distinct_smiles(tok, ITOS, K, token_prob=pr))
        d_times.append(dt)
        dt, _ = timed(lambda: M.tensor_to_smiles_and_prob_2(tok, pr, ITOS))
        h_times.append(dt)
    n_dist = sum(len(c) for c in got)
    out = dict(card=card(), geometry=f"{B} x {K} x 128, bf16", call_s=times,
               distinct_smiles_s=d_times, tensor_to_smiles_and_prob_2_s=h_times,
               candidates=B * K, distinct=n_dist)
    print(json.dumps(out, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
