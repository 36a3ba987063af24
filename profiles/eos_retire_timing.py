"""Stop at <EOS> against the plain decode, in one process on one GPU.

  1. The bench job: 1024 spectra x 128 candidates x 128 positions, bf16, multinomial, bench weights
     (torch.manual_seed(0) model) and inputs (make_spectra(1024, seed=1000), sampling seed 1234).  Plain call and
     stop_at_eos alternate, three repetitions each, wall time around a device synchronise (encode excluded).
  2. The config-2 shape: 256 spectra greedy (one sequence each), fp32 and bf16, on the bench weights with
     fc_out.bias[<EOS>] raised (greedy sequences of the random init never end).

Prints the card name and power limit, the rows computed per position, the live fraction and the time ratio, as JSON.
Usage: python profiles/eos_retire_timing.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import multimodalspectraltransformer_b200 as M                      # noqa: E402
from multimodalspectraltransformer_b200 import synthetic             # noqa: E402
from multimodalspectraltransformer_b200.engine import engine_for     # noqa: E402
from multimodalspectraltransformer_b200.generate import _mask_to_bias  # noqa: E402

STOI = {"<PAD>": 0, "<UNK>": 1, "<EOS>": 2, "<SOS>": 3, "<MASK>": 4}
EOS = 2


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
    return time.perf_counter() - t0, out


def first_eos(tok):
    hit = tok == EOS
    return torch.where(hit.any(0), hit.int().argmax(0), torch.full_like(hit[0], tok.shape[0], dtype=torch.long))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"card": card()}

    # ---- 1. bench job
    cfg = M.default_config(device="cuda", precision="bf16")
    torch.manual_seed(0)
    model = M.MultimodalTransformer(cfg).eval()
    data = {k: v.cuda() for k, v in synthetic.make_spectra(1024, seed=1000).items()}
    memory, mask, *_ = M.run_model(model, data, cfg)
    gen = torch.cuda.default_generators[torch.cuda.current_device()]

    def job(stop):
        torch.manual_seed(1234)
        return M.multinomial_sequence_multi(model, memory, mask, STOI, cfg, n_candidates=128, stop_at_eos=stop)

    job(False); job(True)                                           # warm-up: graphs, arena
    t_plain, t_eos = [], []
    for _ in range(3):
        dt, (ta, pa) = timed(lambda: job(False)); t_plain.append(dt)
        dt, (tb, pb) = timed(lambda: job(True)); t_eos.append(dt)
    L = first_eos(ta)
    keep = torch.arange(128, device=ta.device)[:, None] <= L[None]
    same = bool(torch.equal(ta[keep], tb[keep]) and torch.equal(pa[keep], pb[keep]) and bool((tb[~keep] == 0).all()))
    eng = engine_for(model, cfg)
    torch.manual_seed(1234)
    seed, off = int(gen.initial_seed()), int(gen.get_offset())
    _, _, steps, lens, rows = eng.decode_until_eos(memory, _mask_to_bias(mask), eos=EOS, n_cand=128, max_len=128,
                                                   sampling="multinomial", precision="bf16", seed=seed, offset=off)
    N, T = 1024 * 128, 128
    live = (torch.arange(T, device=lens.device)[:, None] <= lens.long()[None]).sum(1).cpu()
    res["bench_job"] = {
        "shape": "1024 spectra x 128 candidates x 128 positions, bf16, multinomial",
        "plain_s": t_plain, "stop_at_eos_s": t_eos,
        "time_ratio_median": sorted(t_eos)[1] / sorted(t_plain)[1],
        "outputs_equal_up_to_eos": same,
        "rows_per_position": rows.tolist(), "live_per_position": live.tolist(),
        "rows_fraction": int(rows.sum()) / (N * T), "live_fraction": int(live.sum()) / (N * T),
        "never_eos": int((lens == T).sum()), "length_quartiles": torch.quantile(lens.float().cpu(), torch.tensor([.25, .5, .75])).tolist(),
        "steps": steps,
    }
    del ta, pa, tb, pb
    engine_for(model, cfg)       # keep the engine; free the rest before the next shape
    torch.cuda.empty_cache()

    # ---- 2. config-2 shape, greedy on raised <EOS> weights
    torch.manual_seed(0)
    raised = M.MultimodalTransformer(M.default_config(device="cuda")).eval()
    with torch.no_grad():
        raised.fc_out.bias[EOS] += 0.5       # spreads greedy lengths on these weights (+1.0 ends all at position 0)
    data2 = {k: v.cuda() for k, v in synthetic.make_spectra(256, seed=2000).items()}
    res["config2_greedy"] = {}
    for prec in ("fp32", "bf16"):
        cfg2 = M.default_config(device="cuda", precision=prec)
        mem2, mask2, *_ = M.run_model(raised, data2, cfg2)
        run = lambda stop: M.greedy_sequence(raised, STOI, None, mem2, mask2, cfg2, stop_at_eos=stop)
        run(False); run(True)
        tp, te = [], []
        for _ in range(3):
            dt, (a, _) = timed(lambda: run(False)); tp.append(dt)
            dt, (b, _) = timed(lambda: run(True)); te.append(dt)
        e2 = engine_for(raised, cfg2)
        _, _, steps2, lens2, rows2 = e2.decode_until_eos(mem2, _mask_to_bias(mask2), eos=EOS, n_cand=1, max_len=128,
                                                         sampling="greedy", stop_on_all_pad=True, precision=prec)
        res["config2_greedy"][prec] = {
            "plain_s": tp, "stop_at_eos_s": te, "time_ratio_median": sorted(te)[1] / sorted(tp)[1],
            "plain_steps": int(a.shape[0]), "stop_at_eos_steps": int(b.shape[0]),
            "never_eos": int((lens2 == 128).sum()), "max_len_of_finished": int(lens2[lens2 < 128].max()) if bool((lens2 < 128).any()) else None,
            "rows_per_position": rows2.tolist(),
        }
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
