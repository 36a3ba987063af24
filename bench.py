#!/usr/bin/env python
"""bench.py -- generated SMILES tokens/s of the MMT candidate-generation path.

    python bench.py --gpus N --steps K --warmup W                     # this framework
    python bench.py --impl reference --gpus N --steps K --warmup W    # CPU reference arm (oracle port)
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR  # also write the last timed step's ids to DIR

Workload (BASELINE.json configs[2], the configuration the metric "tokens/s at 1/2/4/8 B200" is quoted on and the
reference's production call, mmt_result_test_functions_15_4.py:504-570): config_V8 random-init weights, MULTINOMIAL
sampling of 128 candidates for each of 1024 synthetic 1H+13C+HSQC+COSY+IR(+MF+MW) spectra, 128 tokens each
= 131,072 sequences, 16,777,216 generated tokens per step.  STRONG scaling: the 1024 spectra are sharded over the N
ranks by ``scheduler.generate_sharded`` (contiguous blocks, shard-invariant Philox draws), every rank encodes its
spectra once, decodes its candidates in waves of up to 151,552 sequences (one wave per rank here) and the ids are all-gathered over NCCL as bytes on a
side stream (overlapping the next step).  One "step" = encode + every wave + gather for all 1024 spectra.

Extra keys of the JSON line: ``config2`` (BASELINE.json configs[1]: greedy, 256 spectra per GPU x 128 tokens, weak
scaling, resident and end to end), ``roofline`` (dominant kernel of the main workload), ``cpu_baseline`` and
``gpu_eager_baseline`` (the oracle port of the reference's full-prefix loop on the host cores / on this B200 under torch
eager, bounded samples), see DESIGN.md section 5.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "generated SMILES tokens/sec"
UNIT = "tokens/s"
N_SPECTRA = 1024                # config 3: spectra in the whole job
N_CAND = 128                    # candidates per spectrum
MAX_LEN = 128
C2_SPECTRA_PER_GPU = 256        # config 2 (extra key): greedy, weak scaling
REF_SAMPLE_CAND = 16            # CPU arms: candidates of ONE spectrum per step (the reference decodes one spectrum at a time)
EAGER_SAMPLE_SPECTRA = 8        # gpu_eager_baseline: spectra x 128 candidates under torch eager
DUMP_SEQUENCES = 65536          # --dump-outputs: 65,536 x 128 ids in float32 = 32 MiB (all 131,072 would be 64 MiB)
STOI = {"<PAD>": 0, "<UNK>": 1, "<EOS>": 2, "<SOS>": 3, "<MASK>": 4}
# algorithmic work model (SURVEY.md 8d / BASELINE.md 4)
FLOP_ENCODE_PER_SPECTRUM = 9.50e9
FLOP_CROSSKV_PER_SPECTRUM = 228.9e6
FLOP_DECODE_PER_TOKEN = 9.468e6


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm=j["hbm_gbs"], tf=j["bf16_tflops"], tf_sustained=j.get("bf16_tflops_sustained", j["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tf=1590.0, tf_sustained=1400.0, src="fallback")


def source_hash():
    """sha256 over the CUDA sources: ties an ncu traffic figure under profiles/ to the build it was captured from."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "multimodalspectraltransformer_b200", "csrc")
    for f in sorted(os.listdir(d)):
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def dump_outputs(out_dir, ids):
    """Write DIR/ids.npy: the rows of the (sequences, positions) u8 ids a caller of the timed path receives, at a fixed
    seeded sample of DUMP_SEQUENCES sequences in ascending order, as float32 (exact for ids < 2**24)."""
    import numpy as np
    import torch
    n = ids.shape[0]
    rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:min(n, DUMP_SEQUENCES)].sort().values
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "ids.npy"), ids[rows.to(ids.device)].cpu().numpy().astype(np.float32))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------- the reference's algorithm
def reference_flow(P, O, data_one, n_cand, cfg, device="cpu", generator=None):
    """What the reference does for ONE spectrum (mmt_result_test_functions_15_4.py:519-535): duplicate_dict(x, n) ->
    run_model on the n identical copies -> multinomial_sequence_multi (full prefix re-run every step, memory
    re-projected every step).  Oracle port (oracle/mmt_oracle.py), torch ops on `device`."""
    import torch
    dup = {k: v.repeat(*([n_cand] + [1] * (v.dim() - 1))).to(device) for k, v in data_one.items()}
    with torch.no_grad():
        mem, mask, _, _ = O.encode(P, dup, cfg)
        tok, _ = O.multinomial_sequence_multi(P, mem, mask, cfg, generator=generator)
    return tok


def cpu_reference_tokens_per_s(steps=1, warmup=0, threads=None):
    import torch
    from oracle import mmt_oracle as O
    from multimodalspectraltransformer_b200 import synthetic
    if threads:
        torch.set_num_threads(threads)
    cfg = O.default_config()
    P = O.random_init_state_dict(cfg, seed=0)
    times, tok = [], None
    for i in range(warmup + steps):
        data = synthetic.make_spectra(1, seed=1000 + i)
        t0 = time.perf_counter()
        tok = reference_flow(P, O, data, REF_SAMPLE_CAND, cfg)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    tokens = tok.numel()
    sec = sum(times) / len(times)
    return tokens / sec, tokens, sec, torch.get_num_threads()


REF_SAMPLE_TEXT = (f"1 of the {N_SPECTRA} spectra x {REF_SAMPLE_CAND} of its {N_CAND} candidates x {MAX_LEN} tokens per step, the reference's own "
                   "per-spectrum flow (duplicate -> encode the copies -> multinomial loop with full-prefix recompute), fp32, oracle port")


def workload_config(n_gpus, precision, ref_sample=False):
    c = {"workload": f"MMT config_V8 random-init, multinomial sampling, {N_SPECTRA} synthetic spectra x {N_CAND} candidates x {MAX_LEN} tokens "
                     "(BASELINE.json configs[2]; encode + KV-cached decode in waves of up to 151,552 sequences (one wave per rank) + NCCL all-gather of the ids per step)",
         "spectra_total": N_SPECTRA, "candidates": N_CAND, "max_len": MAX_LEN, "sequences_total": N_SPECTRA * N_CAND,
         "spectra_per_gpu": (N_SPECTRA + n_gpus - 1) // n_gpus, "peaks": "realistic", "precision": precision,
         "parallelism": f"dp{n_gpus}",
         "l2": "no explicit flush: one step streams > 50 GB of self-attention KV pages (393 KB of pool per sequence) through the 126 MB L2"}
    if ref_sample:
        c["measured_sample"] = REF_SAMPLE_TEXT
    return c


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    try:
        ncores = len(os.sched_getaffinity(0))        # torchrun exports OMP_NUM_THREADS=1 for its workers: use every core we may
    except AttributeError:
        ncores = os.cpu_count() or 1
    precision = args.precision if args.precision != "auto" else os.environ.get("MMT_DEFAULT_PRECISION", "bf16")
    v, tokens, sec, threads = cpu_reference_tokens_per_s(steps=max(1, args.steps), warmup=min(args.warmup, 1), threads=ncores)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(max(1, args.gpus), precision, ref_sample=True),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": REF_SAMPLE_TEXT},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=os.environ.get("MMT_BENCH_PRECISION", "auto"), choices=["auto", "fp32", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the cpu / gpu-eager comparator legs")
    ap.add_argument("--no-config2", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the ids of the last timed step of the main workload to DIR/ids.npy (float32, a fixed sample "
                         f"of {DUMP_SEQUENCES:,} of the {N_SPECTRA * N_CAND:,} sequences), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs needs --impl b200")
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import multimodalspectraltransformer_b200 as M
    from multimodalspectraltransformer_b200 import synthetic, scheduler
    from multimodalspectraltransformer_b200.engine import engine_for

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = max(3, args.warmup)
    K = args.steps

    precision = args.precision
    if precision == "auto":
        precision = os.environ.get("MMT_DEFAULT_PRECISION", "bf16")
    cfg = M.default_config(device=str(dev), precision=precision, max_len=MAX_LEN)
    torch.manual_seed(0)
    model = M.MultimodalTransformer(cfg).eval()
    eng = engine_for(model, cfg)
    torch.manual_seed(1234)                                             # the sampling stream (same on every rank: shard-invariant draws)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def timed_pipeline(issue, consume, k, flush=None):
        """k steps; step i's gathered ids are consumed after step i+1 has been issued, so the collective (side stream) and
        the rendezvous with the slowest rank overlap the next step.  Device time from CUDA events on the launching stream,
        barrier + synchronize on both sides, max over ranks.  With `flush` (an L2 flush between steps) every step has its
        own event pair and the flushes fall between the pairs.  Returns (device ms, wall s, what the last step's issue()
        returned)."""
        barrier()
        t0 = time.perf_counter()
        evs = []
        prev = None
        if flush is None:
            evs.append((torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)))
            evs[0][0].record()
        for _ in range(k):
            if flush is not None:
                flush()
                evs.append((torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)))
                evs[-1][0].record()
            cur = issue()
            if prev is not None:
                consume(prev)
            prev = cur
            if flush is not None:
                evs[-1][1].record()
        if flush is not None:
            evs.append((torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)))
            evs[-1][0].record()
        consume(prev)
        evs[-1][1].record()
        barrier()
        wall = time.perf_counter() - t0
        return max_over_ranks(sum(a.elapsed_time(b) for a, b in evs)), wall, prev

    COPIED = ("src_1H", "mask_1H", "src_13C", "mask_13C", "src_HSQC", "src_HSQC", "mask_HSQC", "src_COSY", "src_COSY", "mask_COSY",
              "src_IR", "src_MF", "mask_MF", "trg_MW", "trg_enc_SMI")      # what run_model moves to the device (HSQC / COSY twice: it also returns them)

    def h2d_bytes(d):
        return sum(d[k].numel() * d[k].element_size() for k in COPIED)

    # ------------------------------------------------------------------ main workload: config 3, strong scaling
    host = synthetic.make_spectra(N_SPECTRA, seed=1000)
    pinned = {k: v.pin_memory() for k, v in host.items()}
    resident = {k: v.to(dev) for k, v in host.items()}
    out_host = torch.empty(N_SPECTRA * N_CAND, MAX_LEN, dtype=torch.uint8).pin_memory()
    lo, hi = scheduler.shard_bounds(N_SPECTRA, world, rank)

    def issue_resident():
        return scheduler.generate_sharded(model, resident, cfg, STOI, n_candidates=N_CAND, sampling="multinomial", async_gather=True)

    def issue_e2e():        # host buffers in: generate_sharded slices this rank's spectra, run_model copies them to the device
        return scheduler.generate_sharded(model, pinned, cfg, STOI, n_candidates=N_CAND, sampling="multinomial", async_gather=True)

    def consume_resident(p):
        p.packed()

    def consume_e2e(p):     # device -> host read of the step's result (the gathered ids, bytes)
        out_host.copy_(p.packed(), non_blocking=True)

    for _ in range(W):
        consume_resident(issue_resident())
    consume_e2e(issue_e2e())
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = eng.launch_count()
    ms_res, wall_res, last = timed_pipeline(issue_resident, consume_resident, K)
    launches = eng.launch_count() - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last.packed())
    del last
    ms_e2e, wall_e2e, _ = timed_pipeline(issue_e2e, consume_e2e, K)
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([launches], device=dev, dtype=torch.int64)
        dist.all_reduce(t)
        launches = int(t.item())
    tokens_per_step = MAX_LEN * N_SPECTRA * N_CAND
    value = tokens_per_step * K / (ms_res / 1e3)
    e2e_value = tokens_per_step * K / (ms_e2e / 1e3)
    h2d = h2d_bytes(pinned)
    d2h = out_host.numel() * out_host.element_size() * world

    # ------------------------------------------------------------------ config 2 (extra key): greedy, 256 spectra per GPU, weak scaling
    c2 = None
    if not args.no_config2:
        K2 = min(K, 10)
        host2 = synthetic.make_spectra(C2_SPECTRA_PER_GPU * world, seed=2000)
        pinned2 = {k: v.pin_memory() for k, v in host2.items()}
        resident2 = {k: v.to(dev) for k, v in host2.items()}
        out2 = torch.empty(C2_SPECTRA_PER_GPU * world, MAX_LEN, dtype=torch.uint8).pin_memory()
        flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        g_res = lambda: scheduler.generate_sharded(model, resident2, cfg, STOI, n_candidates=1, sampling="greedy", async_gather=True)
        g_e2e = lambda: scheduler.generate_sharded(model, pinned2, cfg, STOI, n_candidates=1, sampling="greedy", async_gather=True)
        for _ in range(W):
            g_res().packed()
        g_e2e().packed()
        l0 = eng.launch_count()
        ms2, _, _ = timed_pipeline(g_res, lambda p: p.packed(), K2, flush=lambda: flush_buf.fill_(1))
        launches2 = eng.launch_count() - l0
        ms2e, _, _ = timed_pipeline(g_e2e, lambda p: out2.copy_(p.packed(), non_blocking=True), K2, flush=lambda: flush_buf.fill_(1))
        tok2 = MAX_LEN * C2_SPECTRA_PER_GPU * world
        c2 = {"workload": f"BASELINE.json configs[1]: greedy decode, {C2_SPECTRA_PER_GPU} spectra per GPU x {MAX_LEN} tokens, weak scaling, "
                          "explicit 256 MiB L2 flush between steps (untimed)",
              "value": tok2 * K2 / (ms2 / 1e3), "unit": UNIT, "ms_per_step": ms2 / K2, "steps": K2, "scaling": "weak",
              "e2e": {"value": tok2 * K2 / (ms2e / 1e3), "unit": UNIT, "ms_per_step": ms2e / K2,
                      "h2d_bytes_per_step": h2d_bytes(pinned2),
                      "d2h_bytes_per_step": out2.numel() * world},
              "gpu_launches_per_rank": launches2,
              "frac_bf16_tensor_peak": tok2 * K2 / (ms2 / 1e3) / world
              * (FLOP_DECODE_PER_TOKEN + (FLOP_ENCODE_PER_SPECTRUM + FLOP_CROSSKV_PER_SPECTRUM) / MAX_LEN) / (peaks()["tf"] * 1e12)}
        del flush_buf

    # ------------------------------------------------------------------ config 5 (extra key): max peak counts, greedy, 512 spectra per GPU
    c5 = None
    if not args.no_config2:
        K5 = min(K, 5)
        res5 = {k: v.to(dev) for k, v in synthetic.make_spectra(512, seed=5000 + rank, peaks="max").items()}
        def step5():
            memory, mask, *_ = M.run_model(model, res5, cfg)
            tok, _ = M.greedy_sequence(model, STOI, None, memory, mask, cfg)
            return tok
        for _ in range(2):
            step5()
        barrier()
        a5, b5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a5.record()
        for _ in range(K5):
            step5()
        b5.record()
        barrier()
        ms5 = max_over_ranks(a5.elapsed_time(b5))
        c5 = {"workload": "BASELINE.json configs[4] per-GPU share: 512 spectra with every peak slot valid (582 attended memory rows each), greedy, "
                          f"{MAX_LEN} tokens, encode + decode per step, inputs resident, weak scaling",
              "value": 512 * MAX_LEN * world * K5 / (ms5 / 1e3), "unit": UNIT, "ms_per_step": ms5 / K5, "steps": K5, "scaling": "weak",
              "hbm_floor_note": "cross K/V of 512 x 582 rows x 6 layers in bf16 = 915 MB per position: 140 us per position at the measured HBM peak"}
        del res5

    # ------------------------------------------------------------------ roofline of the dominant kernel (rank 0's GPU)
    pk = peaks()
    roof = None
    if rank == 0:
        wave = min(1184, hi - lo)            # one wave as the timed loop runs it on this rank (148 SMs x 8 rounds of 128-row tiles at most)
        data_w = {k: v[:wave] for k, v in resident.items()}
        eng.profile(True)
        memory, mask, *_ = M.run_model(model, data_w, cfg)
        M.multinomial_sequence_multi(model, memory, mask, STOI, cfg, n_candidates=N_CAND)
        prof = eng.profile_report()
        eng.profile(False)
        total_ms = sum(v["ms"] for v in prof.values())
        dom = max(prof, key=lambda k: prof[k]["ms"])
        esz = 4 if precision == "fp32" else 2
        Nw = wave * N_CAND
        n_valid = int((~mask.bool()).sum().item()) if mask.dtype == torch.bool else mask.numel()
        kv_self = Nw * ((MAX_LEN + 1) / 2) * 2 * 128 * esz                # mean over positions of the cache read (t + 1 rows of K and V)
        kv_cross = n_valid * 2 * 128 * esz + n_valid * 4                  # shared by the 128 candidates of a spectrum
        alg_bytes = {
            # per launch = one decoder layer, one position, one wave: DESIGN.md section 5
            # cache pages read + the dense fp32 query rows in + bf16 attention rows out (bf16 mode: K | V of the new position are
            # appended by the QKV projection's epilogue, not here; fp32 check mode reads the whole qkv row and appends)
            "decode_self_attention": kv_self + (Nw * 128 * 4 + Nw * 128 * 2 if precision != "fp32" else Nw * 2 * 128 * esz + Nw * 3 * 128 * 4 + Nw * 128 * 4),
            "decode_layer": kv_self + Nw * 2 * 128 * esz + kv_cross + Nw * 128 * (4 + 4 + 2),
            "decode_cross_attention": kv_cross + Nw * 128 * 4 + Nw * 128 * 2,
            "decode_attn": kv_cross + kv_self + Nw * 128 * (4 + 4 + 2),
        }
        d = prof[dom]
        per_launch_ms = d["ms"] / d["launches"]
        if d.get("flops", 0) > 0:
            achieved = d["flops"] / d["launches"] / (per_launch_ms * 1e-3) / 1e12
            roof = {"kernel": dom, "bound": "tensor", "achieved": achieved, "peak": pk["tf"], "unit": "TFLOP/s", "frac": achieved / pk["tf"],
                    "traffic": None, "peak_source": pk["src"] + " bf16 burst"}
        elif alg_bytes.get(dom):
            achieved = alg_bytes[dom] / (per_launch_ms * 1e-3) / 1e9
            roof = {"kernel": dom, "bound": "hbm", "achieved": achieved, "peak": pk["hbm"], "unit": "GB/s", "frac": achieved / pk["hbm"],
                    "traffic": None, "peak_source": pk["src"], "algorithmic_bytes_per_launch": alg_bytes[dom]}
        else:
            roof = {"kernel": dom, "bound": "hbm", "achieved": None, "peak": pk["hbm"], "unit": "GB/s", "frac": None, "traffic": None}
        roof["profile_mode"] = (f"one wave ({wave} spectra x {N_CAND} candidates = {Nw} sequences x {MAX_LEN} positions) + its encode, eager launches "
                                "bracketed by CUDA events on the launching stream (the timed loop replays the same kernels as CUDA graphs)")
        try:     # DRAM bytes per launch from an ncu --set full capture -- only if it was taken from THIS build of the kernels
            tj = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")))
            if tj.get("source_hash") == source_hash() and dom in tj.get("kernels", {}):
                kj = tj["kernels"][dom]
                roof["traffic"] = kj["dram_bytes_read"] + kj["dram_bytes_write"]
                roof["traffic_source"] = f"profiles/r02_ncu_traffic.json ({kj.get('note', 'ncu --set full')}; same source hash as this build)"
                if kj.get("algorithmic_bytes_of_captured_launch"):     # the capture is ONE position; `achieved` averages all of them
                    roof["traffic_capture"] = kj.get("capture")
                    roof["traffic_algorithmic_bytes"] = kj["algorithmic_bytes_of_captured_launch"]
                    roof["traffic_over_algorithmic"] = roof["traffic"] / kj["algorithmic_bytes_of_captured_launch"]
            else:
                roof["traffic_source"] = "none: profiles/r02_ncu_traffic.json was captured from another build (source hash differs)"
        except (OSError, ValueError, KeyError):
            pass
        roof["share_of_step"] = d["ms"] / total_ms if total_ms else None
        roof["launch_us"] = per_launch_ms * 1e3
        roof["kernels"] = {k: {"launches": v["launches"], "ms": round(v["ms"], 3)} for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}

    if rank == 0:
        flop_per_token = FLOP_DECODE_PER_TOKEN + (FLOP_ENCODE_PER_SPECTRUM + FLOP_CROSSKV_PER_SPECTRUM) / (N_CAND * MAX_LEN)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_res / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32" if precision == "fp32" else "bf16", "data": "synthetic", "config": workload_config(world, precision),
                "frac_bf16_tensor_peak": value / world * flop_per_token / (pk["tf"] * 1e12),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / K},
                "gpu_launches": launches, "clocks": clocks, "roofline": roof, "wall_s": {"resident": wall_res, "e2e": wall_e2e}}
        if c2 is not None:
            line["config2"] = c2
        if c5 is not None:
            line["config5"] = c5
        if world == 1 and not args.no_cpu_baseline:
            try:     # the reference's algorithm under torch eager on this same B200 (library kernels): how much is the GPU, how much the engine
                from oracle import mmt_oracle as O
                ocfg = O.default_config()
                Pd = {k: v.to(dev) for k, v in O.random_init_state_dict(ocfg, seed=0).items()}
                d8 = synthetic.make_spectra(EAGER_SAMPLE_SPECTRA, seed=1000)
                dup = {k: v.repeat_interleave(N_CAND, dim=0).to(dev) for k, v in d8.items()}
                with torch.no_grad():
                    O.encode(Pd, {k: v[:N_CAND] for k, v in dup.items()}, ocfg)             # warm-up (cuBLAS handles, kernels)
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    mem, msk, _, _ = O.encode(Pd, dup, ocfg)
                    tok_e, _ = O.multinomial_sequence_multi(Pd, mem, msk, ocfg)
                    torch.cuda.synchronize()
                    sec = time.perf_counter() - t0
                v_eager = tok_e.numel() / sec
                line["gpu_eager_baseline"] = {
                    "value": v_eager, "unit": UNIT, "kind": "port", "seconds": sec,
                    "sample": f"{EAGER_SAMPLE_SPECTRA} of the {N_SPECTRA} spectra x {N_CAND} candidates x {MAX_LEN} tokens in ONE batch of {EAGER_SAMPLE_SPECTRA * N_CAND} sequences "
                              "(8x the reference's own batch), fp32, oracle port of the reference's loop (encode the duplicated copies, full-prefix "
                              "decoder re-run and memory re-projection every step) as torch 2.11 eager ops on this B200",
                    "engine_over_eager": value / v_eager}
                del Pd, dup, mem, msk
            except Exception as exc:      # never let a comparator cost the bench line
                line["gpu_eager_baseline"] = {"error": str(exc)[:200]}
            CPU_STEPS = 5       # ~10-15 s of host work: 5 spectra after one untimed warm-up spectrum
            v, toks, sec, threads = cpu_reference_tokens_per_s(steps=CPU_STEPS, warmup=1)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": REF_SAMPLE_TEXT + f" ({CPU_STEPS} such steps timed: {toks} tokens and {sec:.1f} s each)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
