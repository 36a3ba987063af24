"""A/B of two builds of libmmt_b200.so on the decode drivers: the same seeded calls, outputs compared bit for bit.

Every decode path (greedy stop_on_all_pad in one and in several waves, multinomial plain and with per-memory streams,
stop at <EOS> in a small fused and a large compacting wave, sampling controls with and without <EOS>, teacher forcing,
beam search, sampling without replacement twice) runs under the default engine and under each driver switch
(MMT_NO_GRAPH, MMT_NO_GRAPH_CACHE, MMT_GRAPH_STEPS=3, MMT_DECODE_LANES=4, MMT_DECODE_LANES_LARGE=2).  Per call it
records the outputs, h_steps, h_rows and the launch-counter delta; a separate profiled pass records the launches per
kernel name from mmt_profile_report.  Each build runs in its own process (MMT_B200_LIB selects the library).

    python profiles/decode_driver_ab.py --lib-a OLD.so [--lib-b NEW.so] --out profiles/r03_decode_driver_ab.json

--lib-b defaults to the package's in-tree build.  Exit status 1 when anything differs.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENVS = {"default": {}, "no_graph": {"MMT_NO_GRAPH": "1"}, "no_graph_cache": {"MMT_NO_GRAPH_CACHE": "1"},
        "graph_steps_3": {"MMT_GRAPH_STEPS": "3"}, "decode_lanes_4": {"MMT_DECODE_LANES": "4"},
        "decode_lanes_large_2": {"MMT_DECODE_LANES_LARGE": "2"}}
MULTI_WAVE = {"MMT_MAX_WAVE_SEQS": "64"}     # 16 spectra x 16 candidates -> four waves
EOS, PAD = 2, 0


def worker(out_path):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import multimodalspectraltransformer_b200 as M
    from multimodalspectraltransformer_b200 import synthetic
    from multimodalspectraltransformer_b200.engine import Engine
    from multimodalspectraltransformer_b200.generate import _mask_to_bias

    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    cfg0 = M.default_config(device="cuda")
    base = M.MultimodalTransformer(cfg0).eval()

    def raised(tok, delta):      # the same weights with fc_out.bias[tok] raised: greedy sequences end / pad
        sd = {k: v.detach().clone() for k, v in base.state_dict().items()}
        sd["fc_out.bias"][tok] += delta
        return sd

    models = {"base": base.state_dict(), "pad1": raised(PAD, 1.0), "pad3": raised(PAD, 3.0), "eos1": raised(EOS, 1.0)}
    mem = {}

    def inputs(B, prec, seed):
        if (B, prec, seed) not in mem:
            cfg = M.default_config(device="cuda", precision=prec)
            memory, mask, *_ = M.run_model(base, synthetic.make_spectra(B, seed=seed), cfg)
            mem[(B, prec, seed)] = (memory, _mask_to_bias(mask))
        return mem[(B, prec, seed)]

    def cols(B, lo, hi, seed):
        return np.random.default_rng(seed).uniform(lo, hi, B).astype(np.float32)

    rng = dict(seed=1234, offset=4 * 17)
    # name -> (model, multi-wave engine, call(engine) -> tuple of outputs, h_steps, h_rows or None)
    cases = {}

    def case(name, model="base", multi=False):
        def deco(fn):
            cases[name] = (model, multi, fn)
            return fn
        return deco

    for prec in ("fp32", "bf16"):
        for m in ("base", "pad1", "pad3"):
            @case(f"greedy_pad_1wave_{prec}_{m}", m)
            def _(e, prec=prec):
                memory, bias = inputs(16, prec, 21)
                t, p, s = e.decode(memory, bias, n_cand=4, max_len=128, sampling="greedy", stop_on_all_pad=True, precision=prec)
                return (t, p), s, None

            @case(f"greedy_pad_waves_{prec}_{m}", m, multi=True)
            def _(e, prec=prec):
                memory, bias = inputs(16, prec, 21)
                t, p, s = e.decode(memory, bias, n_cand=16, max_len=128, sampling="greedy", stop_on_all_pad=True, precision=prec)
                return (t, p), s, None

        @case(f"until_eos_small_{prec}")
        def _(e, prec=prec):
            memory, bias = inputs(24, prec, 11)
            t, p, s, L, rows = e.decode_until_eos(memory, bias, eos=EOS, n_cand=16, max_len=128, sampling="multinomial",
                                                  precision=prec, **rng)
            return (t, p, L), s, rows

        @case(f"until_eos_large_{prec}")
        def _(e, prec=prec):
            memory, bias = inputs(300, prec, 13)
            t, p, s, L, rows = e.decode_until_eos(memory, bias, eos=EOS, n_cand=16, max_len=128, sampling="multinomial",
                                                  precision=prec, **rng)
            return (t, p, L), s, rows

        @case(f"until_eos_greedy_pad_{prec}", "eos1")
        def _(e, prec=prec):
            memory, bias = inputs(24, prec, 12)
            t, p, s, L, rows = e.decode_until_eos(memory, bias, eos=EOS, n_cand=4, max_len=128, sampling="greedy",
                                                  stop_on_all_pad=True, precision=prec)
            return (t, p, L), s, rows

        @case(f"until_eos_waves_{prec}", multi=True)
        def _(e, prec=prec):
            memory, bias = inputs(16, prec, 14)
            t, p, s, L, rows = e.decode_until_eos(memory, bias, eos=EOS, n_cand=16, max_len=128, sampling="multinomial",
                                                  precision=prec, **rng)
            return (t, p, L), s, rows

    for name, B, k, pmr in (("multinomial_small", 16, 16, False), ("multinomial_large", 64, 128, False),
                            ("memory_streams_small", 16, 16, True), ("memory_streams_large", 64, 128, True)):
        @case(name)
        def _(e, B=B, k=k, pmr=pmr):
            memory, bias = inputs(B, "bf16", 31)
            t, p, s = e.decode(memory, bias, n_cand=k, max_len=128, sampling="multinomial", precision="bf16",
                               per_memory_rng=pmr, **rng)
            return (t, p), s, None

    for name, B, k, eos in (("controlled_small", 16, 16, None), ("controlled_small_eos", 16, 16, EOS),
                            ("controlled_large", 64, 128, None), ("controlled_large_eos", 64, 128, EOS)):
        @case(name)
        def _(e, B=B, k=k, eos=eos):
            memory, bias = inputs(B, "bf16", 41)
            r = e.decode_controlled(memory, bias, n_cand=k, max_len=128, temperature=cols(B, 0.6, 1.6, 1),
                                    top_k=np.where(np.arange(B) % 3 == 0, 0, 10).astype(np.int32), top_p=cols(B, 0.7, 1.0, 2),
                                    eos=eos, precision="bf16", **rng)
            return (r[0], r[1]) + ((r[3],) if eos is not None else ()), r[2], r[4] if eos is not None else None

    for prec in ("fp32", "bf16"):
        @case(f"teacher_forced_{prec}")
        def _(e, prec=prec):
            memory, bias = inputs(8, prec, 51)
            trg = torch.randint(0, e.vocab, (40, 8 * 4), generator=torch.Generator().manual_seed(5)).to(dev)
            return (e.teacher_forced(memory, bias, trg, n_cand=4, precision=prec),), None, None

        @case(f"teacher_forced_scores_{prec}")
        def _(e, prec=prec):
            memory, bias = inputs(8, prec, 51)
            g = torch.Generator().manual_seed(6)
            trg, tgt = (torch.randint(0, e.vocab, (40, 8 * 4), generator=g).to(dev) for _ in range(2))
            return e.teacher_forced_scores(memory, bias, trg, tgt, n_cand=4, sampling="multinomial", precision=prec, **rng), None, None

        @case(f"beam_search_{prec}")
        def _(e, prec=prec):
            memory, bias = inputs(6, prec, 61)
            *out, s = e.beam_search(memory, bias, beam_size=8, gen_len=128, eos=EOS, precision=prec)
            return tuple(out), s, None

        @case(f"sample_without_replacement_twice_{prec}")
        def _(e, prec=prec):
            memory, bias = inputs(12, prec, 71)
            res = []
            for temp in (1.0, cols(12, 0.5, 1.5, 3)):      # the second call reuses the first call's step graph
                *out, s = e.sample_without_replacement(memory, bias, n_cand=16, max_len=128, temperature=temp, eos=EOS,
                                                       precision=prec, **rng)
                res += out
            return tuple(res), s, None

    def run_case(e, fn):
        l0 = e.launch_count()
        out, steps, rows = fn(e)
        torch.cuda.synchronize()
        out = [t.detach().cpu() for t in out if t is not None]
        return {"out": out, "steps": steps, "rows": None if rows is None else rows.cpu().tolist(),
                "launches": e.launch_count() - l0}

    def engine(model, env):
        for k, v in env.items():
            os.environ[k] = v
        try:
            return Engine(models[model], cfg0, dev)
        finally:
            for k in env:
                del os.environ[k]

    res = {}
    for env_name, env in ENVS.items():
        engines = {}
        for name, (model, multi, fn) in cases.items():
            key = (model, multi)
            if key not in engines:
                engines[key] = engine(model, {**env, **(MULTI_WAVE if multi else {})})
            e = engines[key]
            r = run_case(e, fn)
            e.profile(True)            # profiled pass: launches per kernel name (the path without graphs)
            fn(e)
            rep = e.profile_report()
            e.profile(False)
            r["profile"] = {k: v["launches"] for k, v in rep.items()}
            res[f"{env_name}/{name}"] = r
        del engines, e
        gc.collect()
        torch.cuda.empty_cache()
    res["_device"] = torch.cuda.get_device_name(0)
    torch.save(res, out_path)


def compare(a, b):
    import torch

    def same(x, y):
        return x.dtype == y.dtype and x.shape == y.shape and torch.equal(x.contiguous().view(torch.uint8), y.contiguous().view(torch.uint8))

    rows, bad = [], 0
    for k in sorted(x for x in a if not x.startswith("_")):
        ra, rb = a[k], b.get(k)
        r = {"call": k, "outputs_bit_identical": rb is not None and len(ra["out"]) == len(rb["out"]) and all(same(x, y) for x, y in zip(ra["out"], rb["out"]))}
        for f in ("steps", "rows", "launches", "profile"):
            r[f + "_equal"] = rb is not None and ra[f] == rb[f]
        r.update(h_steps=ra["steps"], launches=ra["launches"], profiled_launches=sum(ra["profile"].values()),
                 rows_sum=None if ra["rows"] is None else sum(ra["rows"]))
        ok = all(v for f, v in r.items() if f.endswith("_equal") or f == "outputs_bit_identical")
        bad += not ok
        rows.append(r)
    missing = sorted(set(x for x in b if not x.startswith("_")) - set(a))
    return rows, bad + len(missing), missing


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib-a", help="the reference build (e.g. the parent commit's)")
    ap.add_argument("--lib-b", default=None, help="the build under test (default: the in-tree build)")
    ap.add_argument("--out", default=None, help="JSON summary")
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        return worker(args.worker)
    if not args.lib_a:
        ap.error("--lib-a is required")
    import torch
    with tempfile.TemporaryDirectory() as tmp:
        res = {}
        for tag, lib in (("a", args.lib_a), ("b", args.lib_b)):
            env = dict(os.environ)
            env.pop("MMT_B200_LIB", None)
            if lib:
                env["MMT_B200_LIB"] = os.path.abspath(lib)
            path = os.path.join(tmp, tag + ".pt")
            subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", path], env=env, check=True)
            res[tag] = torch.load(path, weights_only=False)
    rows, bad, missing = compare(res["a"], res["b"])
    summary = {"device": res["a"]["_device"], "lib_a": args.lib_a, "lib_b": args.lib_b or "in-tree build",
               "calls": len(rows), "calls_differing": bad, "missing_in_a": missing, "envs": ENVS, "multi_wave_env": MULTI_WAVE,
               "results": rows}
    text = json.dumps(summary, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(json.dumps({k: v for k, v in summary.items() if k != "results"}))
    for r in rows:
        if not all(v for f, v in r.items() if f.endswith("_equal") or f == "outputs_bit_identical"):
            print("DIFFERS", json.dumps(r))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
