"""Batched candidate generation in per-memory RNG streams, and distinct SMILES per memory column on the device.

Per-memory streams (``per_memory_rng=True``, ``mmt_decode_memory_streams``): the k candidates of memory column b draw
what the reference's per-spectrum loop draws -- one torch.multinomial((k, V), 1) per step, spectrum after spectrum --
so one call over many spectra reproduces that loop seed for seed.  Column b at step t uses generator offset
off + ((b0 + b) * max_len + t) * inc(k * V) with b0 = seq_index_base / k.

``distinct_smiles`` (``mmt_distinct_smiles``) is compared with the host path: tensor_to_smiles + dict.fromkeys per column.

Near-tie rule (fp32 check mode, as test_gpu_parity / test_gpu_baseline_sizes): the engine and the oracle are two fp32
evaluations of the same model, so a sequence may leave the oracle's ids only where the oracle's own p / q has a near-tie
between the two picks; the rest of that sequence is a different continuation and is not compared.
"""
import os
import sys

import pytest
import torch

STOI = {"<PAD>": 0, "<UNK>": 1, "<EOS>": 2, "<SOS>": 3, "<MASK>": 4}
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
V = 43
_S = {}

gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------------- fixtures
def setup():
    if "model" not in _S:
        import multimodalspectraltransformer_b200 as M
        from oracle import mmt_oracle as O
        cfg = M.default_config(device="cuda")
        torch.manual_seed(0)
        model = M.MultimodalTransformer(cfg).eval()
        _S.update(M=M, O=O, model=model, P=O.random_init_state_dict(O.default_config(), seed=0))
    return _S


@pytest.fixture(autouse=True, scope="module")
def _release_engines():
    """Free this module's engines (the bench-geometry decode leaves a one-wave arena of tens of GB) before the modules
    that follow in the same process allocate theirs."""
    yield
    _S.clear()
    import gc
    gc.collect()
    if torch.cuda.is_available():
        torch.cuda.empty_cache()


def cfg_for(**over):
    return setup()["M"].default_config(device="cuda", **over)


def model_with(monkeypatch, **env):
    """A model with the same seeded weights whose engine is created under the given MMT_* knobs."""
    M = setup()["M"]
    from multimodalspectraltransformer_b200.engine import engine_for
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    torch.manual_seed(0)
    m = M.MultimodalTransformer(cfg_for()).eval()
    engine_for(m, cfg_for())
    for k in env:
        monkeypatch.delenv(k)
    return m


def _engine_of(s):
    from multimodalspectraltransformer_b200.engine import engine_for
    return engine_for(s["model"], cfg_for())


def _gen():
    return torch.cuda.default_generators[torch.cuda.current_device()]


def _near_tie_check(eng, Pd, O, mem, mask, ocfg, tok, otok, k, col0, off0, inc, T):
    """Sequences whose ids differ from the oracle's: the first divergence must be a near-tie of p / q under the oracle's
    p (its prefix, fp32) and the bit-exact Exp(1) variates of that column's call.  Returns the fraction identical."""
    same = (tok == otok).all(dim=0)
    for n in torch.nonzero(~same)[:, 0].tolist():
        b, j = n // k, n % k
        t = int(torch.nonzero(tok[:, n] != otok[:, n])[0])
        prefix = torch.cat([torch.full((1,), 3, dtype=torch.long, device="cuda"), otok[:t, n]])[:, None]
        with torch.no_grad():
            lg = O.teacher_forced_logits(Pd, mem[:, b:b + 1], mask[b:b + 1], prefix, ocfg)[-1, 0]
        p = torch.softmax(lg / ocfg.temperature, dim=0)
        q = eng.exponential(V, seed=_S["seed"], offset=off0 + ((col0 + b) * T + t) * inc, elem_base=j * V, numel_total=k * V)
        r = p / q
        a, m = r[otok[t, n]], r[tok[t, n]]
        assert float((a - m).abs()) <= 1e-5 * float(a), (n, t, float(a), float(m))
    return same.float().mean().item()


# ---------------------------------------------------------------------------------------------- CPU: bookkeeping
class _FakeEng:
    def philox_increment(self, n_total):
        from multimodalspectraltransformer_b200 import _lib
        return int(_lib.lib().mmt_philox_increment(n_total * V, 148, 2048))


def test_philox_advance_is_one_call_per_column_and_step():
    """Per-memory streams consume what the reference's loop does: B columns x T steps of one (k, V) call each."""
    from multimodalspectraltransformer_b200.generate import _philox_advance
    eng = _FakeEng()
    for B, k, T in ((1, 1, 1), (7, 5, 12), (1024, 128, 128), (3, 30000, 4)):
        inc = eng.philox_increment(k)
        assert _philox_advance(eng, k, B * k, T, True) == B * T * inc
        off = 0
        for _ in range(B):            # the reference: one multinomial_sequence_multi per spectrum
            for _ in range(T):
                off += inc
        assert _philox_advance(eng, k, B * k, T, True) == off
        assert _philox_advance(eng, k, B * k, T, False) == T * eng.philox_increment(B * k)
    assert eng.philox_increment(128) == 4 and eng.philox_increment(1024 * 128) == 20


def test_per_memory_rng_argument_validation():
    """Greedy with per-memory streams, or a base that is not a column boundary, is refused before any device work."""
    import types
    from multimodalspectraltransformer_b200 import generate as G, scheduler
    model = types.SimpleNamespace(eval=lambda: None)
    with pytest.raises(ValueError, match="per_memory_rng"):
        G._decode(model, None, None, None, "greedy", False, 4, 0, 0, per_memory_rng=True)
    with pytest.raises(ValueError, match="per_memory_rng"):
        G._decode(model, None, None, None, "multinomial", False, 4, 6, 0, per_memory_rng=True)
    with pytest.raises(ValueError, match="per_memory_rng"):
        scheduler.generate_sharded(model, {}, None, STOI, sampling="greedy", per_memory_rng=True)


def test_distinct_smiles_argument_validation():
    from multimodalspectraltransformer_b200 import smiles
    itos = {"0": "<PAD>", "2": "<EOS>"}
    with pytest.raises(ValueError):
        smiles.distinct_smiles(torch.zeros(4, 6, dtype=torch.long), itos, 3)       # host tensor
    with pytest.raises(ValueError):
        smiles.distinct_smiles(torch.zeros(6, dtype=torch.long), itos, 3)          # not (T, N)


# ------------------------------------------------------------------------------------------- GPU: RNG, bit-exact
@gpu
@pytest.mark.parametrize("k,B,base_cols", [(1, 40, 3), (16, 9, 5), (128, 6, 2), (130, 5, 1), (8000, 3, 4), (30000, 2, 1)])
def test_sample_memory_streams_reproduces_per_column_torch_multinomial(k, B, base_cols):
    """Torch's own probabilities through the per-memory mapping == a Python loop of torch.multinomial(p[b*k:(b+1)*k], 1)
    with the generator at each column's offset, for every step checked.  k = 8000 reaches the .y/.z/.w components,
    30,000 the second loop iteration.  A reference with the global mapping, or with a column stride off by one step,
    does not match."""
    s = setup()
    from multimodalspectraltransformer_b200.engine import engine_for
    eng = engine_for(s["model"], cfg_for())
    N, T = B * k, 5
    g = torch.Generator().manual_seed(k)
    W, bias = s["model"].fc_out.weight.detach().cuda(), s["model"].fc_out.bias.detach().cuda()
    x = torch.randn(N, 128, generator=g).cuda()
    p = torch.softmax(torch.nn.functional.linear(x, W, bias), dim=1)
    gen = _gen()
    torch.manual_seed(99)
    torch.empty(10, device="cuda").uniform_()
    seed, off0 = gen.initial_seed(), gen.get_offset()
    inc = eng.philox_increment(k)
    base = base_cols * k
    for t in (0, 2, T - 1):
        want = []
        for b in range(B):
            gen.set_offset(off0 + ((base_cols + b) * T + t) * inc)
            want.append(torch.multinomial(p[b * k:(b + 1) * k], 1)[:, 0])
            assert gen.get_offset() - (off0 + ((base_cols + b) * T + t) * inc) == inc
        want = torch.cat(want)
        got, _ = eng.sample_memory_streams(p=p, n_cand=k, max_len=T, step=t, seed=seed, offset=off0, seq_index_base=base)
        assert torch.equal(got, want), (k, t)
        # sharpness: the global mapping, and a stride of T - 1 or T + 1 steps per column, draw other ids
        gen.set_offset(off0 + t * eng.philox_increment(N))
        glob = torch.multinomial(p, 1)[:, 0]
        assert not torch.equal(glob, want)
        for stride in (T - 1, T + 1):
            if stride < 1 or t >= stride:
                continue
            off_by = torch.cat([_draw(gen, p[b * k:(b + 1) * k], off0 + ((base_cols + b) * stride + t) * inc) for b in range(B)])
            assert not torch.equal(off_by, want), stride
        # the fused sampler (fc_out + softmax + pick in one kernel): one row per warp below 8,192 rows, four at and above
        tok, pr = eng.sample_memory_streams(x=x, n_cand=k, max_len=T, step=t, seed=seed, offset=off0, seq_index_base=base)
        assert (tok == want).float().mean().item() > 0.9995
        bad = torch.nonzero(tok != want)[:, 0]
        for n in bad.tolist():
            b, j = n // k, n % k
            q = eng.exponential(V, seed=seed, offset=off0 + ((base_cols + b) * T + t) * inc, elem_base=j * V, numel_total=k * V)
            r = p[n] / q
            assert float((r[want[n]] - r[tok[n]]).abs()) <= 1e-5 * float(r[want[n]]), (n, t)
        torch.testing.assert_close(pr, p.gather(1, tok[:, None])[:, 0], atol=1e-6, rtol=1e-5)


def _draw(gen, p, off):
    gen.set_offset(off)
    return torch.multinomial(p, 1)[:, 0]


# ------------------------------------------------------------------------- GPU: end to end against the reference
def _oracle_serial(s, memory, mask, k, T, seed_val, col_range=None):
    """The reference's production loop: torch.manual_seed once, then one multinomial_sequence_multi per spectrum on k
    duplicates (the oracle, full-prefix decoder, on this device).  -> (tokens (T, B*k), offset consumed)."""
    O = s["O"]
    Pd = s.setdefault("Pd", {kk: v.cuda() for kk, v in s["P"].items()})
    ocfg = O.default_config(max_len=T)
    gen = _gen()
    torch.manual_seed(seed_val)
    off0 = gen.get_offset()
    out = []
    for b in range(memory.shape[1]) if col_range is None else col_range:
        with torch.no_grad():
            tok, _ = O.multinomial_sequence_multi(Pd, memory[:, b:b + 1].expand(-1, k, -1).contiguous(),
                                                  mask[b:b + 1].expand(k, -1).contiguous(), ocfg, max_len=T)
        out.append(tok)
    return torch.cat(out, dim=1), gen.get_offset() - off0, Pd, ocfg


@gpu
@pytest.mark.parametrize("geometry", ["fused", "unfused_waves"])
def test_batched_call_equals_reference_per_spectrum_loop_fp32(geometry, monkeypatch):
    """One engine call with per_memory_rng=True == the reference's loop over spectra, fp32 check mode: the same generator
    offset afterwards and identical ids for >= 95 % of sequences, every other one leaving at a near-tie.  'fused': one
    small wave on the fused kernels, split into lanes.  'unfused_waves': MMT_FUSED_DECODE_ROWS=0 and waves of 4 columns,
    so the column base of every wave after the first follows n0."""
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    from multimodalspectraltransformer_b200.engine import engine_for
    M = s["M"]
    B, k, T = (8, 16, 10) if geometry == "fused" else (10, 64, 6)
    model = s["model"] if geometry == "fused" else model_with(monkeypatch, MMT_FUSED_DECODE_ROWS="0", MMT_MAX_WAVE_SEQS="256")
    cfg = cfg_for(precision="fp32", max_len=T)
    eng = engine_for(model, cfg)
    data = synthetic.make_spectra(B, seed=5150 + B)
    memory, mask, *_ = M.run_model(model, data, cfg)
    otok, oinc, Pd, ocfg = _oracle_serial(s, memory, mask, k, T, 2024)
    gen = _gen()
    torch.manual_seed(2024)
    off0 = gen.get_offset()
    _S["seed"] = gen.initial_seed()
    tok, _ = M.multinomial_sequence_multi(model, memory, mask, STOI, cfg, n_candidates=k, per_memory_rng=True)
    assert gen.get_offset() - off0 == oinc == B * T * eng.philox_increment(k)
    frac = _near_tie_check(eng, Pd, s["O"], memory, mask, ocfg, tok, otok, k, 0, off0, eng.philox_increment(k), T)
    assert frac >= 0.95, frac
    assert bool((tok[0] == otok[0]).all())


@gpu
def test_bench_geometry_bf16_columns_of_first_middle_last_wave():
    """1024 spectra x 128 candidates in the bf16 tensor-core mode, 16 positions: columns of the first, a middle and the
    last 128-spectrum block against the reference's per-spectrum call (generator at that spectrum's offset in the serial
    loop), under the bf16 floor of test_gpu_baseline_sizes; and the whole call's offset bookkeeping."""
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    from multimodalspectraltransformer_b200.engine import engine_for
    M, O = s["M"], s["O"]
    B, k, T = 1024, 128, 16
    data = synthetic.make_spectra(B, seed=3003)
    cfg = cfg_for(precision="bf16", max_len=T)
    eng = engine_for(s["model"], cfg)
    memory, mask, *_ = M.run_model(s["model"], data, cfg)
    mem32, mask32, *_ = M.run_model(s["model"], data, cfg_for(precision="fp32"))
    gen = _gen()
    torch.manual_seed(4242)
    off0 = gen.get_offset()
    tok, pr = M.multinomial_sequence_multi(s["model"], memory, mask, STOI, cfg, n_candidates=k, per_memory_rng=True)
    inc = eng.philox_increment(k)
    assert inc == 4 and gen.get_offset() == off0 + B * T * inc
    Pd = s.setdefault("Pd", {kk: v.cuda() for kk, v in s["P"].items()})
    ocfg = O.default_config(max_len=T)
    for b in (5, 3 * 128 + 77, 7 * 128 + 127):
        gen.set_offset(off0 + b * T * inc)
        with torch.no_grad():
            otok, opr = O.multinomial_sequence_multi(Pd, mem32[:, b:b + 1].expand(-1, k, -1).contiguous(),
                                                     mask32[b:b + 1].expand(k, -1).contiguous(), ocfg, max_len=T)
        cols = slice(b * k, (b + 1) * k)
        same = (tok[:, cols] == otok).all(dim=0)
        assert bool((tok[0, cols] == otok[0]).all())
        assert same.float().mean().item() >= 0.6, (b, same.float().mean().item())
        assert float((pr[:, cols][:, same] - opr[:, same]).abs().max()) < 2e-2


# ---------------------------------------------------------------------------------------- GPU: self-consistency
@gpu
def test_batched_equals_per_column_calls_and_shards():
    """fp32 small waves: one call over B columns == B one-column calls at seq_index_base = b*k, and a shard
    memory[:, lo:hi] at seq_index_base = lo*k reproduces those columns, bit for bit (ids and probabilities)."""
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    M = s["M"]
    B, k, T = 6, 16, 8
    cfg = cfg_for(precision="fp32", max_len=T)
    memory, mask, *_ = M.run_model(s["model"], synthetic.make_spectra(B, seed=77), cfg)
    gen = _gen()
    torch.manual_seed(5)
    off0 = gen.get_offset()
    tok, pr = M.multinomial_sequence_multi(s["model"], memory, mask, STOI, cfg, n_candidates=k, per_memory_rng=True)
    off1 = gen.get_offset()
    for b in range(B):
        gen.set_offset(off0)
        tb, pb = M.multinomial_sequence_multi(s["model"], memory[:, b:b + 1], mask[b:b + 1], STOI, cfg, n_candidates=k,
                                              seq_index_base=b * k, n_total=B * k, per_memory_rng=True)
        assert torch.equal(tb, tok[:, b * k:(b + 1) * k]) and torch.equal(pb, pr[:, b * k:(b + 1) * k]), b
        assert gen.get_offset() == off1          # every shard advances by the whole call
    lo, hi = 2, 5
    gen.set_offset(off0)
    ts, ps = M.multinomial_sequence_multi(s["model"], memory[:, lo:hi], mask[lo:hi], STOI, cfg, n_candidates=k,
                                          seq_index_base=lo * k, n_total=B * k, per_memory_rng=True)
    assert torch.equal(ts, tok[:, lo * k:hi * k]) and torch.equal(ps, pr[:, lo * k:hi * k])
    # the serial pattern: column b alone with the generator where the loop leaves it == column b of the batched call
    gen.set_offset(off0 + 3 * T * _engine_of(s).philox_increment(k))
    t3, _ = M.multinomial_sequence_multi(s["model"], memory[:, 3:4], mask[3:4], STOI, cfg, n_candidates=k, per_memory_rng=True)
    assert torch.equal(t3, tok[:, 3 * k:4 * k])
    # the global mapping draws something else
    gen.set_offset(off0)
    tg, _ = M.multinomial_sequence_multi(s["model"], memory, mask, STOI, cfg, n_candidates=k)
    assert not torch.equal(tg, tok)


@gpu
def test_graph_cache_tells_the_modes_apart(monkeypatch):
    """Alternating both RNG modes and two seeds on one engine (cached decode graphs) gives, every time, the draws of an
    engine that caches no graph."""
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    M = s["M"]
    B, k, T = 4, 16, 8
    cfg = cfg_for(precision="fp32", max_len=T)
    memory, mask, *_ = M.run_model(s["model"], synthetic.make_spectra(B, seed=31), cfg)
    fresh = model_with(monkeypatch, MMT_NO_GRAPH_CACHE="1")

    def run(m, per_memory, seed):
        torch.manual_seed(seed)
        return M.multinomial_sequence_multi(m, memory, mask, STOI, cfg, n_candidates=k, per_memory_rng=per_memory)[0]

    want = {(pm, sd): run(fresh, pm, sd) for pm in (False, True) for sd in (11, 12)}
    assert not torch.equal(want[(False, 11)], want[(True, 11)])
    for pm, sd in [(False, 11), (True, 11), (False, 12), (True, 12), (True, 11), (False, 11), (True, 12)]:
        assert torch.equal(run(s["model"], pm, sd), want[(pm, sd)]), (pm, sd)


@gpu
def test_greedy_or_misaligned_base_raises():
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    from multimodalspectraltransformer_b200.engine import engine_for
    M = s["M"]
    cfg = cfg_for(precision="fp32", max_len=4)
    memory, mask, *_ = M.run_model(s["model"], synthetic.make_spectra(2, seed=1), cfg)
    with pytest.raises(ValueError):
        M.multinomial_sequence_multi(s["model"], memory, mask, STOI, cfg, n_candidates=4, seq_index_base=2, n_total=16,
                                     per_memory_rng=True)
    eng = engine_for(s["model"], cfg)
    bias = torch.zeros(2, memory.shape[0], device="cuda")
    with pytest.raises(ValueError):
        eng.decode(memory, bias, n_cand=4, max_len=4, sampling="greedy", per_memory_rng=True)
    # the C ABI refuses too
    import ctypes as C
    from multimodalspectraltransformer_b200 import _lib
    for smp, base in ((_lib.SAMPLE_GREEDY, 0), (_lib.SAMPLE_MULTINOMIAL, 3)):
        a, keep = eng._decode_args(memory, bias, 4, 4, 1.0, smp, False, "fp32", 1, 0, base, 0)
        tokens = torch.empty(4, 8, dtype=torch.long, device="cuda")
        assert eng.L.mmt_decode_memory_streams(eng.h, C.byref(a), tokens.data_ptr(), None, None, eng._stream()) != 0
    with pytest.raises(RuntimeError):
        eng.sample_memory_streams(p=torch.full((8, V), 1.0 / V, device="cuda"), n_cand=4, max_len=4, seed=1, offset=0,
                                  seq_index_base=2)


def _sharded_worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from multimodalspectraltransformer_b200 import scheduler
    M, cfg, model, data = _sharded_single(dev)
    gen = torch.cuda.default_generators[rank]
    torch.manual_seed(321)
    off0 = gen.get_offset()
    tok, pr, span = scheduler.generate_sharded(model, data, cfg, STOI, n_candidates=5, sampling="multinomial",
                                               gather_probs=True, per_memory_rng=True)
    torch.cuda.synchronize()
    q.put((rank, tok.cpu(), pr.cpu(), gen.get_offset() - off0, span))
    dist.barrier()
    dist.destroy_process_group()


def _sharded_single(dev):
    import multimodalspectraltransformer_b200 as M
    from multimodalspectraltransformer_b200 import synthetic
    cfg = M.default_config(device=str(dev), max_len=12, precision="bf16")
    torch.manual_seed(0)
    model = M.MultimodalTransformer(cfg).eval()
    return M, cfg, model, synthetic.make_spectra(7, seed=909)


@gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_generate_sharded_per_memory_rng_two_ranks_equals_single_gpu():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29800 + os.getpid() % 90
    procs = [ctx.Process(target=_sharded_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=600) for _ in procs], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=120)
    M, cfg, model, data = _sharded_single(torch.device("cuda", 0))
    memory, mask, *_ = M.run_model(model, data, cfg)
    gen = torch.cuda.default_generators[0]
    torch.manual_seed(321)
    off0 = gen.get_offset()
    tok1, pr1 = M.multinomial_sequence_multi(model, memory, mask, STOI, cfg, n_candidates=5, per_memory_rng=True)
    inc1 = gen.get_offset() - off0
    assert [r[4] for r in res] == [(0, 4), (4, 7)]
    for rank, tok, pr, inc, _ in res:
        assert torch.equal(tok, tok1.cpu()) and torch.equal(pr, pr1.cpu()) and inc == inc1, rank


# ------------------------------------------------------------------------------------------ GPU: distinct SMILES
ITOS = {str(i): c for i, c in enumerate(["<PAD>", "<UNK>", "<EOS>", "<SOS>", "<MASK>", "C", "c", "O", "N", "(", ")", "=",
                                          "1", "2", "3", "[", "]", "Cl", "l", "Br", "r", "F", "S", "#", "@", "H", "+", "-",
                                          "n", "o", "s", "/", "\\", "4", "5", "6", "P", "I", "B", "%", "Si", "Se", "."])}
# multi-byte UTF-8 entries, "C"+"l" == "Cl" and "é"+"ü" == "éü" spelled both ways, and an id gap (44) that has no entry
ITOS_U = dict(ITOS, **{"43": "é", "45": "ü", "46": "éü", "47": "→", "48": ""})


def _host_distinct(tokens, itos, k, token_prob=None):
    from multimodalspectraltransformer_b200 import smiles
    out = []
    for b in range(tokens.shape[1] // k):
        cols = tokens[:, b * k:(b + 1) * k]
        strs = smiles.tensor_to_smiles(cols, itos)
        probs = smiles.tensor_to_smiles_and_prob_2(cols, token_prob[:, b * k:(b + 1) * k], itos)[1] if token_prob is not None else None
        firsts = {}
        for i, st in enumerate(strs):
            firsts.setdefault(st, i)
        assert list(firsts) == list(dict.fromkeys(strs))
        out.append([(st, i, strs.count(st), probs[i] if probs is not None else None) for st, i in firsts.items()])
    return out


def _compare(tokens, itos, k, token_prob=None):
    from multimodalspectraltransformer_b200 import distinct_smiles
    got = distinct_smiles(tokens, itos, k, token_prob=token_prob)
    want = _host_distinct(tokens, itos, k, token_prob)
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert [(d.smiles, d.index, d.count) for d in g] == [x[:3] for x in w]
        if token_prob is not None:
            for d, x in zip(g, w):
                assert torch.equal(d.prob, x[3])
    return got


def _rand_tokens(T, N, seed, vocab=(5, 43), eos_rate=0.08, device="cuda"):
    g = torch.Generator().manual_seed(seed)
    t = torch.randint(vocab[0], vocab[1], (T, N), generator=g)
    t[torch.rand(T, N, generator=g) < eos_rate] = 2
    return t.to(device)


@gpu
@pytest.mark.parametrize("k", [1, 33, 128, 4096, 5000])
def test_distinct_smiles_equals_host_path(k):
    """Random columns with many repeated candidates, at k = 1, 33, 128 and 4,096 (first-occurrence table in shared
    memory) and 5,000 (table in global memory), with probabilities."""
    B = max(1, 2048 // k) if k < 4096 else 2
    T = 24
    t = _rand_tokens(T, B * k, seed=k, vocab=(5, 9), eos_rate=0.15)       # few tokens, early <EOS>: many repeats
    prob = torch.rand(T - 1, B * k, generator=torch.Generator().manual_seed(k + 1)).cuda()
    got = _compare(t, ITOS, k, token_prob=prob)
    assert sum(d.count for col in got for d in col) == B * k


@gpu
def test_distinct_smiles_edges():
    """All-identical and all-distinct columns, <EOS> at position 0 (the empty string) and no <EOS> at all."""
    T, k = 16, 64
    same = torch.full((T, k), 5, dtype=torch.long)
    same[7] = 2
    distinct = _rand_tokens(T, k, seed=3, eos_rate=0.0).cpu()
    distinct[0] = torch.arange(k) % 38 + 5
    distinct[1] = torch.arange(k) // 38 + 5
    eos0 = _rand_tokens(T, k, seed=4).cpu()
    eos0[0, ::2] = 2
    no_eos = _rand_tokens(T, k, seed=5, eos_rate=0.0).cpu()
    t = torch.cat([same, distinct, eos0, no_eos], dim=1).cuda()
    got = _compare(t, ITOS, k)
    assert len(got[0]) == 1 and got[0][0].count == k
    assert len(got[1]) == k and all(d.count == 1 for d in got[1])
    assert got[2][0].smiles == "" and got[2][0].count >= k // 2
    assert all(d.count == 1 and len(d.smiles) >= T for d in got[3])      # T ids, each at least one character


@gpu
def test_distinct_smiles_multibyte_and_non_injective_spelling():
    """Strings are compared as bytes: "C","l" and "Cl", "é","ü" and "éü", and an empty entry all spell one string each."""
    T, k = 6, 8
    seqs = [[17, 2], [5, 18, 2], [43, 45, 2], [46, 2], [46, 48, 2], [47, 43, 2], [5, 18, 48, 2], [47, 43, 45, 2]]
    t = torch.full((T, k), 0, dtype=torch.long)
    for i, sq in enumerate(seqs):
        t[:len(sq), i] = torch.tensor(sq)
    got = _compare(t.cuda(), ITOS_U, k)
    assert [(d.smiles, d.index, d.count) for d in got[0]] == [("Cl", 0, 3), ("éü", 2, 3), ("→é", 5, 1), ("→éü", 7, 1)]
    ids = torch.tensor([5, 17, 18, 43, 45, 46, 47, 48])
    t = ids[_rand_tokens(20, 4 * 256, seed=8, vocab=(0, 8), eos_rate=0.0, device="cpu")]
    t[torch.rand(t.shape, generator=torch.Generator().manual_seed(9)) < 0.2] = 2
    _compare(t.cuda(), ITOS_U, 256)


@gpu
def test_distinct_smiles_permutations_defeat_weak_hashes():
    """Many equal-length permutations of the same tokens (equal sums and xors of ids and of bytes) stay apart."""
    import itertools
    base = [5, 6, 7, 8, 9, 10, 12]
    perms = list(itertools.permutations(base))[:2000]
    k = len(perms) * 2
    t = torch.full((9, k), 2, dtype=torch.long)
    for i, pm in enumerate(perms + perms[::-1]):
        t[:7, i] = torch.tensor(pm)
    got = _compare(t.cuda(), ITOS, k)
    assert len(got[0]) == len(perms) and all(d.count == 2 for d in got[0])


@gpu
def test_distinct_smiles_unknown_id_raises_key_error():
    from multimodalspectraltransformer_b200 import distinct_smiles, smiles
    t = _rand_tokens(10, 64, seed=9, eos_rate=0.0)
    t[3, 17] = 44                       # a gap of ITOS_U
    with pytest.raises(KeyError):
        smiles.tensor_to_smiles(t, ITOS_U)
    with pytest.raises(KeyError):
        distinct_smiles(t, ITOS_U, 16)
    t[0, 17], t[3, 17] = 2, 44          # after <EOS> an unknown id is never looked up
    _compare(t, ITOS_U, 16)


@gpu
def test_distinct_smiles_of_a_bench_decode():
    """The real output of a 1024 x 128 bf16 decode in per-memory streams, with the mrtf probability layout."""
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    M = s["M"]
    cfg = cfg_for(precision="bf16", max_len=128)
    memory, mask, *_ = M.run_model(s["model"], synthetic.make_spectra(1024, seed=3003), cfg)
    torch.manual_seed(8)
    tok, pr = M.multinomial_sequence_multi_2(s["model"], memory, mask, STOI, cfg, n_candidates=128, per_memory_rng=True)
    _compare(tok, ITOS, 128, token_prob=pr)
