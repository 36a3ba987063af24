"""Per-spectrum sampling controls: temperature, top-k and nucleus (top-p) in one multinomial decode call
(``mmt_decode_controlled``, ``mmt_sample_controlled``; the contract is in include/mmt_b200.h, mmt_sampling_controls).

The sampler draws argmax_i p_i / q_i with q the Exp(1) variates of the plain call, so restricting the arg-max to a kept set
leaves every draw the plain call makes inside that set unchanged, and a column's temperature only changes its own p: a
column of a mixed call equals that column of a uniform call with its settings, bit for bit.  Those two properties, the
kept-set rule restated in numpy fp32 (sums in ascending token index, top-k before top-p, ties to the lower index) and
the neutral controls' bit identity with the plain entry points are what this module checks.
"""
import os
import sys

import numpy as np
import pytest
import torch

STOI = {"<PAD>": 0, "<UNK>": 1, "<EOS>": 2, "<SOS>": 3, "<MASK>": 4}
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
V = 43
EOS = 2
_S = {}

gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------------- fixtures
def setup():
    if "model" not in _S:
        import multimodalspectraltransformer_b200 as M
        torch.manual_seed(0)
        _S.update(M=M, model=M.MultimodalTransformer(M.default_config(device="cuda")).eval())
    return _S


@pytest.fixture(autouse=True, scope="module")
def _release_engines():
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
    from multimodalspectraltransformer_b200.engine import engine_for
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    torch.manual_seed(0)
    m = setup()["M"].MultimodalTransformer(cfg_for()).eval()
    engine_for(m, cfg_for())
    for k in env:
        monkeypatch.delenv(k)
    return m


def inputs(model, B, prec, seed):
    from multimodalspectraltransformer_b200 import synthetic
    from multimodalspectraltransformer_b200.engine import engine_for
    from multimodalspectraltransformer_b200.generate import _mask_to_bias
    cfg = cfg_for(precision=prec)
    memory, mask, *_ = setup()["M"].run_model(model, synthetic.make_spectra(B, seed=seed), cfg)
    return engine_for(model, cfg), memory, _mask_to_bias(mask)


def mixed_controls(B, seed):
    """Per-column temperatures, top-k and top-p covering off / sharp / loose values."""
    g = np.random.default_rng(seed)
    t = g.choice(np.array([0.6, 1.0, 1.7], np.float32), B)
    k = g.choice(np.array([0, 1, 2, 20, V], np.int32), B)
    p = g.choice(np.array([1e-4, 0.5, 0.9, 1.0], np.float32), B)
    return t, k, p


# ------------------------------------------------------------------------------------------- the contract in numpy
def restate_kept(P, k, tp, *, sum_rank_order=False, p_first=False, tie_high=False):
    """Kept set (N,V) bool of probabilities P (N,V) f32 under per-row top-k k (N,) and top-p tp (N,) f32.  The keyword
    arguments select wrong restatements (sums in rank order, top-p before top-k, ties kept by the higher index) for the
    sharpness check."""
    N, Vv = P.shape
    idx = np.arange(Vv)
    gt = P[:, None, :] > P[:, :, None]                                  # [n, i, j]: p_j > p_i
    eq = P[:, None, :] == P[:, :, None]
    lower = (idx[None, :] > idx[:, None]) if tie_high else (idx[None, :] < idx[:, None])   # [i, j]
    before = gt | (eq & lower[None])                                      # j ranks before i
    rank = before.sum(2)
    kk = np.where((k <= 0) | (k >= Vv), Vv, k)[:, None]
    surv = rank < kk
    base = np.ones_like(surv) if p_first else surv
    mass = np.zeros(N, np.float32)
    bf = np.zeros((N, Vv), np.float32)
    if sum_rank_order:
        order = np.argsort(rank, axis=1)
        rows = np.arange(N)
        for r in range(Vv):
            j = order[:, r]
            pj = P[rows, j]
            mass = np.where(base[rows, j], mass + pj, mass).astype(np.float32)
            bf = np.where(rank > r, bf + pj[:, None], bf).astype(np.float32)
    else:
        for j in range(Vv):
            pj = P[:, j]
            mass = np.where(base[:, j], mass + pj, mass).astype(np.float32)
            bf = np.where(before[:, :, j], bf + pj[:, None], bf).astype(np.float32)
    lim = (tp.astype(np.float32) * mass).astype(np.float32)
    keep_p = (rank == 0) | (bf < lim[:, None]) | (tp >= 1)[:, None]
    return surv & keep_p, bf, lim, rank


def draw(P, kept, q):
    r = np.where(kept, P / q, -np.inf).astype(np.float32)
    return r.argmax(1)


# ---------------------------------------------------------------------------------------------- unit exactness
def probe_probs(N, seed):
    """Probabilities the controlled pick is checked on: even rows a softmax of random logits (inexact fp32 sums), odd
    rows multiples of 1/64 with many ties; every fourth row's top-p is set so that a token sits exactly on the nucleus
    boundary of the index-order sums (the rank-order sums then land on the other side on some rows)."""
    g = np.random.default_rng(seed)
    lg = g.standard_normal((N, V)).astype(np.float32) * g.uniform(0.5, 4.0, (N, 1)).astype(np.float32)
    P = np.exp(lg - lg.max(1, keepdims=True))
    P = (P / P.sum(1, keepdims=True)).astype(np.float32)
    P[1::2] = (np.floor(P[1::2] * 64) / 64 + g.integers(0, 2, (N // 2, V)) / 64).astype(np.float32)
    P[1::2, 0] += 1.0 / 64
    return P


@gpu
@pytest.mark.parametrize("N", [128, 8193, 75779])
def test_sample_controlled_on_probabilities_is_the_contract(N):
    """The kept set and the draw on given probabilities equal the numpy restatement bit for bit, both RNG mappings; the
    wrong restatements differ on some rows of the same inputs."""
    from multimodalspectraltransformer_b200.engine import engine_for
    eng = engine_for(setup()["model"], cfg_for())
    P = probe_probs(N, N)
    g = np.random.default_rng(N + 1)
    k = g.choice(np.array([0, 1, 2, 20, V], np.int32), N)
    tp = g.choice(np.array([1e-4, 0.5, 0.9, 1.0], np.float32), N)
    # rows on the nucleus boundary: top_p * mass == before_i of a middle-ranked token (index-order sums)
    _, bf, _, rank = restate_kept(P, k, np.ones(N, np.float32))
    kept_k, _, _, _ = restate_kept(P, k, np.ones(N, np.float32))
    for n in range(0, N, 4):
        m = np.float32(0)
        for j in range(V):
            if kept_k[n, j]:
                m = np.float32(m + P[n, j])
        i = int(np.argmax(rank[n] == min(3, int(kept_k[n].sum()) - 1)))
        if rank[n, i] == 0:
            continue
        c = np.float32(bf[n, i] / m)
        while np.float32(c * m) < bf[n, i]:
            c = np.nextafter(c, np.float32(2))
        if 0 < c < 1:
            tp[n] = c
    seed, off, step, T = 4242, 8 * 13, 2, 4
    want_kept, _, _, _ = restate_kept(P, k, tp)
    for per_memory in (False, True):
        tok, pr, _, kept = eng.sample_controlled(p=torch.from_numpy(P), n_cand=1, top_k=k, top_p=tp, per_memory_rng=per_memory,
                                                 max_len=T, step=step, seed=seed, offset=off, want_kept=True)
        assert np.array_equal(kept.cpu().numpy().astype(bool), want_kept)
        tok, pr = tok.cpu().numpy(), pr.cpu().numpy()
        assert np.array_equal(pr, P[np.arange(N), tok])
        if not per_memory:
            inc = eng.philox_increment(N)
            q = eng.exponential(N * V, seed=seed, offset=off + step * inc).view(N, V).cpu().numpy()
            assert np.array_equal(tok, draw(P, want_kept, q))
        # the plain draw where it is kept, a kept token everywhere
        plain = (eng.sample_memory_streams(p=torch.from_numpy(P), n_cand=1, max_len=T, step=step, seed=seed, offset=off)[0] if per_memory else
                 _plain_probs_draw(eng, P, seed, off + step * eng.philox_increment(N))).cpu().numpy()
        inside = want_kept[np.arange(N), plain]
        assert np.array_equal(tok[inside], plain[inside])
        assert bool(want_kept[np.arange(N), tok].all())
        assert (~inside).any() and inside.any()
    # sharpness (on the larger inputs, whose boundary rows are many): each wrong restatement differs on some rows
    for wrong in () if N < 8193 else (dict(sum_rank_order=True), dict(p_first=True), dict(tie_high=True)):
        assert not np.array_equal(restate_kept(P, k, tp, **wrong)[0], want_kept), wrong


def _plain_probs_draw(eng, P, seed, offset):
    return eng.sample_probs(torch.from_numpy(P), seed=seed, offset=offset)


@gpu
@pytest.mark.parametrize("N", [128, 8193, 75779])
@pytest.mark.parametrize("per_memory", [False, True])
def test_sample_controlled_on_hidden_states(N, per_memory):
    """The fused form (fc_out + softmax(logits / T[column]) + controlled pick; one row per warp at N = 128, four from
    8,193 on, with a tail): every draw the plain sampler makes inside the kept set is kept with its probability bit for bit,
    every draw is a kept token, and the kept set is the restatement on the kernel's own logits except where the
    restatement's fp32 sums sit within 1e-6 of the nucleus boundary or p has a near-tie (counted, rare)."""
    from multimodalspectraltransformer_b200.engine import engine_for
    eng = engine_for(setup()["model"], cfg_for())
    n_cand = 128 if per_memory else 7
    Bm = (N + n_cand - 1) // n_cand
    x = torch.randn(N, 128, generator=torch.Generator().manual_seed(N)) * 1.5
    t, k, tp = mixed_controls(Bm, N + per_memory)
    seed, off, T, step = 99, 4 * 31, 6, 3 if per_memory else 0
    tok, pr, lg, kept = eng.sample_controlled(x=x, n_cand=n_cand, temperature=t, top_k=k, top_p=tp, per_memory_rng=per_memory,
                                              max_len=T, step=step, seed=seed, offset=off, want_logits=True, want_kept=True)
    tok, pr, kept = tok.cpu().numpy(), pr.cpu().numpy(), kept.cpu().numpy().astype(bool)
    col = np.arange(N) // n_cand
    assert bool(kept[np.arange(N), tok].all())
    ptok, ppr = np.empty(N, np.int64), np.empty(N, np.float32)
    for temp in np.unique(t):
        rows = t[col] == temp
        if per_memory:
            a, b = eng.sample_memory_streams(x=x, n_cand=n_cand, max_len=T, step=step, temperature=float(temp), seed=seed, offset=off)
        else:
            a, b, _ = eng.sample(x, temperature=float(temp), sampling="multinomial", seed=seed, offset=off)
        ptok[rows], ppr[rows] = a.cpu().numpy()[rows], b.cpu().numpy()[rows]
    inside = kept[np.arange(N), ptok]
    assert np.array_equal(tok[inside], ptok[inside]) and np.array_equal(pr[inside], ppr[inside])
    assert (~inside).any() and inside.any()
    # the kept set against the restatement on the kernel's logits
    z = lg.cpu().numpy() / t[col][:, None]
    P = np.exp(z - z.max(1, keepdims=True))
    P = (P / P.sum(1, keepdims=True)).astype(np.float32)
    want, bf, lim, _ = restate_kept(P, k[col], tp[col])
    bad = np.nonzero((want != kept).any(1))[0]
    for n in bad:
        near = (np.abs(bf[n] - lim[n]) <= 1e-6) | ((np.abs(P[n][:, None] - P[n][None, :]) <= 1e-6 * P[n].max()).sum(1) > 1)
        assert near[want[n] != kept[n]].all(), n
    assert len(bad) <= max(3, N // 1000), len(bad)


# --------------------------------------------------------------------------------------- neutral controls are invisible
NEUTRAL_CASES = ["fused_fp32", "fused_bf16", "bench_bf16", "waves", "per_memory", "eos_large", "eos_fused"]


@gpu
@pytest.mark.parametrize("case", NEUTRAL_CASES)
def test_neutral_controls_equal_the_plain_call(case, monkeypatch):
    """Explicit neutral arrays through mmt_decode_controlled (not the Python short-cut): ids, probabilities, lengths, rows and
    steps bit-identical to the plain call."""
    prec = "fp32" if case == "fused_fp32" else "bf16"
    model = model_with(monkeypatch, MMT_MAX_WAVE_SEQS="4096") if case == "waves" else setup()["model"]
    B, k, T = {"fused_fp32": (24, 16, 64), "fused_bf16": (24, 16, 64), "bench_bf16": (1024, 128, 128), "waves": (80, 128, 32),
               "per_memory": (24, 16, 64), "eos_large": (64, 128, 128), "eos_fused": (24, 16, 128)}[case]
    eng, memory, bias = inputs(model, B, prec, 17)
    kw = dict(n_cand=k, max_len=T, precision=prec, seed=777, offset=4 * 9, per_memory_rng=case == "per_memory")
    eos = EOS if case.startswith("eos") else None
    neutral = dict(temperature=np.full(B, 1.0, np.float32), top_k=np.where(np.arange(B) % 2, 0, V).astype(np.int32),
                   top_p=np.ones(B, np.float32))
    if eos is None:
        want = eng.decode(memory, bias, temperature=1.0, sampling="multinomial", **kw)
        got = eng.decode_controlled(memory, bias, **neutral, **kw)
    else:
        want = eng.decode_until_eos(memory, bias, eos=eos, temperature=1.0, sampling="multinomial", **kw)
        got = eng.decode_controlled(memory, bias, eos=eos, **neutral, **kw)
    assert len(want) == len(got)
    for a, b in zip(want, got):
        assert (torch.equal(a, b) if isinstance(a, torch.Tensor) else a == b)


# ---------------------------------------------------------------------------------------------- columns are independent
INDEP_CASES = ["fused_fp32", "fused_bf16", "unfused_bf16", "waves", "eos_large", "per_memory", "bench_bf16"]


@gpu
@pytest.mark.parametrize("case", INDEP_CASES)
def test_columns_equal_uniform_calls_with_their_settings(case, monkeypatch):
    prec = "fp32" if case == "fused_fp32" else "bf16"
    model = model_with(monkeypatch, MMT_MAX_WAVE_SEQS="4096") if case == "waves" else setup()["model"]
    B, k, T = {"fused_fp32": (24, 16, 48), "fused_bf16": (24, 16, 48), "unfused_bf16": (64, 128, 48), "waves": (80, 128, 32),
               "eos_large": (64, 128, 128), "per_memory": (40, 64, 48), "bench_bf16": (1024, 128, 128)}[case]
    eng, memory, bias = inputs(model, B, prec, 23)
    t, kk, tp = mixed_controls(B, B + k)
    cols = [0, B // 2, B - 1]
    t[cols], kk[cols], tp[cols] = [0.6, 1.0, 1.7], [20, 1, 0], [0.9, 1.0, 0.5]
    kw = dict(n_cand=k, max_len=T, precision=prec, seed=31, offset=4 * 5, per_memory_rng=case == "per_memory")
    eos = EOS if case == "eos_large" else None
    if eos is not None:
        kw["eos"] = eos
    mixed = eng.decode_controlled(memory, bias, temperature=t, top_k=kk, top_p=tp, **kw)
    for b in (cols if case == "bench_bf16" else range(0, B, max(1, B // 6))):
        one = eng.decode_controlled(memory, bias, temperature=float(t[b]), top_k=int(kk[b]), top_p=float(tp[b]), **kw)
        s = slice(b * k, (b + 1) * k)
        assert torch.equal(mixed[0][:, s], one[0][:, s]) and torch.equal(mixed[1][:, s], one[1][:, s]), b
        if eos is not None:
            assert torch.equal(mixed[3][s], one[3][s]), b


# ------------------------------------------------------------------------------------ truncation moves only excluded draws
@gpu
@pytest.mark.parametrize("B,k", [(24, 16), (64, 128)])
def test_truncation_moves_only_draws_outside_the_kept_set(B, k):
    """fp32, fused (24 x 16) and un-fused (64 x 128) waves: every sequence follows the plain call up to the first step t*
    at which the plain draw is outside the kept set (from the teacher-forced logits of the shared prefix), and at t* the
    controlled draw is the kept-set arg-max of p / q.  Cases within 1e-6 of the nucleus boundary are exempt (counted)."""
    eng, memory, bias = inputs(setup()["model"], B, "fp32", 29)
    T, seed, off = 24, 55, 4 * 3
    N = B * k
    kw = dict(n_cand=k, max_len=T, precision="fp32", seed=seed, offset=off)
    ptok, ppr, _ = eng.decode(memory, bias, temperature=1.0, sampling="multinomial", **kw)
    topk = np.full(B, 20, np.int32)
    topp = np.full(B, 0.9, np.float32)
    ctok, cpr, _ = eng.decode_controlled(memory, bias, temperature=1.0, top_k=topk, top_p=topp, **kw)
    trg = torch.cat([torch.full((1, N), 3, dtype=torch.long, device=ptok.device), ptok[:-1]])
    lg = eng.teacher_forced(memory, bias, trg, n_cand=k, precision="fp32").cpu().numpy()
    P = np.exp(lg - lg.max(2, keepdims=True))
    P = (P / P.sum(2, keepdims=True)).astype(np.float32)
    pt, ct = ptok.cpu().numpy(), ctok.cpu().numpy()
    inc = eng.philox_increment(N)
    exempt, moved = 0, 0
    kept_all = [restate_kept(P[t], np.full(N, 20, np.int32), np.full(N, 0.9, np.float32)) for t in range(T)]
    for n in range(N):
        for t in range(T):
            kept, bf, lim, _ = kept_all[t]
            near = np.abs(bf[n] - lim[n]) <= 1e-6
            if not kept[n, pt[t, n]]:
                if near[pt[t, n]]:
                    exempt += 1
                    break
                q = eng.exponential(V, seed=seed, offset=off + t * inc, elem_base=n * V, numel_total=N * V).cpu().numpy()
                want = int(draw(P[t, n][None], kept[n][None], q[None])[0])
                r = np.where(kept[n], P[t, n] / q, -np.inf)
                top2 = np.sort(r)[-2:]
                if near.any() or top2[1] - top2[0] <= 1e-6 * top2[1]:
                    exempt += 1
                else:
                    assert ct[t, n] == want, (n, t)
                moved += 1
                break
            assert ct[t, n] == pt[t, n], (n, t)
    assert moved > N // 10, moved
    assert exempt <= max(2, moved // 50), (exempt, moved)


# ------------------------------------------------------------------------------------------------------- graph cache
@gpu
def test_cached_graph_serves_other_control_values(monkeypatch):
    eng, memory, bias = inputs(setup()["model"], 24, "bf16", 41)
    kw = dict(n_cand=16, max_len=32, precision="bf16", seed=5, offset=4 * 7)
    A = dict(temperature=np.linspace(0.6, 1.8, 24).astype(np.float32), top_k=np.full(24, 20, np.int32), top_p=np.full(24, 0.9, np.float32))
    Bc = dict(temperature=np.full(24, 1.3, np.float32), top_k=np.arange(24, dtype=np.int32) % 5, top_p=np.full(24, 0.5, np.float32))
    a1 = eng.decode_controlled(memory, bias, **A, **kw)
    b1 = eng.decode_controlled(memory, bias, **Bc, **kw)
    a2 = eng.decode_controlled(memory, bias, **A, **kw)
    assert torch.equal(a1[0], a2[0]) and torch.equal(a1[1], a2[1])
    assert not torch.equal(a1[0], b1[0])
    m2 = model_with(monkeypatch, MMT_NO_GRAPH="1")
    eng2, memory2, bias2 = inputs(m2, 24, "bf16", 41)
    for ctl, got in ((A, a1), (Bc, b1)):
        ref = eng2.decode_controlled(memory2, bias2, **ctl, **kw)
        assert torch.equal(ref[0], got[0]) and torch.equal(ref[1], got[1])


# ------------------------------------------------------------------------------------------------ Python entry points
@gpu
def test_generate_entry_points_take_per_spectrum_controls():
    """multinomial_sequence_multi with per-spectrum controls = Engine.decode with the same arrays; the generator advances as
    the plain call's; neutral values equal the plain call."""
    M = setup()["M"]
    model = setup()["model"]
    from multimodalspectraltransformer_b200 import synthetic
    cfg = cfg_for(max_len=24, precision="bf16", temperature=1.2)
    memory, mask, *_ = M.run_model(model, synthetic.make_spectra(6, seed=3), cfg)
    gen = torch.cuda.default_generators[torch.cuda.current_device()]
    t, k, p = mixed_controls(6, 8)
    torch.manual_seed(11)
    off0 = gen.get_offset()
    tok0, pr0 = M.multinomial_sequence_multi(model, memory, mask, STOI, cfg, n_candidates=8)
    inc0 = gen.get_offset() - off0
    torch.manual_seed(11)
    tok1, pr1 = M.multinomial_sequence_multi(model, memory, mask, STOI, cfg, n_candidates=8, temperature=[1.2] * 6, top_k=V, top_p=1.0)
    assert torch.equal(tok0, tok1) and torch.equal(pr0, pr1) and gen.get_offset() - off0 == inc0
    torch.manual_seed(11)
    tok2, pr2 = M.multinomial_sequence_multi(model, memory, mask, STOI, cfg, n_candidates=8, temperature=torch.from_numpy(t),
                                             top_k=k, top_p=p)
    assert gen.get_offset() - off0 == inc0
    from multimodalspectraltransformer_b200.engine import engine_for
    from multimodalspectraltransformer_b200.generate import _mask_to_bias
    ref = engine_for(model, cfg).decode_controlled(memory, _mask_to_bias(mask), n_cand=8, max_len=24, temperature=t, top_k=k, top_p=p,
                                                   precision="bf16", seed=int(gen.initial_seed()), offset=off0)
    assert torch.equal(tok2, ref[0]) and torch.equal(pr2, ref[1])
    with pytest.raises(ValueError):
        engine_for(model, cfg).decode(memory, _mask_to_bias(mask), n_cand=2, max_len=4, sampling="greedy", top_k=5)


# ----------------------------------------------------------------------------------------------------- sharding
def _sharded_worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from multimodalspectraltransformer_b200 import scheduler
    out = []
    for B in (7, 1):
        M, cfg, model, data = _sharded_single(dev, B)
        gen = torch.cuda.default_generators[rank]
        torch.manual_seed(321)
        off0 = gen.get_offset()
        t, k, p = mixed_controls(B, B)
        tok, pr, span = scheduler.generate_sharded(model, data, cfg, STOI, n_candidates=5, sampling="multinomial", gather_probs=True,
                                                   per_memory_rng=True, temperature=t, top_k=k, top_p=p)
        torch.cuda.synchronize()
        out.append((tok.cpu(), pr.cpu(), gen.get_offset() - off0, span))
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


def _sharded_single(dev, B):
    import multimodalspectraltransformer_b200 as M
    from multimodalspectraltransformer_b200 import synthetic
    cfg = M.default_config(device=str(dev), max_len=12, precision="bf16")
    torch.manual_seed(0)
    model = M.MultimodalTransformer(cfg).eval()
    return M, cfg, model, synthetic.make_spectra(B, seed=909)


@gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_generate_sharded_with_controls_two_ranks_equals_single_gpu():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + os.getpid() % 90
    procs = [ctx.Process(target=_sharded_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=600) for _ in procs], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=120)
    for i, B in enumerate((7, 1)):
        M, cfg, model, data = _sharded_single(torch.device("cuda", 0), B)
        memory, mask, *_ = M.run_model(model, data, cfg)
        gen = torch.cuda.default_generators[0]
        torch.manual_seed(321)
        off0 = gen.get_offset()
        t, k, p = mixed_controls(B, B)
        tok1, pr1 = M.multinomial_sequence_multi(model, memory, mask, STOI, cfg, n_candidates=5, per_memory_rng=True,
                                                 temperature=t, top_k=k, top_p=p)
        inc1 = gen.get_offset() - off0
        for rank, out in res:
            tok, pr, inc, _ = out[i]
            assert torch.equal(tok, tok1.cpu()) and torch.equal(pr, pr1.cpu()) and inc == inc1, (B, rank)
    assert [r[1][1][3] for r in res] == [(0, 1), (1, 1)]          # B = 1: rank 1's shard is empty


# ------------------------------------------------------------------------------------------------------- validation
BAD = [dict(temperature=[1.0, 1.0]), dict(temperature=0.0, top_k=3), dict(temperature=-1.0, top_k=3),
       dict(temperature=float("nan"), top_k=3), dict(temperature=float("inf"), top_k=3), dict(top_k=-1), dict(top_k=V + 1),
       dict(top_k=2.5), dict(top_k=[1, 2]), dict(top_p=0.0), dict(top_p=1.5), dict(top_p=float("nan")), dict(top_p=[0.5] * 4)]


@pytest.mark.parametrize("bad", BAD)
def test_bad_controls_raise_before_any_engine(bad):
    """CPU: the Python entry points check the controls (3 spectra) before they create an engine."""
    import multimodalspectraltransformer_b200 as M
    from multimodalspectraltransformer_b200 import scheduler, synthetic
    cfg = M.default_config(device="cuda", num_encoder_layers=1, num_decoder_layers=1)
    model = M.MultimodalTransformer(cfg)
    memory, mask = torch.zeros(5, 3, 128), torch.zeros(3, 5, dtype=torch.bool)
    for fn in (M.multinomial_sequence_multi, M.multinomial_sequence_multi_2):
        with pytest.raises(ValueError):
            fn(model, memory, mask, STOI, cfg, n_candidates=2, **bad)
    with pytest.raises(ValueError):
        M.multinomial_sequence(model, STOI, memory, mask, cfg, n_candidates=2, **bad)
    with pytest.raises(ValueError):
        scheduler.generate_sharded(model, synthetic.make_spectra(3), cfg, STOI, n_candidates=2, **bad)


def test_greedy_with_controls_raises():
    import multimodalspectraltransformer_b200 as M
    from multimodalspectraltransformer_b200 import scheduler, synthetic
    from multimodalspectraltransformer_b200.engine import sampling_controls
    cfg = M.default_config(device="cuda", num_encoder_layers=1, num_decoder_layers=1)
    model = M.MultimodalTransformer(cfg)
    with pytest.raises(ValueError):
        scheduler.generate_sharded(model, synthetic.make_spectra(3), cfg, STOI, sampling="greedy", top_k=5)
    with pytest.raises(ValueError):
        sampling_controls(3, V, [1.0, 1.1, 1.0], sampling="greedy")
    assert sampling_controls(3, V, [1.0, 1.0, 1.0], top_k=V, top_p=1.0, sampling="greedy") == (1.0, None)


@gpu
def test_c_entry_points_refuse_bad_host_controls():
    from multimodalspectraltransformer_b200 import _lib
    from multimodalspectraltransformer_b200.engine import _controls_struct
    import ctypes as C
    eng, memory, bias = inputs(setup()["model"], 3, "fp32", 1)
    a, keep = eng._decode_args(memory, bias, 2, 4, 1.0, _lib.SAMPLE_MULTINOMIAL, False, "fp32")
    tok = torch.empty(4, 6, dtype=torch.int64, device="cuda")
    pr = torch.empty(4, 6, device="cuda")
    good = (np.ones(3, np.float32), np.zeros(3, np.int32), np.ones(3, np.float32))
    bads = [(np.ones(2, np.float32),) + good[1:], (np.array([1, 0, 1], np.float32),) + good[1:],
            (np.array([1, np.nan, 1], np.float32),) + good[1:], (good[0], np.array([0, V + 1, 0], np.int32), good[2]),
            (good[0], np.array([0, -1, 0], np.int32), good[2]), good[:2] + (np.array([1, 0, 1], np.float32),),
            good[:2] + (np.array([1, 1.5, 1], np.float32),)]
    steps = C.c_int32(0)
    for ctl in bads + [good]:
        c = _controls_struct(ctl)
        rc = eng.L.mmt_decode_controlled(eng.h, C.byref(a), 0, -1, C.byref(c), tok.data_ptr(), pr.data_ptr(), None, C.byref(steps),
                                         None, eng._stream())
        if ctl is good:
            assert rc == 0, eng.L.mmt_last_error()
        else:
            assert rc != 0 and eng.L.mmt_last_error()
        x = torch.randn(6, 128, device="cuda")
        rc = eng.L.mmt_sample_controlled(eng.h, x.data_ptr(), None, 6, 2, C.byref(c), 0, 1, 0, 1, 0, 0, 0, 0, 0, tok.data_ptr(), None,
                                         None, None, eng._stream())
        assert (rc == 0) == (ctl is good)
    g = eng._decode_args(memory, bias, 2, 4, 1.0, _lib.SAMPLE_GREEDY, False, "fp32")[0]
    assert eng.L.mmt_decode_controlled(eng.h, C.byref(g), 0, -1, C.byref(_controls_struct(good)), tok.data_ptr(), pr.data_ptr(), None,
                                       C.byref(steps), None, eng._stream()) != 0
    torch.cuda.synchronize()
