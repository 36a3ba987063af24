"""Stop at <EOS> (``stop_at_eos=True``, ``mmt_decode_until_eos``): a sequence stops being computed once it has emitted
<EOS>, and large waves drop finished rows at 8-position group boundaries.

Everything is compared with the plain call (same arguments, same generator state): ids and probabilities bit-identical
up to and including each sequence's first <EOS>, <PAD> / 0.0 after it, the lengths equal to mmt_first_eos of the plain
ids, the generator advanced by the same amount.  Each case asserts the length spread it relies on, so it cannot pass
with sequences that all finish at once or never.  ``rows`` (the decode-step rows computed per position) shows that the
retirement happens.
"""
import pytest
import torch

STOI = {"<PAD>": 0, "<UNK>": 1, "<EOS>": 2, "<SOS>": 3, "<MASK>": 4}
ITOS = {str(i): c for i, c in enumerate(["<PAD>", "<UNK>", "<EOS>", "<SOS>", "<MASK>", "C", "c", "O", "N", "(", ")", "=",
                                          "1", "2", "3", "[", "]", "Cl", "l", "Br", "r", "F", "S", "#", "@", "H", "+", "-",
                                          "n", "o", "s", "/", "\\", "4", "5", "6", "P", "I", "B", "%", "Si", "Se", "."])}
EOS = 2
GROUP = 8
_S = {}

gpu = pytest.mark.gpu


def setup():
    if "M" not in _S:
        import multimodalspectraltransformer_b200 as M
        torch.manual_seed(0)
        _S.update(M=M, model=M.MultimodalTransformer(M.default_config(device="cuda")).eval(), raised={})
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


def raised_model(delta):
    """The bench weights with fc_out.bias[<EOS>] raised by ``delta`` (greedy sequences then end too)."""
    s = setup()
    if delta not in s["raised"]:
        torch.manual_seed(0)
        m = s["M"].MultimodalTransformer(cfg_for()).eval()
        with torch.no_grad():
            m.fc_out.bias[EOS] += delta
        s["raised"][delta] = m
    return s["raised"][delta]


def greedy_model():
    """The smallest raise (of a few) under which greedy sequences of the test spectra both end at spread positions and
    run to max_len."""
    s = setup()
    if "greedy" not in s:
        for delta in (0.25, 0.5, 0.75, 1.0, 1.25, 1.5, 2.0):
            m = raised_model(delta)
            eng, memory, bias = inputs(m, 24, "fp32", 12)
            tok, _, _ = eng.decode(memory, bias, n_cand=1, max_len=128, sampling="greedy", precision="fp32")
            L = first_eos(tok)
            if len(torch.unique(L)) >= 4 and bool((L == 128).any()):
                s["greedy"] = m
                break
        else:
            raise AssertionError("no raise of fc_out.bias[<EOS>] spreads the greedy lengths")
    return s["greedy"]


def model_with(monkeypatch, **env):
    from multimodalspectraltransformer_b200.engine import engine_for
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    torch.manual_seed(0)
    m = setup()["M"].MultimodalTransformer(cfg_for()).eval()
    engine_for(m, cfg_for())
    for k in env:
        monkeypatch.delenv(k)
    return m


def first_eos(tok):
    T = tok.shape[0]
    hit = tok == EOS
    return torch.where(hit.any(0), hit.int().argmax(0), torch.full_like(hit[0], T, dtype=torch.long))


def inputs(model, B, prec, seed):
    from multimodalspectraltransformer_b200 import synthetic
    from multimodalspectraltransformer_b200.engine import engine_for
    from multimodalspectraltransformer_b200.generate import _mask_to_bias
    cfg = cfg_for(precision=prec)
    memory, mask, *_ = setup()["M"].run_model(model, synthetic.make_spectra(B, seed=seed), cfg)
    return engine_for(model, cfg), memory, _mask_to_bias(mask)


def check_against_plain(eng, memory, bias, *, k, T, prec, sampling, per_memory_rng=False, spread=30, large=False):
    """One plain call and one retiring call on the same generator state; returns (lengths, rows)."""
    kw = dict(n_cand=k, max_len=T, temperature=1.0, sampling=sampling, precision=prec, seed=1234, offset=4 * 17,
              per_memory_rng=per_memory_rng)
    ptok, ppr, _ = eng.decode(memory, bias, **kw)
    tok, pr, steps, L, rows = eng.decode_until_eos(memory, bias, eos=EOS, **kw)
    Lref = first_eos(ptok)
    assert torch.equal(L.long(), Lref)
    # the spread this case relies on
    assert len(torch.unique(Lref)) >= spread, torch.unique(Lref)
    assert bool((Lref < T).any()) and bool((Lref == T).any())
    if spread >= 30:
        assert bool((Lref == 0).any())
    pos = torch.arange(T, device=ptok.device)[:, None]
    keep = pos <= Lref[None]
    assert torch.equal(tok[keep], ptok[keep])
    assert torch.equal(pr[keep], ppr[keep])
    assert bool((tok[~keep] == 0).all()) and bool((pr[~keep] == 0).all())
    assert steps == (T if bool((Lref == T).any()) else int(Lref.max()) + 1)
    # retirement: rows never below the sequences still live, never rising; compacted large waves follow the polls
    live = (pos <= Lref[None]).sum(1).cpu()
    assert bool((rows[:steps] >= live[:steps]).all())
    assert bool((rows[1:] <= rows[:-1]).all())
    if large:
        for t in range(2 * GROUP, T):
            tp = GROUP * (t // GROUP - 1) - 1            # end of the group polled when t's group was enqueued
            assert rows[t] * 7 <= live[tp] * 8, (t, int(rows[t]), int(live[tp]))
    return Lref, rows


@gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_small_fused_wave_multinomial(prec):
    eng, memory, bias = inputs(setup()["model"], 24, prec, 11)
    check_against_plain(eng, memory, bias, k=16, T=128, prec=prec, sampling="multinomial")


@gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_small_fused_wave_greedy_raised_eos(prec):
    """Greedy candidates of one spectrum are identical: the spread is over the 24 spectra."""
    eng, memory, bias = inputs(greedy_model(), 24, prec, 12)
    check_against_plain(eng, memory, bias, k=16, T=128, prec=prec, sampling="greedy", spread=3)


@gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("per_memory_rng", [False, True])
def test_300x100_crosses_variant_boundaries(prec, per_memory_rng):
    """30,000 rows retire through 24,576 (chained projection), 8,192 (sampler rows per warp) and 2,048 (FFN prologue /
    fused step) rows while keeping the variants of the starting size."""
    eng, memory, bias = inputs(setup()["model"], 300, prec, 13)
    L, rows = check_against_plain(eng, memory, bias, k=100, T=128, prec=prec, sampling="multinomial",
                                  per_memory_rng=per_memory_rng, large=True)
    assert int(rows[-1]) < 2048 < 8192 < 24576 < int(rows[0])


@gpu
@pytest.mark.parametrize("per_memory_rng", [False, True])
def test_bench_geometry_one_wave(per_memory_rng):
    eng, memory, bias = inputs(setup()["model"], 1024, "bf16", 3003)
    N, T = 1024 * 128, 128
    L, rows = check_against_plain(eng, memory, bias, k=128, T=T, prec="bf16", sampling="multinomial",
                                  per_memory_rng=per_memory_rng, large=True)
    assert int(rows.sum()) <= 0.5 * N * T


@gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_several_waves(monkeypatch, prec):
    m = model_with(monkeypatch, MMT_MAX_WAVE_SEQS="4096")
    eng, memory, bias = inputs(m, 96, prec, 14)
    check_against_plain(eng, memory, bias, k=128, T=128, prec=prec, sampling="multinomial")


@gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_simt_cross_attention_path(prec):
    """n_cand < 8: the SIMT cross attention reads each compacted row's memory column from the row map."""
    eng, memory, bias = inputs(setup()["model"], 3000, prec, 15)
    check_against_plain(eng, memory, bias, k=3, T=128, prec=prec, sampling="multinomial", large=True)


@gpu
@pytest.mark.parametrize("B,k", [(64, 16), (300, 16)])
def test_stops_when_all_finished(B, k):
    """fc_out.bias[<EOS>] + 8: every sequence ends within a few positions; the generator still advances in full."""
    s = setup()
    M, model = s["M"], raised_model(8.0)
    cfg = cfg_for(precision="bf16")
    from multimodalspectraltransformer_b200 import synthetic
    memory, mask, *_ = M.run_model(model, synthetic.make_spectra(B, seed=16), cfg)
    eng, _, bias = inputs(model, B, "bf16", 16)
    kw = dict(n_cand=k, max_len=128, sampling="multinomial", precision="bf16", seed=5, offset=0)
    ptok, ppr, _ = eng.decode(memory, bias, **kw)
    tok, pr, steps, L, rows = eng.decode_until_eos(memory, bias, eos=EOS, **kw)
    Lref = first_eos(ptok)
    assert int(Lref.max()) < 16 and steps == int(Lref.max()) + 1 < 128
    assert int(rows[steps + 2 * GROUP:].sum()) == 0
    keep = torch.arange(128, device=tok.device)[:, None] <= Lref[None]
    assert torch.equal(tok[keep], ptok[keep]) and torch.equal(pr[keep], ppr[keep]) and bool((tok[~keep] == 0).all())
    gen = torch.cuda.default_generators[torch.cuda.current_device()]
    torch.manual_seed(77)
    o0 = gen.get_offset()
    t1, _ = M.multinomial_sequence_multi(model, memory, mask, STOI, cfg, n_candidates=k)
    o1 = gen.get_offset()
    torch.manual_seed(77)
    t2, _ = M.multinomial_sequence_multi(model, memory, mask, STOI, cfg, n_candidates=k, stop_at_eos=True)
    assert gen.get_offset() == o1 > o0
    assert t1.shape == t2.shape


@gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_python_surface(prec):
    s = setup()
    M = s["M"]
    from multimodalspectraltransformer_b200 import synthetic
    cfg = cfg_for(precision=prec)
    model, k, B = s["model"], 16, 40
    memory, mask, *_ = M.run_model(model, synthetic.make_spectra(B, seed=17), cfg)
    gen = torch.cuda.default_generators[torch.cuda.current_device()]

    def both(fn, *args, **kw):
        torch.manual_seed(9)
        a = fn(*args, **kw)
        off = gen.get_offset()
        torch.manual_seed(9)
        b = fn(*args, stop_at_eos=True, **kw)
        assert gen.get_offset() == off
        for x, y in zip(a, b):
            assert x.shape == y.shape
        return a, b

    for fn in (M.multinomial_sequence_multi, M.generate.multinomial_sequence_multi_2):
        (ta, pa), (tb, pb) = both(fn, model, memory, mask, STOI, cfg, n_candidates=k, per_memory_rng=True)
        assert M.tensor_to_smiles(ta, ITOS) == M.tensor_to_smiles(tb, ITOS)
        (sa, qa), (sb, qb) = M.tensor_to_smiles_and_prob_2(ta, pa, ITOS), M.tensor_to_smiles_and_prob_2(tb, pb, ITOS)
        assert sa == sb and all(torch.equal(x, y) for x, y in zip(qa, qb))
        da, db = M.distinct_smiles(ta, ITOS, k), M.distinct_smiles(tb, ITOS, k)
        assert [[(d.smiles, d.index, d.count) for d in c] for c in da] == [[(d.smiles, d.index, d.count) for d in c] for c in db]
    (ta, pa), (tb, pb) = both(M.multinomial_sequence, model, STOI, memory, mask, cfg, n_candidates=k)
    assert M.tensor_to_smiles(ta, ITOS) == M.tensor_to_smiles(tb, ITOS)
    gm = greedy_model()
    gmem, gmask, *_ = M.run_model(gm, synthetic.make_spectra(B, seed=17), cfg)
    for fn in (M.greedy_sequence, M.greedy_sequence_2):
        ta, pa = fn(gm, STOI, ITOS, gmem, gmask, cfg)
        tb, pb = fn(gm, STOI, ITOS, gmem, gmask, cfg, stop_at_eos=True)
        assert tb.shape[0] <= ta.shape[0] and tb.shape[1] == ta.shape[1]
        assert M.tensor_to_smiles(ta[:tb.shape[0]], ITOS) == M.tensor_to_smiles(tb, ITOS)


@gpu
@pytest.mark.parametrize("per_memory_rng", [False, True])
def test_shards_equal_the_whole_call(per_memory_rng):
    s = setup()
    M = s["M"]
    from multimodalspectraltransformer_b200 import synthetic
    cfg = cfg_for(precision="bf16")
    model, k, B = s["model"], 32, 200
    memory, mask, *_ = M.run_model(model, synthetic.make_spectra(B, seed=18), cfg)
    torch.manual_seed(3)
    whole, wp = M.multinomial_sequence_multi(model, memory, mask, STOI, cfg, n_candidates=k, per_memory_rng=per_memory_rng,
                                             stop_at_eos=True)
    parts = []
    for lo, hi in ((0, 90), (90, B)):      # both shards, like the whole call, above the fused-step size
        torch.manual_seed(3)
        parts.append(M.multinomial_sequence_multi(model, memory[:, lo:hi], mask[lo:hi], STOI, cfg, n_candidates=k,
                                                  seq_index_base=lo * k, n_total=B * k, per_memory_rng=per_memory_rng,
                                                  stop_at_eos=True))
    assert torch.equal(whole, torch.cat([p[0] for p in parts], dim=1))
    assert torch.equal(wp, torch.cat([p[1] for p in parts], dim=1))


@gpu
def test_errors():
    s = setup()
    eng, memory, bias = inputs(s["model"], 4, "bf16", 19)
    for eos in (-1, 43):
        with pytest.raises(RuntimeError):
            eng.decode_until_eos(memory, bias, eos=eos, n_cand=4, max_len=8, sampling="multinomial", precision="bf16")
    from multimodalspectraltransformer_b200 import _lib
    import ctypes as C
    a, keep = eng._decode_args(memory, bias, 4, 8, 1.0, _lib.SAMPLE_GREEDY, False, "bf16")
    tok = torch.empty(8, 16, dtype=torch.int64, device="cuda")
    ln = torch.empty(16, dtype=torch.int32, device="cuda")
    assert eng.L.mmt_decode_until_eos(eng.h, C.byref(a), 1, EOS, tok.data_ptr(), None, ln.data_ptr(), None, None,
                                      eng._stream()) != 0


def test_stoi_without_eos_is_rejected():
    from multimodalspectraltransformer_b200 import generate as G
    stoi = {k: v for k, v in STOI.items() if k != "<EOS>"}
    with pytest.raises(ValueError):
        G.greedy_sequence(None, stoi, ITOS, None, None, None, stop_at_eos=True)
    with pytest.raises(ValueError):
        G.multinomial_sequence_multi(None, None, None, stoi, None, stop_at_eos=True)
