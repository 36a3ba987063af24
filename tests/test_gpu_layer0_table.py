"""Decoder layer 0 on the position x token table (large bf16 waves): bit-identical to the paged layer 0.

Layer 0's input at position t is E_tok[tok] + E_pos[t], so its Q and K | V rows depend on (t, tok) alone; the un-fused bf16
step with token-major pages reads them from a table built once per engine instead of projecting, appending and re-reading
them through the paged cache (DESIGN.md section 4.6).  The table rows come from the same bf16 input rows, projection,
bias add and rounding as the cache rows, and the attention arithmetic is the same lane for lane, so every case compares an
engine created with MMT_NO_L0_TABLE=1 (the paged layer 0) with a default one BITWISE: sampled ids and probabilities (one
bench-geometry wave, several waves with a short and a fused last wave, per-memory RNG streams), stop at <EOS> (compacted
waves: ids, probabilities, lengths, rows per position) and teacher-forced logits of all 128 positions.  Both weight sets:
the trained-like one has non-zero in_proj biases, which the table bakes in."""
import gc

import pytest
import torch

from test_gpu_trained_weights import engine_with

pytestmark = pytest.mark.gpu

MODE = "1H_13C_HSQC_COSY_IR_MF_MW"
EOS = 2
WEIGHTS = ["init", "trained"]
_E = {}


def engines(weights, **env):
    """(default engine, MMT_NO_L0_TABLE=1 engine) on the weight set and knobs; one pair alive at a time (an engine keeps the
    arena of the largest wave it ran, ~50 GB for the bench wave)."""
    key = (weights, tuple(sorted(env.items())))
    if _E.get("key") != key:
        _E.clear()
        gc.collect()
        torch.cuda.empty_cache()
        _E["pair"] = (engine_with(weights, **env), engine_with(weights, MMT_NO_L0_TABLE=1, **env))
        _E["key"] = key
    return _E["pair"]


@pytest.fixture(autouse=True, scope="module")
def _release_engines():
    yield
    _E.clear()
    gc.collect()
    if torch.cuda.is_available():
        torch.cuda.empty_cache()


def inputs(eng, Bm, seed):
    from multimodalspectraltransformer_b200 import synthetic
    data = {k: v.cuda() for k, v in synthetic.make_spectra(Bm, seed=seed).items()}
    memory, _, kb, *_ = eng.encode(data, MODE, "bf16")
    return memory, kb


def check_decode(weights, Bm, K, seed, per_memory_rng=False, **env):
    eng, ref = engines(weights, **env)
    memory, kb = inputs(eng, Bm, seed)
    kw = dict(n_cand=K, max_len=128, temperature=1.0, sampling="multinomial", precision="bf16", seed=77, offset=8,
              per_memory_rng=per_memory_rng)
    l0, r0 = eng.launch_count(), ref.launch_count()
    tok, pr, steps = eng.decode(memory, kb, **kw)
    rtok, rpr, rsteps = ref.decode(memory, kb, **kw)
    # the table path ran: no layer-0 projection launch per position of an un-fused wave
    assert eng.launch_count() - l0 < ref.launch_count() - r0
    assert steps == rsteps
    assert torch.equal(tok, rtok)
    assert torch.equal(pr, rpr)
    # the ids are not degenerate: position 1 alone takes many tokens, so the table rows read differ between sequences
    assert len(torch.unique(tok[0])) >= 10
    return tok


@pytest.mark.parametrize("weights", WEIGHTS)
def test_bench_geometry_one_wave(weights):
    """1024 spectra x 128 candidates x 128 tokens: one wave of 131,072 sequences, multinomial."""
    check_decode(weights, 1024, 128, 3101)


@pytest.mark.parametrize("weights", WEIGHTS)
def test_several_waves_short_and_fused_last(weights):
    """Waves of 128 spectra (16,384 sequences): 128 + 128 + 8 spectra -- the last wave (1,024 sequences) takes the fused
    small-wave step with its paged layer 0, so the run plans layer 0's pages next to the table path."""
    check_decode(weights, 264, 128, 3102, MMT_MAX_WAVE_SEQS="16384")


@pytest.mark.parametrize("weights", WEIGHTS)
def test_several_waves_all_unfused(weights):
    """Waves of 40 spectra x 100 candidates with a short last one (40 + 40 + 30): no fused wave, no layer-0 pages."""
    check_decode(weights, 110, 100, 3103, MMT_MAX_WAVE_SEQS="4000")


@pytest.mark.parametrize("weights", WEIGHTS)
def test_per_memory_rng(weights):
    check_decode(weights, 256, 128, 3104, per_memory_rng=True)


@pytest.mark.parametrize("weights", WEIGHTS)
def test_two_term_projection(weights):
    """MMT_DEC_PROJ_TWO_TERM=1: the step's projections use both terms of the bf16 weight split, so must the table's."""
    check_decode(weights, 256, 128, 3107, MMT_DEC_PROJ_TWO_TERM="1")


@pytest.mark.parametrize("weights", WEIGHTS)
@pytest.mark.parametrize("per_memory_rng", [False, True])
def test_stop_at_eos(weights, per_memory_rng):
    """Stop at <EOS>: the wave is compacted (row n is sequence orig[n]) at 8-position group boundaries."""
    eng, ref = engines(weights)
    memory, kb = inputs(eng, 300, 3105)
    kw = dict(eos=EOS, n_cand=100, max_len=128, temperature=1.0, sampling="multinomial", precision="bf16", seed=5, offset=0,
              per_memory_rng=per_memory_rng)
    tok, pr, steps, L, rows = eng.decode_until_eos(memory, kb, **kw)
    rtok, rpr, rsteps, rL, rrows = ref.decode_until_eos(memory, kb, **kw)
    assert steps == rsteps
    assert torch.equal(L, rL) and torch.equal(rows, rrows)
    assert torch.equal(tok, rtok) and torch.equal(pr, rpr)
    # compaction happened: fewer rows at the end than at the start, and sequences of many lengths
    assert int(rows[steps - 1]) < int(rows[0])
    assert len(torch.unique(L)) >= 10


@pytest.mark.parametrize("weights", WEIGHTS)
def test_teacher_forced_logits(weights):
    """All 128 positions of the un-fused step (32 x 128 = 4,096 sequences), forced inputs with every candidate distinct:
    the trg path of decode_embed resolves the tokens the history records; ids >= vocab (clamped to 0) included."""
    eng, ref = engines(weights)
    Bm, K, T = 32, 128, 128
    memory, kb = inputs(eng, Bm, 3106)
    g = torch.Generator().manual_seed(3106)
    trg = torch.randint(0, 43, (T, Bm * K), generator=g)
    trg[0] = 3
    trg[5, ::7] = 50
    trg = trg.cuda()
    a = eng.teacher_forced(memory, kb, trg, n_cand=K, precision="bf16")
    b = ref.teacher_forced(memory, kb, trg, n_cand=K, precision="bf16")
    assert torch.isfinite(a).all()
    assert torch.equal(a, b)
