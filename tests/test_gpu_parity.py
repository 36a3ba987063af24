"""GPU parity tests (run on the B200 box with -m gpu): the CUDA engine, called through
the C ABI, against (a) the golden vectors produced by the reference's own code and
(b) the oracle restatement on the same seeded inputs."""
import json

import numpy as np
import pytest
import torch

from golden_util import CASES, load_case

pytestmark = pytest.mark.gpu

_S = {}
STOI = {"<PAD>": 0, "<UNK>": 1, "<EOS>": 2, "<SOS>": 3, "<MASK>": 4}


def setup():
    if "model" not in _S:
        import multimodalspectraltransformer_b200 as M
        from oracle import mmt_oracle as O
        cfg = M.default_config(device="cuda")
        torch.manual_seed(0)
        model = M.MultimodalTransformer(cfg)
        model.eval()
        _S.update(M=M, O=O, cfg=cfg, model=model, P=O.random_init_state_dict(O.default_config(), seed=0))
        from multimodalspectraltransformer_b200.engine import engine_for
        _S["eng"] = engine_for(model, cfg)
    return _S


def cfg_for(case=None, **over):
    s = setup()
    c = s["M"].default_config(device="cuda", **over)
    if case is not None:
        c.training_mode = case["mode"]
    return c


# --------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("M,N,K,act", [(5, 128, 128, 0), (256, 384, 128, 0), (300, 2048, 128, 1), (33, 128, 2048, 0),
                                        (7, 128, 1000, 1), (4097, 384, 128, 0), (2500, 128, 2048, 0), (1500, 512, 128, 0)])
def test_linear_fp32(M, N, K, act):
    s = setup()
    g = torch.Generator().manual_seed(M * 7 + N)
    A = torch.randn(M, K, generator=g).cuda()
    W = (torch.randn(N, K, generator=g) / K ** 0.5).cuda()
    b = torch.randn(N, generator=g).cuda()
    out = s["eng"].linear(A, W, b, act=act)
    ref = torch.nn.functional.linear(A.double(), W.double(), b.double())
    if act:
        ref = torch.relu(ref)
    torch.testing.assert_close(out.double(), ref, atol=2e-5, rtol=1e-5)


def test_sampler_greedy_matches_torch():
    """Logits against the fp64 product, ids and probabilities: N = 1000 takes the one-row-per-warp form, N >= 8192 the
    four-rows-per-warp form (8193 and 75,779: a tail that is not a multiple of the 32 rows of a CTA pass).  At N = 1000
    the ids equal torch's fp32 argmax; at all sizes they equal the fp64 argmax wherever its top-2 margin exceeds a few
    fp32 ulps."""
    s = setup()
    W, b = s["model"].fc_out.weight.detach().cuda(), s["model"].fc_out.bias.detach().cuda()
    for N in (1000, 8192, 8193, 75779):
        g = torch.Generator().manual_seed(5 + N)
        x = torch.randn(N, 128, generator=g).cuda()
        ref = torch.nn.functional.linear(x.double(), W.double(), b.double())
        top2 = torch.topk(ref, 2, dim=1).values
        clear = (top2[:, 0] - top2[:, 1]) > 1e-5
        for T in (1.0, 0.7, 1.3):
            tok, pr, lg = s["eng"].sample(x, temperature=T, sampling="greedy", want_logits=True)
            torch.testing.assert_close(lg.double(), ref, atol=2e-6, rtol=1e-5)
            assert torch.equal(tok[clear], ref.argmax(dim=1)[clear]), N
            p = torch.softmax(ref / T, dim=1)
            torch.testing.assert_close(pr.double(), p.gather(1, tok[:, None])[:, 0], atol=1e-6, rtol=1e-5)
            if N == 1000:
                assert torch.equal(tok, torch.argmax(torch.softmax(torch.nn.functional.linear(x, W, b) / T, dim=1), dim=1))


@pytest.mark.parametrize("N", [128, 5000, 20000, 40000])
def test_sampler_multinomial_reproduces_torch_philox_stream(N):
    """Same seed/offset -> same ids as torch.multinomial on this device (SURVEY.md appendix D).
    N = 20000 exercises the .y/.z/.w components, N = 40000 the second loop iteration."""
    s = setup()
    g = torch.Generator().manual_seed(N)
    x = torch.randn(N, 128, generator=g).cuda()
    W, b = s["model"].fc_out.weight.detach().cuda(), s["model"].fc_out.bias.detach().cuda()
    p = torch.softmax(torch.nn.functional.linear(x, W, b) / 1.0, dim=1)
    gen = torch.cuda.default_generators[torch.cuda.current_device()]
    torch.manual_seed(777)
    torch.empty(10, device="cuda").uniform_()           # move the offset off zero
    seed, off = gen.initial_seed(), gen.get_offset()
    want = torch.multinomial(p, 1)[:, 0]
    inc = gen.get_offset() - off
    assert inc == s["eng"].philox_increment(N)
    tok, pr, _ = s["eng"].sample(x, sampling="multinomial", seed=seed, offset=off)
    # (a) the RNG stream alone: torch's own probabilities through our Philox mapping -> torch's ids, all of them
    assert torch.equal(s["eng"].sample_probs(p, seed=seed, offset=off), want)
    # (b) the fused kernel computes fc_out + softmax itself (fp32 FMA order differs from cuBLAS by an ulp or two): every id
    # that differs from torch's must be a near-tie of p / q under torch's OWN p and q, never a different draw
    agree = (tok == want).float().mean().item()
    assert agree > 0.9995, agree
    bad = torch.nonzero(tok != want)[:, 0]
    if bad.numel():
        q = s["eng"].exponential(N * 43, seed=seed, offset=off).view(N, 43)
        r = (p / q)[bad]
        r_want, r_mine = r.gather(1, want[bad, None])[:, 0], r.gather(1, tok[bad, None])[:, 0]
        assert bool(((r_want - r_mine).abs() <= 1e-5 * r_want).all()), (bad.tolist(), r_want.tolist(), r_mine.tolist())
    # shard invariance: rows [lo,hi) sampled alone, placed inside the N-row call
    lo, hi = N // 3, N // 3 + 50
    tok_s, _, _ = s["eng"].sample(x[lo:hi], sampling="multinomial", seed=seed, offset=off, seq_index_base=lo, n_total=N)
    assert torch.equal(tok_s, tok[lo:hi])


@pytest.mark.parametrize("numel", [43 * 128, 43 * 5000, 43 * 20000, 43 * 40000, 43 * 131072, 1000003])
def test_exponential_variates_bit_equal_torch(numel):
    """The Exp(1) variates behind torch.multinomial (SURVEY.md App. D): bit equality with exponential_() on this device
    in all launch-geometry regimes (single float4 component; .y/.z/.w; second loop iteration; config 3's 131,072 x 43
    with its offset increment of 20), at a non-zero generator offset, plus a window placed inside the big tensor."""
    s = setup()
    gen = torch.cuda.default_generators[torch.cuda.current_device()]
    torch.manual_seed(31337)
    torch.empty(7, device="cuda").normal_()             # offset off zero
    seed, off = gen.initial_seed(), gen.get_offset()
    want = torch.empty(numel, device="cuda").exponential_(1)
    assert gen.get_offset() - off == s["eng"].L.mmt_philox_increment(numel, s["eng"].sm_count, s["eng"].max_threads_per_sm)
    got = s["eng"].exponential(numel, seed=seed, offset=off)
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))
    lo = numel // 2 + 3
    win = s["eng"].exponential(1000, seed=seed, offset=off, elem_base=lo, numel_total=numel)
    assert torch.equal(win, want[lo:lo + 1000])


def test_philox_numpy_restatement_matches_device():
    """oracle.cuda_exponential_like (numpy) == torch's exponential_ on this device: same Philox
    words, same offset increment; values agree to the error of the device's fast __logf
    (lg2.approx, a few ulp), which numpy cannot reproduce bit for bit."""
    s = setup()
    props = torch.cuda.get_device_properties(0)
    for numel in (43 * 128, 400000, 1300000):
        torch.manual_seed(4242)
        gen = torch.cuda.default_generators[torch.cuda.current_device()]
        seed, off = gen.initial_seed(), gen.get_offset()
        q = torch.empty(numel, device="cuda").exponential_(1).cpu().numpy()
        mine, inc = s["O"].cuda_exponential_like(numel, seed, off, props.multi_processor_count, props.max_threads_per_multi_processor)
        assert gen.get_offset() - off == inc
        assert np.max(np.abs(q - mine)) < 2e-6 and np.max(np.abs(q - mine) / np.maximum(np.abs(q), 1e-3)) < 1e-3


# --------------------------------------------------------------------------- encoder
@pytest.mark.parametrize("name", CASES)
def test_encoder_vs_reference_golden(name):
    s = setup()
    case, data, z = load_case(name)
    cfg = cfg_for(case)
    memory, mask, trg, fp, hs, co = s["M"].run_model(s["model"], data, cfg)
    ref_mask = torch.from_numpy(z["mask"])
    assert mask.dtype == ref_mask.dtype and torch.equal(mask.cpu(), ref_mask)
    stride = int(z["memory_stride"])
    np.testing.assert_allclose(memory[::stride].cpu().numpy(), z["memory_sample"], atol=5e-5, rtol=0)
    np.testing.assert_allclose(memory.double().sum(dim=(0, 2)).cpu().numpy(), z["memory_sum"], atol=5e-3)
    np.testing.assert_allclose(fp.cpu().numpy(), z["fingerprint"], atol=5e-5, rtol=0)
    assert torch.equal(trg.cpu(), data["trg_enc_SMI"])
    # forward(trg=None) returns the same memory + embedding_src (models_MMT_v15_4.py:952-953)
    s["model"].config = cfg
    args = [data[k] for k in ("src_1H", "mask_1H", "src_13C", "mask_13C", "src_HSQC", "mask_HSQC", "src_COSY", "mask_COSY",
                              "src_IR", "mask_IR", "src_MF", "mask_MF", "src_MS", "mask_MS", "trg_MW")]
    mem2, emb, mask2, fp2 = s["model"](*args)
    assert torch.equal(mem2, memory) and torch.equal(fp2, fp) and torch.equal(mask2, mask)
    np.testing.assert_allclose(emb.double().sum(dim=(0, 2)).cpu().numpy(), z["embedding_src_sum"], atol=1e-3)


def test_repeated_encode_is_served_from_the_last_one_only_when_inputs_are_bit_identical(monkeypatch):
    """SURVEY 8 f4: CLIP's forward(trg=None) on the batch run_model has just encoded costs one comparison kernel, not a
    second encode; any change of the inputs (new tensors or in-place), of the mode, or of the returned outputs misses."""
    s = setup()
    from multimodalspectraltransformer_b200.engine import Engine, engine_for
    case, data, z = load_case("full_b5")
    cfg = cfg_for(case)
    model = s["model"]
    model.config = cfg
    eng = engine_for(model, cfg)
    keys = ("src_1H", "mask_1H", "src_13C", "mask_13C", "src_HSQC", "mask_HSQC", "src_COSY", "mask_COSY",
            "src_IR", "mask_IR", "src_MF", "mask_MF", "src_MS", "mask_MS", "trg_MW")
    memory, mask, _, fp, _, _ = s["M"].run_model(model, data, cfg)
    h0, l0 = eng.encode_cache_hits, eng.launch_count()
    mem2, emb, mask2, fp2 = model(*[data[k] for k in keys])             # host tensors again -> fresh device copies
    assert eng.encode_cache_hits == h0 + 1 and eng.launch_count() - l0 <= 3
    assert torch.equal(mem2, memory) and torch.equal(fp2, fp) and torch.equal(mask2, mask) and mem2.data_ptr() != memory.data_ptr()
    monkeypatch.setenv("MMT_NO_ENCODE_CACHE", "1")
    fresh = Engine(model.state_dict(), cfg, eng.device).encode(data, case["mode"], "fp32", True)
    monkeypatch.delenv("MMT_NO_ENCODE_CACHE")
    assert torch.equal(fresh[0], mem2) and torch.equal(fresh[5], emb) and torch.equal(fresh[3], fp2)
    mem3, emb3, _, _ = model(*[data[k] for k in keys])                   # second hit: embedding_src now remembered too
    assert eng.encode_cache_hits == h0 + 2 and torch.equal(emb3, emb)
    # one peak moved -> miss, different memory
    d2 = {k: v.clone() for k, v in data.items()}
    d2["src_13C"][1, 0] += 0.25
    mem4, _, _, _ = model(*[d2[k] for k in keys])
    assert eng.encode_cache_hits == h0 + 2 and not torch.equal(mem4, memory)
    # device-resident inputs changed in place -> miss
    dd = {k: v.cuda() for k, v in data.items()}
    m5 = model(*[dd[k] for k in keys])[0]
    assert torch.equal(m5, memory)
    hits = eng.encode_cache_hits
    m5b = model(*[dd[k] for k in keys])[0]
    assert eng.encode_cache_hits == hits + 1 and torch.equal(m5b, memory)
    dd["src_1H"][0, 0, 0] += 0.5
    m6 = model(*[dd[k] for k in keys])[0]
    assert eng.encode_cache_hits == hits + 1 and not torch.equal(m6, memory)
    # the caller wrote into the returned memory -> the remembered outputs are stale -> miss
    mem7, mask7, *_ = s["M"].run_model(model, data, cfg)
    mem7.zero_()
    hits = eng.encode_cache_hits
    mem8 = model(*[data[k] for k in keys])[0]
    assert eng.encode_cache_hits == hits and torch.equal(mem8, memory)
    # another training_mode on the same data -> miss
    cfg2 = cfg_for(case)
    cfg2.training_mode = "1H_13C_HSQC_COSY_MF_MW"
    model.config = cfg2
    hits = eng.encode_cache_hits
    mem9 = model(*[data[k] for k in keys])[0]
    assert eng.encode_cache_hits == hits and mem9.shape[0] != 0
    model.config = cfg


# --------------------------------------------------------------------------- decoder
@pytest.mark.parametrize("name", CASES)
def test_teacher_forced_and_greedy_vs_reference_golden(name):
    s = setup()
    case, data, z = load_case(name)
    cfg = cfg_for(case)
    memory, mask, *_ = s["M"].run_model(s["model"], data, cfg)
    logits = s["M"].teacher_forced_logits(s["model"], memory, mask, torch.from_numpy(z["tf_tokens"]), cfg)
    np.testing.assert_allclose(logits.cpu().numpy(), z["tf_logits"], atol=1e-4, rtol=0)
    cfg.max_len = case["glen"]
    tok, pr = s["M"].greedy_sequence(s["model"], STOI, None, memory, mask, cfg)
    assert tok.dtype == torch.int64 and tuple(tok.shape) == z["greedy_tokens"].shape
    assert np.array_equal(tok.cpu().numpy(), z["greedy_tokens"])          # bit-exact ids (fp32 check mode)
    np.testing.assert_allclose(pr.cpu().numpy(), z["greedy_probs"], atol=2e-5, rtol=0)
    cfg.max_len, cfg.temperature = 12, 1.3
    tok, pr = s["M"].greedy_sequence(s["model"], STOI, None, memory, mask, cfg)
    assert np.array_equal(tok.cpu().numpy(), z["greedy_T13_tokens"])
    np.testing.assert_allclose(pr.cpu().numpy(), z["greedy_T13_probs"], atol=2e-5, rtol=0)
    # forward(..., trg): 4-tuple with logits first (models_MMT_v15_4.py:976)
    s["model"].config = cfg_for(case)
    args = [data[k] for k in ("src_1H", "mask_1H", "src_13C", "mask_13C", "src_HSQC", "mask_HSQC", "src_COSY", "mask_COSY",
                              "src_IR", "mask_IR", "src_MF", "mask_MF", "src_MS", "mask_MS", "trg_MW")]
    out, fp, mem, msk = s["model"](*args, torch.from_numpy(z["tf_tokens"]).cuda())
    np.testing.assert_allclose(out.cpu().numpy(), z["tf_logits"], atol=1e-4, rtol=0)


def test_greedy_b24_full_length_vs_oracle():
    """24 spectra x 128 steps: ids identical to the CPU restatement (itself pinned to the reference)."""
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    data = synthetic.make_spectra(24, seed=101)
    cfg = cfg_for()
    memory, mask, *_ = s["M"].run_model(s["model"], data, cfg)
    tok, pr = s["M"].greedy_sequence(s["model"], STOI, None, memory, mask, cfg)
    O = s["O"]
    ocfg = O.default_config()
    with torch.no_grad():
        omem, omask, ofp, _ = O.encode(s["P"], data, ocfg)
        otok, opr = O.greedy_sequence(s["P"], omem, omask, ocfg)
    torch.testing.assert_close(memory.cpu(), omem, atol=5e-5, rtol=0)
    assert tuple(tok.shape) == (128, 24) and tuple(pr.shape) == (127, 24)
    assert torch.equal(tok.cpu(), otok)
    torch.testing.assert_close(pr.cpu(), opr, atol=2e-5, rtol=0)


def test_candidates_share_memory_equals_duplication():
    """n_candidates=k == the reference's tensor duplication (run_batch_gen_val_MMT_v15_4.py:93-107)."""
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    data = synthetic.make_spectra(3, seed=55)
    cfg = cfg_for(max_len=20)
    memory, mask, *_ = s["M"].run_model(s["model"], data, cfg)
    k = 4
    dup_mem = memory.repeat_interleave(k, dim=1)
    dup_mask = mask.repeat_interleave(k, dim=0)
    t1, p1 = s["M"].greedy_sequence(s["model"], STOI, None, memory, mask, cfg, n_candidates=k)
    t2, p2 = s["M"].greedy_sequence(s["model"], STOI, None, dup_mem, dup_mask, cfg)
    assert torch.equal(t1, t2) and torch.equal(p1, p2)
    torch.manual_seed(9)
    m1, q1 = s["M"].multinomial_sequence_multi(s["model"], memory, mask, STOI, cfg, n_candidates=k)
    torch.manual_seed(9)
    m2, q2 = s["M"].multinomial_sequence_multi(s["model"], dup_mem, dup_mask, STOI, cfg)
    assert torch.equal(m1, m2) and torch.equal(q1, q2)
    # duplicate_dict path: encode the k copies like the reference does
    dd = s["M"].duplicate_dict({kk: v[:1] for kk, v in data.items()}, k)
    eng = engine_for_cfg(s, cfg)
    l0 = eng.launch_count()
    mem_d, mask_d, _, fp_d, *_ = s["M"].run_model(s["model"], dd, cfg)
    one = eng.launch_count() - l0
    torch.testing.assert_close(mem_d, memory[:, :1].expand(-1, k, -1), atol=1e-6, rtol=0)
    assert tuple(mem_d.shape) == (582, k, 128) and tuple(mask_d.shape) == (k, 582) and tuple(fp_d.shape) == (k, 512)
    # the copies are encoded once (same launch count as a single spectrum), in tensor.repeat's order for B0 > 1 ...
    dd2 = s["M"].duplicate_dict({kk: v[:2] for kk, v in data.items()}, 3)
    mem2, mask2, trg2, *_ = s["M"].run_model(s["model"], dd2, cfg)
    torch.testing.assert_close(mem2, memory[:, :2].repeat(1, 3, 1), atol=1e-6, rtol=0)
    assert torch.equal(trg2.cpu(), data["trg_enc_SMI"][:2].repeat(3, 1))
    # ... unless the caller changed an entry after duplicating: then every copy is encoded as given
    dd3 = s["M"].duplicate_dict({kk: v[:1] for kk, v in data.items()}, k)
    dd3["src_13C"][2, 0] += 0.25
    l0 = eng.launch_count()
    mem3, *_ = s["M"].run_model(s["model"], dd3, cfg)
    assert eng.launch_count() - l0 >= one
    assert torch.equal(mem3[:, 0], mem3[:, 1]) and not torch.equal(mem3[:, 0], mem3[:, 2])
    dd4 = s["M"].duplicate_dict({kk: v[:1] for kk, v in data.items()}, k)
    dd4["src_IR"] = torch.zeros_like(dd4["src_IR"])
    mem4, *_ = s["M"].run_model(s["model"], dd4, cfg)
    assert not torch.allclose(mem4[:, 0], mem_d[:, 0])


def engine_for_cfg(s, cfg):
    from multimodalspectraltransformer_b200.engine import engine_for
    return engine_for(s["model"], cfg)


def test_multinomial_vs_oracle_on_device_same_seed():
    """End to end: same torch seed -> same sampled ids as the restated reference loop run with
    torch.multinomial on this GPU; generator offset advanced identically."""
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    data = synthetic.make_spectra(6, seed=77)
    cfg = cfg_for(max_len=40)
    memory, mask, *_ = s["M"].run_model(s["model"], data, cfg)
    k = 16
    O = s["O"]
    Pd = {kk: v.cuda() for kk, v in s["P"].items()}
    ocfg = O.default_config(max_len=40)
    dup_mem, dup_mask = memory.repeat_interleave(k, dim=1), mask.repeat_interleave(k, dim=0)
    gen = torch.cuda.default_generators[torch.cuda.current_device()]
    torch.manual_seed(2024)
    with torch.no_grad():
        otok, opr = O.multinomial_sequence_multi(Pd, dup_mem, dup_mask, ocfg)
    off_ref = gen.get_offset()
    torch.manual_seed(2024)
    tok, pr = s["M"].multinomial_sequence_multi(s["model"], memory, mask, STOI, cfg, n_candidates=k)
    assert gen.get_offset() == off_ref
    assert tuple(tok.shape) == (40, 96) and tuple(pr.shape) == (40, 96)
    same_seq = (tok == otok).all(dim=0).float().mean().item()
    assert (tok[0] == otok[0]).all()
    assert same_seq >= 0.95, same_seq
    ok = (tok == otok).all(dim=0)
    torch.testing.assert_close(pr[:, ok], opr[:, ok], atol=2e-5, rtol=0)
    # reference return layouts
    torch.manual_seed(2024)
    tok2, pr2 = s["M"].multinomial_sequence(s["model"], STOI, memory, mask, cfg, n_candidates=k)
    assert torch.equal(tok2, tok) and tuple(pr2.shape) == (96, 40) and torch.equal(pr2, pr.transpose(0, 1))
    torch.manual_seed(2024)
    tok3, pr3 = s["M"].multinomial_sequence_multi_2(s["model"], memory, mask, STOI, cfg, n_candidates=k)
    assert torch.equal(tok3, tok) and torch.equal(pr3, pr[1:])


def test_multinomial_shard_invariance():
    """Spectra sharded over ranks draw the unsharded run's numbers (SURVEY.md 8e)."""
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    data = synthetic.make_spectra(8, seed=31)
    cfg = cfg_for(max_len=16)
    memory, mask, *_ = s["M"].run_model(s["model"], data, cfg)
    k = 8
    torch.manual_seed(5)
    full, _ = s["M"].multinomial_sequence_multi(s["model"], memory, mask, STOI, cfg, n_candidates=k)
    parts = []
    for lo, hi in ((0, 3), (3, 8)):
        torch.manual_seed(5)
        t, _ = s["M"].multinomial_sequence_multi(s["model"], memory[:, lo:hi], mask[lo:hi], STOI, cfg, n_candidates=k,
                                                 seq_index_base=lo * k, n_total=8 * k)
        parts.append(t)
    assert torch.equal(torch.cat(parts, dim=1), full)


def test_greedy_early_exit_on_all_pad():
    """greedy_sequence stops at the first step where every sequence emits <PAD>
    (validate_generate_MMT_v15_4.py:763): force it with a fc_out bias that always picks id 0."""
    s = setup()
    import copy
    from multimodalspectraltransformer_b200 import synthetic
    model = copy.deepcopy(s["model"])
    with torch.no_grad():
        model.fc_out.bias[0] = 1e4
    data = synthetic.make_spectra(4, seed=3)
    cfg = cfg_for(max_len=40)
    memory, mask, *_ = s["M"].run_model(model, data, cfg)
    tok, pr = s["M"].greedy_sequence(model, STOI, None, memory, mask, cfg)
    assert tuple(tok.shape) == (1, 4) and tuple(pr.shape) == (0, 4) and int(tok.abs().sum()) == 0
    tok2, pr2 = s["M"].greedy_sequence_2(model, STOI, None, memory, mask, cfg)
    assert tuple(tok2.shape) == (1, 4) and tuple(pr2.shape) == (1, 4)


def test_token_pack_roundtrip():
    s = setup()
    t = torch.randint(0, 43, (128, 77), device="cuda")
    p = s["eng"].pack_tokens(t)
    assert p.dtype == torch.uint8 and torch.equal(s["eng"].unpack_tokens(p), t)
    # sequence-major form (the scheduler's all-gather payload): (T,N) i64 -> (N,T) u8 and back, ragged tile edges
    for T, N in ((128, 77), (1, 1), (33, 1000), (128, 16384 + 5)):
        t = torch.randint(0, 43, (T, N), device="cuda")
        q = s["eng"].pack_tokens_seqmajor(t)
        assert q.dtype == torch.uint8 and tuple(q.shape) == (N, T) and torch.equal(q, t.t().to(torch.uint8))
        assert torch.equal(s["eng"].unpack_tokens_seqmajor(q, N), t)
        pad = torch.cat([q, torch.zeros(7, T, dtype=torch.uint8, device="cuda")])      # a gathered buffer with padded tail rows
        assert torch.equal(s["eng"].unpack_tokens_seqmajor(pad, N), t)


def test_errors_are_loud():
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    data = synthetic.make_spectra(2, seed=1)
    cfg = cfg_for()
    memory, mask, *_ = s["M"].run_model(s["model"], data, cfg)
    bad = cfg_for(max_len=500)
    with pytest.raises(RuntimeError):
        s["M"].greedy_sequence(s["model"], STOI, None, memory, mask, bad)
    cpu_cfg = s["M"].default_config(device="cpu")
    with pytest.raises(RuntimeError):
        s["M"].run_model(s["model"], data, cpu_cfg)
    with pytest.raises(TypeError):
        s["M"].run_model(s["model"], data, cfg_for(training_mode="IR_MF_MW"))


# --------------------------------------------------------------------------- ragged encoder
def _dense_engine():
    """A second engine over the same weights with the ragged encoder disabled (MMT_DENSE_ENCODER is read at creation)."""
    import os
    s = setup()
    if "eng_dense" not in _S:
        from multimodalspectraltransformer_b200.engine import Engine
        os.environ["MMT_DENSE_ENCODER"] = "1"
        try:
            _S["eng_dense"] = Engine(s["model"].state_dict(), s["cfg"], "cuda")
        finally:
            del os.environ["MMT_DENSE_ENCODER"]
    return _S["eng_dense"]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("peaks", ["realistic", "max"])
def test_ragged_encoder_equals_dense_encoder(precision, peaks):
    """Computing each distinct token row once == running all 582 padded rows (SURVEY.md A.2): same memory, mask and
    fingerprint; padded rows of a segment are exact replicas."""
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    data = {k: v.cuda() for k, v in synthetic.make_spectra(9, seed=77, peaks=peaks).items()}
    mode = "1H_13C_HSQC_COSY_IR_MF_MW"
    mem_r, pad_r, kb_r, fp_r, avg_r, emb_r = s["eng"].encode(data, mode, precision, want_embedding_src=True)
    mem_d, pad_d, kb_d, fp_d, avg_d, emb_d = _dense_engine().encode(data, mode, precision, want_embedding_src=True)
    assert torch.equal(pad_r, pad_d) and torch.equal(kb_r, kb_d) and torch.equal(emb_r, emb_d)
    tol = 1e-5 if precision == "fp32" else 2e-5      # row-local arithmetic is position independent; allow reassociation
    torch.testing.assert_close(mem_r, mem_d, atol=tol, rtol=0)
    torch.testing.assert_close(fp_r, fp_d, atol=1e-4, rtol=0)
    # every padded peak row of a spectrum equals the first padded row of its segment, bit for bit
    m1 = data["mask_1H"][0] != 0
    if int(m1.sum()) > 1:
        rows = mem_r[:64, 0][m1]
        assert torch.equal(rows, rows[:1].expand_as(rows))


def test_ragged_encoder_falls_back_when_padding_hides_data():
    """A caller may leave non-zero data under the mask: padded rows then differ as queries, the ragged path must
    notice (device-side flag) and the dense path must produce the reference's result."""
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    host = synthetic.make_spectra(3, seed=5)
    pad = host["mask_1H"] != 0
    host["src_1H"] = host["src_1H"].clone()
    host["src_1H"][pad] = torch.rand(int(pad.sum()), 2)            # junk under the mask
    cfg = cfg_for()
    memory, mask, *_ = s["M"].run_model(s["model"], host, cfg)
    with torch.no_grad():
        omem, omask, ofp, _ = s["O"].encode(s["P"], host, s["O"].default_config())
    assert torch.equal(mask.cpu(), omask)
    np.testing.assert_allclose(memory.cpu().numpy(), omem.numpy(), atol=5e-5, rtol=0)
    rows = memory[:64, 0][pad[0].cuda()]
    assert not torch.equal(rows, rows[:1].expand_as(rows))        # the padded rows really are distinct here


# --------------------------------------------------------------------------- ids -> SMILES
def _ref_tensor_to_smiles_and_prob_2(tensor, token_prob, itos):
    """The reference's element-by-element loop (helper_functions_pl_v15_4.py:390-410), restated for the check."""
    seqs, cut = [], []
    for i in range(tensor.shape[1]):
        seq = []
        for j in range(tensor.shape[0]):
            tok = itos[str(int(tensor[j, i]))]
            if tok == "<EOS>":
                break
            seq.append(tok)
        seqs.append("".join(seq))
        cut.append(token_prob[:len(seq), i])
    return seqs, cut


def test_tensor_to_smiles_matches_reference_loop():
    s = setup()
    itos = {str(i): f"t{i}|" for i in range(43)}
    itos.update({"0": "<PAD>", "2": "<EOS>", "3": "<SOS>"})
    g = torch.Generator().manual_seed(3)
    tok = torch.randint(0, 43, (128, 300), generator=g)
    tok[:, 5] = 7                        # never emits <EOS>
    tok[0, 6] = 2                        # <EOS> first -> empty string
    pr = torch.rand(128, 300, generator=g)
    ref_s, ref_p = _ref_tensor_to_smiles_and_prob_2(tok, pr, itos)
    got_s, got_p = s["M"].tensor_to_smiles_and_prob_2(tok.cuda(), pr.cuda(), itos)
    assert got_s == ref_s and got_s[6] == "" and len(got_p) == 300
    assert all(torch.equal(a.cpu(), b) for a, b in zip(got_p, ref_p))
    assert s["M"].tensor_to_smiles(tok.cuda(), itos) == ref_s
    got_s1, got_p1 = s["M"].tensor_to_smiles_and_prob(tok.cuda(), pr.t().contiguous().cuda(), itos)   # (N,T) probabilities
    assert got_s1 == ref_s and all(torch.equal(a.cpu(), b) for a, b in zip(got_p1, ref_p))
    one_s, one_p = s["M"].tensor_to_smiles_and_prob_2(tok[:, 9].cuda(), pr[:, 9].cuda(), itos)
    assert one_s == ref_s[9] and torch.equal(one_p.cpu(), ref_p[9])


# --------------------------------------------------------------------------- shapes at the edges
@pytest.mark.parametrize("B,max_len,precision", [(1, 5, "fp32"), (3, 7, "fp32"), (3, 13, "bf16"), (5, 32, "bf16"), (300, 4, "fp32")])
def test_odd_batches_and_lengths_vs_oracle(B, max_len, precision):
    """Single / odd numbers of spectra (half-empty CTAs, uneven decode lanes, encoder chunks of 256 + remainder) and
    lengths that are prime or not multiples of the graph group: greedy ids equal the oracle's (fp32) / the fp32 engine's
    wherever the margin allows (bf16)."""
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    data = synthetic.make_spectra(B, seed=900 + B)
    cfg = cfg_for(max_len=max_len, precision=precision)
    memory, mask, *_ = s["M"].run_model(s["model"], data, cfg)
    tok, pr = s["M"].greedy_sequence_2(s["model"], STOI, None, memory, mask, cfg)
    assert tuple(tok.shape) == (max_len, B) and tuple(pr.shape) == (max_len, B)
    ocfg = s["O"].default_config(max_len=max_len)
    sub = {k: v[:8] for k, v in data.items()}                     # the oracle re-runs the whole prefix: keep it small
    with torch.no_grad():
        omem, omask, _, _ = s["O"].encode(s["P"], sub, ocfg)
        otok, opr = s["O"].greedy_sequence(s["P"], omem, omask, ocfg)
    n = min(B, 8)
    if precision == "fp32":
        np.testing.assert_allclose(memory[:, :n].cpu().numpy(), omem.numpy(), atol=5e-5, rtol=0)
        assert torch.equal(tok[:, :n].cpu(), otok)
    else:
        assert float((tok[:, :n].cpu() == otok).float().mean()) > 0.9
        assert torch.equal(tok[0, :n].cpu(), otok[0])


# --------------------------------------------------------------------------- scheduling must not change results
def _engine_with_env(**env):
    import os
    s = setup()
    from multimodalspectraltransformer_b200.engine import Engine
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        return Engine(s["model"].state_dict(), s["cfg"], "cuda")
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_decode_is_invariant_to_lanes_graphs_pdl_and_repeats(precision):
    """Every sequence is independent: splitting the wave into concurrent lanes, replaying a cached graph, switching
    programmatic dependent launch or graph capture off, or using the un-fused large-wave kernels must give the same
    ids; probabilities agree to rounding (the un-fused path reduces in a different order)."""
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    data = {k: v.cuda() for k, v in synthetic.make_spectra(37, seed=41).items()}
    mode = "1H_13C_HSQC_COSY_IR_MF_MW"
    memory, pad, kb, *_ = s["eng"].encode(data, mode, precision)
    kw = dict(max_len=48, sampling="greedy", precision=precision)
    tok0, pr0, _ = s["eng"].decode(memory, kb, **kw)
    tok1, pr1, _ = s["eng"].decode(memory, kb, **kw)                     # second call: cached graph, staged outputs
    assert torch.equal(tok0, tok1) and torch.equal(pr0, pr1)
    for env in (dict(MMT_DECODE_LANES=1), dict(MMT_DECODE_LANES=4), dict(MMT_NO_PDL=1), dict(MMT_NO_GRAPH=1),
                dict(MMT_NO_GRAPH_CACHE=1), dict(MMT_GRAPH_STEPS=5)):
        eng = _engine_with_env(**env)
        tok, pr, _ = eng.decode(memory, kb, **kw)
        assert torch.equal(tok, tok0), env
        assert torch.equal(pr, pr0), env
    eng = _engine_with_env(MMT_FUSED_DECODE_ROWS=0)                      # tcgen05 / SIMT GEMM per projection
    tok, pr, _ = eng.decode(memory, kb, **kw)
    if precision == "fp32":
        assert torch.equal(tok, tok0)
        torch.testing.assert_close(pr, pr0, atol=1e-5, rtol=0)
    else:
        # bf16 tcgen05 projections vs fp32-accumulated bf16-weight FMA: the two kernel families differ by bf16 round-off, so a
        # free-running sequence may leave the other family's ids -- but only at a near-tie: where the fp32 logits of the
        # shared prefix have a top-2 margin below 2e-2 of the row scale (the north_star tolerance, applied to both sides)
        mem32, _, kb32, *_ = s["eng"].encode(data, mode, "fp32")
        trg = torch.cat([torch.full((1, tok0.shape[1]), 3, dtype=torch.int64, device=tok0.device), tok0[:-1]], dim=0)
        lg = s["eng"].teacher_forced(mem32, kb32, trg, precision="fp32")
        top2 = torch.topk(lg, 2, dim=2).values
        margin = (top2[..., 0] - top2[..., 1]) / lg.abs().amax(dim=2)
        ne = tok != tok0
        for n in torch.nonzero(ne.any(dim=0))[:, 0].tolist():
            t = int(torch.nonzero(ne[:, n])[0])
            assert float(margin[t, n]) < 2e-2, (n, t, float(margin[t, n]))
        assert float(ne.any(dim=0).float().mean()) < 0.5                 # most sequences never meet a near-tie in 48 steps


def test_multinomial_cached_graph_follows_the_generator():
    """The cached decode graph reads the Philox state from device memory: a reseeded / advanced generator must change the
    draws, the same state must reproduce them."""
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    data = {k: v.cuda() for k, v in synthetic.make_spectra(6, seed=2).items()}
    memory, pad, kb, *_ = s["eng"].encode(data, "1H_13C_HSQC_COSY_IR_MF_MW", "bf16")
    kw = dict(n_cand=16, max_len=24, sampling="multinomial", precision="bf16")
    a, _, _ = s["eng"].decode(memory, kb, seed=5, offset=0, **kw)
    b, _, _ = s["eng"].decode(memory, kb, seed=5, offset=0, **kw)
    c, _, _ = s["eng"].decode(memory, kb, seed=5, offset=4 * 24, **kw)
    d, _, _ = s["eng"].decode(memory, kb, seed=6, offset=0, **kw)
    assert torch.equal(a, b) and not torch.equal(a, c) and not torch.equal(a, d)


def test_teacher_forced_scorers_vs_reference_golden():
    """predict_prop_correct_max_sequence(_2,_3): one KV-cached pass == the reference's prefix-by-prefix loop."""
    import os
    from golden_util import GOLDEN
    from multimodalspectraltransformer_b200 import synthetic
    s = setup()
    z = np.load(os.path.join(GOLDEN, "scorer_b3.npz"))
    for tag in ("a", "b"):
        cfg = cfg_for(temperature=float(z[f"{tag}_temperature"]))
        cfg.training_mode = "1H_13C_HSQC_COSY_IR_MF_MW"
        B = int(z[f"{tag}_B"])
        data = synthetic.make_spectra(B, seed=int(z[f"{tag}_seed"]))
        memory, mask, trg_enc_SMI, *_ = s["M"].run_model(s["model"], data, cfg)
        for fn in (s["M"].predict_prop_correct_max_sequence_2, s["M"].predict_prop_correct_max_sequence_3):
            trg, corr, trg_max, mx = fn(s["model"], STOI, memory, mask, trg_enc_SMI, cfg)
            assert trg.shape == z[f"{tag}_trg"].shape and corr.shape == z[f"{tag}_corr"].shape and mx.shape == z[f"{tag}_max"].shape
            assert np.array_equal(trg.cpu().numpy(), z[f"{tag}_trg"])
            assert np.array_equal(trg_max.cpu().numpy(), z[f"{tag}_trg_max"])          # arg-max ids bit-exact (fp32 check mode)
            np.testing.assert_allclose(corr.cpu().numpy(), z[f"{tag}_corr"], atol=2e-5, rtol=0)
            np.testing.assert_allclose(mx.cpu().numpy(), z[f"{tag}_max"], atol=2e-5, rtol=0)
        if B > 1:
            with pytest.raises(ValueError, match="only one element"):            # the reference's own failure for N > 1
                s["M"].predict_prop_correct_max_sequence(s["model"], STOI, memory, mask, trg_enc_SMI, 3, cfg)
            continue
        # five-output variant: the extra output is the probability of one torch.multinomial draw per position
        gen = torch.cuda.default_generators[torch.cuda.current_device()]
        torch.manual_seed(99)
        off0 = gen.get_offset()
        five = s["M"].predict_prop_correct_max_sequence(s["model"], STOI, memory, mask, trg_enc_SMI, 3, cfg)
        assert tuple(five[4].shape) == tuple(z[f"{tag}_multinom_shape"])
        L = five[1].shape[0]
        assert gen.get_offset() - off0 == L * engine_inc(s, 1)
        # the same draws from stock torch on the teacher-forced probabilities
        real_trg = trg_enc_SMI.cuda().transpose(0, 1)[1:]
        trg_in = torch.cat([torch.full((1, 1), 3, dtype=torch.long, device="cuda"), real_trg[:-1]], dim=0)
        logits = s["M"].teacher_forced_logits(s["model"], memory, mask, trg_in, cfg)
        probs = torch.softmax(logits / cfg.temperature, dim=2)
        torch.manual_seed(99)
        want = torch.stack([probs[t].gather(1, torch.multinomial(probs[t], 1)).squeeze() for t in range(L)])
        agree = (torch.isclose(five[4], want, atol=1e-6)).float().mean().item()
        assert agree >= 0.95, agree


def engine_inc(s, n):
    from multimodalspectraltransformer_b200.engine import engine_for
    return engine_for(s["model"], s["cfg"]).philox_increment(n)


def test_calls_are_ordered_on_the_callers_current_stream():
    """SURVEY 8b: everything runs on the current CUDA stream.  Encode + greedy + multinomial + beam search issued on a side
    stream (with work queued in front of them) give the results of the default stream, in both precisions."""
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    data = synthetic.make_spectra(5, seed=91)
    for prec in ("fp32", "bf16"):
        cfg = cfg_for(max_len=24, precision=prec)
        cfg.gen_len = 6

        def go():
            memory, mask, *_ = s["M"].run_model(s["model"], data, cfg)
            tok, pr = s["M"].greedy_sequence(s["model"], STOI, None, memory, mask, cfg)
            torch.manual_seed(5)
            mt, mp = s["M"].multinomial_sequence_multi(s["model"], memory, mask, STOI, cfg, n_candidates=3)
            beams = s["M"].beam_search(s["model"], STOI, memory, mask, cfg, 3)
            return memory, tok, pr, mt, mp, beams

        ref = go()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            junk = torch.randn(4096, 4096, device="cuda")
            for _ in range(20):                    # a backlog in front of the calls
                junk = junk @ junk * 1e-3
            out = go()
        side.synchronize()
        assert torch.equal(out[0], ref[0]) and torch.equal(out[1], ref[1]) and torch.equal(out[2], ref[2])
        assert torch.equal(out[3], ref[3]) and torch.equal(out[4], ref[4]) and out[5] == ref[5]


def test_engines_follow_their_models():
    """Callers pass a live nn.Module on every call (SURVEY 8b): two models interleave without cross-talk, and an in-place
    weight update (optimizer step, checkpoint load) is picked up by the next call."""
    import copy
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    from multimodalspectraltransformer_b200.engine import engine_for
    data = synthetic.make_spectra(3, seed=92)
    cfg = cfg_for(max_len=16)
    a = s["model"]
    b = copy.deepcopy(a)
    with torch.no_grad():
        b.fc_out.bias[7] += 4.0
    mem_a, mask_a, *_ = s["M"].run_model(a, data, cfg)
    mem_b, mask_b, *_ = s["M"].run_model(b, data, cfg)
    assert torch.equal(mem_a, mem_b)                         # same encoder weights
    ta, _ = s["M"].greedy_sequence(a, STOI, None, mem_a, mask_a, cfg)
    tb, _ = s["M"].greedy_sequence(b, STOI, None, mem_b, mask_b, cfg)
    ta2, _ = s["M"].greedy_sequence(a, STOI, None, mem_a, mask_a, cfg)
    assert torch.equal(ta, ta2) and not torch.equal(ta, tb) and (tb == 7).float().mean() > (ta == 7).float().mean()
    assert engine_for(a, cfg) is not engine_for(b, cfg) and engine_for(a, cfg) is engine_for(a, cfg)
    # in-place update of b -> rebuilt engine, results equal a's again
    e_before = engine_for(b, cfg)
    with torch.no_grad():
        b.fc_out.bias[7] -= 4.0
    tb2, _ = s["M"].greedy_sequence(b, STOI, None, mem_b, mask_b, cfg)
    assert engine_for(b, cfg) is not e_before
    assert torch.equal(tb2, ta)
    # load_state_dict (checkpoint) is an in-place copy as well
    with torch.no_grad():
        sd = {k: v.clone() for k, v in b.state_dict().items()}
        sd["fc_out.bias"][9] += 5.0
    b.load_state_dict(sd)
    tb3, _ = s["M"].greedy_sequence(b, STOI, None, mem_b, mask_b, cfg)
    assert (tb3 == 9).float().mean() > (ta == 9).float().mean()
