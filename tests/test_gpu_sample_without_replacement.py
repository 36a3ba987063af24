"""Sampling without replacement by stochastic beam search (mmt_sample_without_replacement, kernels_sbs.cuh).

The selection kernel is checked step by step against a numpy fp64 restatement of the rule on the exact noise
(Engine.exponential), with restatements that are wrong in one detail as sharpness guards; the whole call against a
full-prefix oracle search; the sample against the exact leaf distribution (chi-square); the invariants at the bench
geometry; column independence across waves, graph reuse and no-graph runs; and the argument checks."""
import copy
import ctypes as C
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

STOI = {"<PAD>": 0, "<UNK>": 1, "<EOS>": 2, "<SOS>": 3, "<MASK>": 4}
EOS = 2
MODE = "1H_13C_HSQC_COSY_IR_MF_MW"
_S = {}


def setup():
    if "model" not in _S:
        import multimodalspectraltransformer_b200 as M
        from oracle import mmt_oracle as O
        cfg = M.default_config(device="cuda")
        cfg.training_mode = MODE
        torch.manual_seed(0)
        model = M.MultimodalTransformer(cfg)
        model.eval()
        P = O.random_init_state_dict(O.default_config(), seed=0)
        # <EOS> raised (as in test_gpu_beam.py): finished slots and mixed lengths within a few steps
        m_eos = copy.deepcopy(model)
        with torch.no_grad():
            m_eos.fc_out.bias[EOS] += 1.5
        P_eos = {k: v.clone() for k, v in P.items()}
        P_eos["fc_out.bias"][EOS] += 1.5
        _S.update(M=M, O=O, model=model, model_eos=m_eos, P_eos=P_eos)
    return _S


def config(**over):
    s = setup()
    cfg = s["M"].default_config(device="cuda", **over)
    cfg.training_mode = MODE
    return cfg


def encode(model, B, seed, precision="fp32"):
    s = setup()
    from multimodalspectraltransformer_b200 import synthetic
    cfg = config()
    cfg.precision = precision
    memory, mask, *_ = s["M"].run_model(model, synthetic.make_spectra(B, seed=seed), cfg)
    return memory, mask


def new_engine(model, monkeypatch=None, **env):
    from multimodalspectraltransformer_b200.engine import Engine
    if monkeypatch is not None:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
    eng = Engine(model.state_dict(), config(), torch.device("cuda", torch.cuda.current_device()))
    if monkeypatch is not None:
        for k in env:
            monkeypatch.delenv(k)
    return eng


def bias_of(mask):
    from multimodalspectraltransformer_b200.generate import _mask_to_bias
    return _mask_to_bias(mask)


# ----------------------------------------------------------------------------- numpy restatement of one step
def log1mexp(x):
    x = np.asarray(x, dtype=np.float64)
    with np.errstate(divide="ignore"):
        return np.where(x > -math.log(2.0), np.log(-np.expm1(x)), np.log1p(-np.exp(x)))


def child_keys(G, gh, Z, conditioned=True):
    if not conditioned:
        return gh
    with np.errstate(invalid="ignore"):
        v = G - gh + log1mexp(gh - Z)
        return G - np.maximum(0.0, v) - np.log1p(np.exp(-np.abs(v)))


def select_np(p, E, phi, G, lens, hist, T, eos, k, V, *, row_shift=0, conditioned=True, ties_low_first=True):
    """One column: candidates (key, index c = rank * V + token, parent, token | -1) -> the k selected, in order."""
    cands = []
    for r in range(k):
        if G[r] == -np.inf:
            continue
        L = int(lens[r])
        if L >= T or (L > 0 and hist[r, L - 1] == eos):
            cands.append((G[r], r * V, r, -1))
            continue
        ok = p[r] > 0
        e = E[((r + row_shift) % k) * V:((r + row_shift) % k) * V + V].astype(np.float64)
        with np.errstate(divide="ignore"):
            gh = np.where(ok, phi[r] + np.log(p[r].astype(np.float64)) - np.log(e), -np.inf)
        keys = child_keys(G[r], gh, gh.max(), conditioned)
        cands += [(keys[i], r * V + i, r, i) for i in range(V) if ok[i]]
    sign = 1 if ties_low_first else -1
    cands.sort(key=lambda c: (-c[0], sign * c[1]))
    return cands[:k], cands


def near_ties(cands, k, rel=1e-12):
    """Adjacent keys among the first k + 1 candidates closer than rel without being equal (exact ties follow the rule)."""
    n = 0
    for a, b in zip(cands[:k], cands[1:k + 1]):
        if a[0] != b[0] and abs(a[0] - b[0]) <= rel * max(abs(a[0]), abs(b[0]), 1e-300):
            n += 1
    return n


def random_state(rng, Bm, k, V, T, t):
    """Slots with sorted-ish keys: live ones (length t), finished ones (an <EOS> at length - 1 <= t), empty ones; in
    columns with k >= 5 two finished slots share one key above all others (exercises the tie rule)."""
    N = Bm * k
    phi = np.full(N, -np.inf)
    G = np.full(N, -np.inf)
    lens = np.zeros(N, np.int32)
    hist = np.zeros((N, T), np.uint8)
    probs = np.zeros((N, T), np.float32)
    for b in range(Bm):
        n_live = max(1, int(rng.integers(1, k + 1)))
        keys = np.sort(rng.normal(0, 3, k))[::-1]
        for r in range(k):
            n = b * k + r
            if r >= n_live and r > 0 and rng.random() < 0.5:
                continue                                    # empty
            phi[n] = -abs(rng.normal(0, 5)) - 0.1
            G[n] = keys[r]
            fin = r > 0 and rng.random() < 0.3
            L = int(rng.integers(1, t + 1)) if fin and t > 0 else t
            lens[n] = L
            hist[n, :L] = rng.integers(5, V, L)
            if fin and L > 0:
                hist[n, L - 1] = EOS
            probs[n, :L] = rng.uniform(0.01, 1, L)
        if k >= 5 and t > 0:                                # tied finished slots 1 and 2
            for r in (1, 2):
                n = b * k + r
                G[n], phi[n], lens[n] = keys[0] + 1.0, -1.0, t
                hist[n, :t] = rng.integers(5, V, t)
                hist[n, t - 1] = EOS
                hist[n, 0] = 5 + r
    logits = rng.normal(0, 2.5, (N, V)).astype(np.float32)
    logits[rng.random((N, V)) < 0.05] = -np.inf             # tokens with p = 0 are not candidates
    return logits, phi, G, lens, hist, probs


@pytest.mark.parametrize("k", [1, 5, 43, 64, 128])
def test_select_step_matches_numpy_fp64(k):
    s = setup()
    from multimodalspectraltransformer_b200.engine import engine_for
    eng = engine_for(s["model"], config())
    V, T, Bm, seed, off, base = 43, 24, 3, 1234, 8, 2
    rng = np.random.default_rng(k)
    inc = eng.philox_increment(k)
    guards = {"row": 0, "cond": 0, "tie": 0}
    n_near = 0
    for t in (0, 7, 16):
        logits, phi, G, lens, hist, probs = random_state(rng, Bm, k, V, T, t)
        if t == 0:                                          # the root state
            phi[:], G[:], lens[:], hist[:], probs[:] = -np.inf, -np.inf, 0, 0, 0
            phi[::k], G[::k] = 0.0, 0.0
        temp = rng.uniform(0.5, 1.5, Bm).astype(np.float32)
        out = eng.sbs_select_step(torch.from_numpy(logits), torch.from_numpy(phi), torch.from_numpy(G), torch.from_numpy(lens),
                                  torch.from_numpy(hist), torch.from_numpy(probs), k=k, step=t, eos=EOS, temperature=temp,
                                  seed=seed, offset=off, seq_index_base=base * k)
        phi2, G2, len2, hist2, probs2, p = [x.cpu().numpy() for x in out]
        for b in range(Bm):
            sl = slice(b * k, (b + 1) * k)
            E = eng.exponential(k * V, seed=seed, offset=off + ((base + b) * T + t) * inc).cpu().numpy()
            pb = p[sl]
            args = (pb, E, phi[sl], G[sl], lens[sl], hist[sl], T, EOS, k, V)
            sel, cands = select_np(*args)
            n_near += near_ties(cands, k)
            kk = len(sel)
            # keys, log-probabilities, lengths, histories and probabilities of the selected slots, in order
            np.testing.assert_allclose(G2[sl][:kk], [c[0] for c in sel], rtol=1e-12, atol=1e-12)
            for j, (key, c, q, tok) in enumerate(sel):
                n, nq = b * k + j, b * k + q
                want_len = lens[nq] + (tok >= 0)
                assert len2[n] == want_len
                assert list(hist2[n, :lens[nq]]) == list(hist[nq, :lens[nq]])
                assert (hist2[n, lens[nq]] == tok) if tok >= 0 else True
                assert not hist2[n, want_len:t + 1].any() and not probs2[n, want_len:t + 1].any()
                want_phi = phi[nq] + (math.log(float(pb[q, tok])) if tok >= 0 else 0.0)
                assert phi2[n] == pytest.approx(want_phi, rel=1e-13, abs=1e-13)
                if tok >= 0:
                    assert probs2[n, lens[nq]] == pb[q, tok]
            assert np.all(G2[sl][kk:] == -np.inf) and np.all(len2[sl][kk:] == 0) and not hist2[sl][kk:, :t + 1].any()
            # the restatement is sharp: each wrong detail changes the selection on these inputs
            got = [(int(len2[b * k + j]), bytes(hist2[b * k + j, :t + 1])) for j in range(kk)]

            def as_state(sel_):
                return [(int(lens[b * k + q] + (tok >= 0)),
                         bytes(np.concatenate([hist[b * k + q, :lens[b * k + q]], [tok] if tok >= 0 else [],
                                               np.zeros(t + 1, np.uint8)]).astype(np.uint8)[:t + 1])) for _, _, q, tok in sel_]
            assert as_state(sel) == got
            guards["row"] += as_state(select_np(*args, row_shift=1)[0]) != got
            guards["cond"] += as_state(select_np(*args, conditioned=False)[0]) != got
            guards["tie"] += as_state(select_np(*args, ties_low_first=False)[0]) != got
    assert n_near == 0
    if k >= 2:                                              # (k = 1: one row, one child per leaf-free slot)
        assert guards["row"] > 0 and guards["cond"] > 0, guards
    if k >= 5:
        assert guards["tie"] > 0, guards


def test_select_step_probabilities_are_the_samplers():
    """p of the selection step is bit-identical to the multinomial sampler's at the same temperature."""
    s = setup()
    from multimodalspectraltransformer_b200.engine import engine_for
    eng = engine_for(s["model"], config())
    k, Bm, T = 16, 4, 8
    x = torch.randn(Bm * k, 128, device="cuda")
    temp = np.array([0.7, 1.0, 1.3, 0.45], np.float32)
    tok, pr, lg, _ = eng.sample_controlled(x=x, n_cand=k, temperature=temp, seed=3, offset=0, want_logits=True)
    N = Bm * k
    phi = torch.zeros(N, dtype=torch.float64)
    G = torch.zeros(N, dtype=torch.float64)
    out = eng.sbs_select_step(lg, phi, G, torch.zeros(N, dtype=torch.int32), torch.zeros(N, T, dtype=torch.uint8),
                              torch.zeros(N, T), k=k, step=0, eos=EOS, temperature=temp, seed=1, offset=0)
    p = out[5]
    assert torch.equal(p.gather(1, tok.unsqueeze(1)).squeeze(1), pr)


# ----------------------------------------------------------------------------- whole call against the oracle
def oracle_sbs(P, memory, mask, ocfg, k, T, temps, seed, offset, exp_fn, inc, base=0, tol=2e-5):
    """Full-prefix stochastic beam search per column (fp64 keys), the noise from exp_fn (bit-exact variates).
    -> per column (list of (sequence, probs) in slot order, step at which a near-tie of keys at or inside the
    selection boundary made the order fragile, or None)."""
    O = setup()["O"]
    res = []
    for b in range(memory.shape[1]):
        slots = [(0.0, 0.0, [], [])]                      # (phi, G, tokens, probs)
        fragile = None
        for t in range(T):
            E = exp_fn(k * V_OF, seed, offset + ((base + b) * T + t) * inc)
            live = [r for r, sl in enumerate(slots) if not (sl[2] and (sl[2][-1] == EOS or len(sl[2]) >= T))]
            p_all = {}
            if live:
                trg = torch.tensor([[3] + slots[r][2] for r in live], dtype=torch.long).T
                mem = memory[:, b:b + 1].expand(-1, len(live), -1)
                msk = mask[b:b + 1].expand(len(live), -1)
                with torch.no_grad():
                    lg = O.teacher_forced_logits(P, mem, msk, trg, ocfg)[-1]
                pr = torch.softmax(lg / float(temps[b]), dim=-1).numpy()
                for i, r in enumerate(live):
                    p_all[r] = pr[i]
            cands = []
            for r, (phi, G, toks, prs) in enumerate(slots):
                if r not in p_all:
                    cands.append((G, r * V_OF, phi, toks, prs))
                    continue
                p = p_all[r].astype(np.float64)
                e = E[r * V_OF:(r + 1) * V_OF].astype(np.float64)
                ok = p > 0
                with np.errstate(divide="ignore"):
                    gh = np.where(ok, phi + np.log(p) - np.log(e), -np.inf)
                keys = child_keys(G, gh, gh.max())
                cands += [(keys[i], r * V_OF + i, phi + math.log(p[i]), toks + [i], prs + [float(p_all[r][i])])
                          for i in range(V_OF) if ok[i]]
            cands.sort(key=lambda c: (-c[0], c[1]))
            top = [c[0] for c in cands[:k + 1]]
            if fragile is None and any(abs(a - b_) <= tol * max(1.0, abs(a)) for a, b_ in zip(top, top[1:])):
                fragile = t
            slots = [(c[2], c[0], c[3], c[4]) for c in cands[:k]]
        res.append(([(sl[2], sl[3]) for sl in slots], fragile))
    return res


V_OF = 43


@pytest.mark.parametrize("k,T", [(1, 5), (7, 5), (128, 5), (1, 20), (7, 20), (128, 20)])
def test_whole_call_matches_oracle(k, T):
    """fp32 engine vs the full-prefix oracle on the <EOS>-heavy weights, four columns.  Rule: every column's slots must
    equal the oracle's in order (sequences exactly, probabilities to 5e-5), except a column in which the oracle met
    two keys within 2e-5 among its k + 1 best candidates at some step (the two fp32 decoders differ by ~1e-6 in the
    logits, so such an order may flip, and every later step then follows other parents and other noise rows); at
    most half the columns may be excused so."""
    s = setup()
    from multimodalspectraltransformer_b200.engine import engine_for
    model, P = s["model_eos"], s["P_eos"]
    memory, mask = encode(model, 4, seed=5 + k + T)
    eng = engine_for(model, config())
    temps = np.array([1.0, 0.8, 1.2, 0.6], np.float32)
    seed, off = 77, 12
    tokens, probs, lens, logp, key, steps = eng.sample_without_replacement(
        memory, bias_of(mask), n_cand=k, max_len=T, temperature=temps, eos=EOS, seed=seed, offset=off)
    ocfg = s["O"].default_config(training_mode=MODE)
    inc = eng.philox_increment(k)
    exp_fn = lambda n, sd, of: eng.exponential(n, seed=sd, offset=of).cpu().numpy()
    want = oracle_sbs(P, memory.cpu(), mask.cpu(), ocfg, k, T, temps, seed, off, exp_fn, inc)
    tokens, probs, lens = tokens.cpu().numpy(), probs.cpu().numpy(), lens.cpu().numpy()
    excused = 0
    for b, (slots, fragile) in enumerate(want):
        same = all(lens[b * k + j] == len(toks) and list(tokens[:len(toks), b * k + j]) == toks for j, (toks, _) in enumerate(slots))
        same = same and all(lens[b * k + j] == 0 for j in range(len(slots), k))
        if not same:
            assert fragile is not None, f"column {b} differs from the oracle without a near-tie of keys"
            excused += 1
            continue
        for j, (toks, prs) in enumerate(slots):
            np.testing.assert_allclose(probs[:len(toks), b * k + j], prs, rtol=0, atol=5e-5)
    assert excused <= 2
    if k > 1 and T == 20:
        assert len(set(lens.tolist())) > 1, "expected finished slots of different lengths"


# ----------------------------------------------------------------------------- distribution
def chi2_p(obs, exp):
    from scipy.stats import chisquare
    obs, exp = np.asarray(obs, float), np.asarray(exp, float)
    return chisquare(obs, exp * obs.sum() / exp.sum()).pvalue


def bins(counts, probs, n, min_expected=5.0):
    """Leaves with n * P >= min_expected as bins, every other leaf (and anything unseen) pooled into one bin."""
    keys = [s for s, pr in probs.items() if n * pr >= min_expected]
    obs = [counts.get(s, 0) for s in keys]
    exp = [probs[s] for s in keys]
    obs.append(n - sum(obs))
    exp.append(max(1.0 - sum(exp), 0.0))
    return obs, exp


def test_slots_are_a_sample_without_replacement():
    s = setup()
    from multimodalspectraltransformer_b200.engine import engine_for
    model = s["model"]
    memory, mask = encode(model, 1, seed=21)
    eng = engine_for(model, config())
    Bn, T, k = 4096, 2, 2
    # exact leaf probabilities: p(a) at position 0, p(b | a) at position 1 (fp32 engine logits, softmax in fp64), at the
    # highest of a few temperatures under which the likeliest leaf has P >= 0.05
    trg = torch.stack([torch.full((V_OF,), 3, dtype=torch.long), torch.arange(V_OF)]).cuda()
    lg = eng.teacher_forced(memory[:, :1].expand(-1, V_OF, -1).contiguous(), bias_of(mask[:1].expand(V_OF, -1)), trg).double().cpu()
    for tau in (1.0, 0.7, 0.5, 0.35, 0.25, 0.15):
        p0 = torch.softmax(lg[0, 0] / tau, -1).numpy()
        p1 = torch.softmax(lg[1] / tau, -1).numpy()
        P = {(EOS,): p0[EOS]}
        for a in range(V_OF):
            if a != EOS:
                for c in range(V_OF):
                    P[(a, c)] = p0[a] * p1[a, c]
        if max(P.values()) >= 0.05:
            break
    assert max(P.values()) >= 0.05, "no temperature made a few leaves dominant"
    mem = memory[:, [0] * Bn].contiguous()
    msk = mask[[0] * Bn]
    for seed in (11, 12):
        tokens, _, lens, _, key, _ = eng.sample_without_replacement(mem, bias_of(msk), n_cand=k, max_len=T, temperature=tau,
                                                                    eos=EOS, seed=seed, offset=0)
        tokens, lens = tokens.cpu().numpy(), lens.cpu().numpy()
        seqs = [tuple(tokens[:lens[n], n]) for n in range(Bn * k)]
        s0 = [seqs[b * k] for b in range(Bn)]
        s1 = [seqs[b * k + 1] for b in range(Bn)]
        assert all(a != b for a, b in zip(s0, s1))
        c0 = {}
        for x in s0:
            c0[x] = c0.get(x, 0) + 1
        assert chi2_p(*bins(c0, P, Bn)) > 1e-4
        pair = {}
        for a, b in zip(s0, s1):
            pair[(a, b)] = pair.get((a, b), 0) + 1
        big = [x for x, pr in P.items() if pr > 1e-3]
        PP = {(a, b): P[a] * P[b] / (1 - P[a]) for a in big for b in big if a != b}
        assert chi2_p(*bins(pair, PP, Bn)) > 1e-4


def test_fewer_leaves_than_slots_leaves_empty_slots():
    s = setup()
    from multimodalspectraltransformer_b200.engine import engine_for
    memory, mask = encode(s["model"], 3, seed=4)
    eng = engine_for(s["model"], config())
    tokens, probs, lens, logp, key, _ = eng.sample_without_replacement(memory, bias_of(mask), n_cand=64, max_len=1,
                                                                       temperature=1.0, eos=EOS, seed=5, offset=0)
    for b in range(3):
        sl = slice(b * 64, (b + 1) * 64)
        assert sorted(tokens[0, sl][:43].tolist()) == list(range(43))
        assert torch.all(lens[sl][:43] == 1) and torch.all(lens[sl][43:] == 0)
        assert torch.all(key[sl][43:] == -math.inf) and torch.all(logp[sl][43:] == -math.inf)
        assert torch.all(torch.isfinite(key[sl][:43])) and torch.all(tokens[0, sl][43:] == 0) and torch.all(probs[0, sl][43:] == 0)
        assert torch.all(key[sl][:42] >= key[sl][1:43])


# ----------------------------------------------------------------------------- bench geometry
def test_invariants_at_bench_geometry():
    """1024 spectra x 128 candidates x 128 positions in bf16 through the public call: two waves by default."""
    s = setup()
    M = s["M"]
    from multimodalspectraltransformer_b200.engine import engine_for
    model = copy.deepcopy(s["model"])      # its engine (and tens of GB of arena) goes when the test ends
    cfg = config()
    cfg.precision = "bf16"
    memory, mask = encode(model, 1024, seed=0, precision="bf16")
    eng = engine_for(model, cfg)
    g = torch.cuda.default_generators[torch.cuda.current_device()]
    off0 = g.get_offset()
    tokens, probs, logp, key = M.sample_without_replacement(model, STOI, memory, mask, cfg, n_candidates=128)
    assert g.get_offset() == off0 + 1024 * 128 * eng.philox_increment(128)
    T, N = tokens.shape
    assert (T, N) == (128, 1024 * 128)
    tok = tokens.to(torch.uint8).T.contiguous()                    # (N, T)
    is_eos = tok == EOS
    has = is_eos.any(1)
    first = torch.where(has, is_eos.to(torch.int32).argmax(1), torch.full_like(has, T, dtype=torch.int64))
    lens = torch.where(has, first + 1, first)
    pos = torch.arange(T, device=tok.device).unsqueeze(0)
    after = pos >= lens.unsqueeze(1)
    assert not tok[after].any() and not probs.T[after].any()
    assert torch.all(probs.T[~after] > 0)
    assert torch.all(tok[~after & (pos < (lens - 1).unsqueeze(1))] != EOS)
    lp = torch.where(after, torch.zeros((), dtype=torch.float64, device=tok.device), probs.T.double().clamp_min(1e-300).log()).sum(1)
    assert torch.allclose(lp, logp, rtol=0, atol=1e-9)
    kk = key.view(1024, 128)
    assert torch.all(kk[:, :-1] >= kk[:, 1:]) and torch.all(torch.isfinite(kk))
    rows = tok.cpu().numpy().view(np.dtype((np.void, T))).reshape(1024, 128)
    assert all(len(set(r.tolist())) == 128 for r in rows), "sequences of a column must be pairwise distinct"
    itos = {str(i): c for i, c in enumerate(["<PAD>", "<UNK>", "<EOS>", "<SOS>", "<MASK>"] + list("CcONnSsFP()=#123+-[]H@lrBo") + ["C"] * 12)}
    d = M.distinct_smiles(tokens, itos, 128, token_prob=probs)
    assert len(d) == 1024


# ----------------------------------------------------------------------------- column independence, graphs
def test_columns_equal_single_spectrum_calls(monkeypatch):
    """A multi-wave call with a short last wave (7 spectra in waves of 3) at seq_index_base = 3k equals, column by
    column and bit for bit, single-spectrum calls at the shifted seq_index_base -- on the un-fused bf16 family, whose
    kernel variants do not depend on the wave size at these sizes."""
    s = setup()
    model = s["model_eos"]
    k, T, Bm = 16, 24, 7
    memory, mask = encode(model, Bm, seed=8, precision="bf16")
    kb = bias_of(mask)
    eng = new_engine(model, monkeypatch, MMT_FUSED_DECODE_ROWS="0", MMT_MAX_WAVE_SEQS=str(2 * 3 * k))
    temps = np.linspace(0.6, 1.4, Bm).astype(np.float32)
    kw = dict(n_cand=k, max_len=T, eos=EOS, seed=99, offset=40, precision="bf16")
    full = eng.sample_without_replacement(memory, kb, temperature=temps, seq_index_base=3 * k, **kw)
    for b in range(Bm):
        one = eng.sample_without_replacement(memory[:, b:b + 1], kb[b:b + 1], temperature=float(temps[b]),
                                             seq_index_base=(3 + b) * k, **kw)
        sl = slice(b * k, (b + 1) * k)
        assert torch.equal(full[0][:, sl], one[0]) and torch.equal(full[1][:, sl], one[1]), b
        for i in (2, 3, 4):
            assert torch.equal(full[i][sl], one[i]), (b, i)


def test_graph_cache_reuse_and_no_graph(monkeypatch):
    s = setup()
    model = s["model_eos"]
    k, T, Bm = 8, 24, 4
    memory, mask = encode(model, Bm, seed=9)
    kb = bias_of(mask)
    kw = dict(n_cand=k, max_len=T, eos=EOS, seed=5, offset=16)
    t1, t2 = 1.0, np.array([0.5, 0.9, 1.3, 2.0], np.float32)
    eng = new_engine(model)
    a1 = eng.sample_without_replacement(memory, kb, temperature=t1, **kw)
    a2 = eng.sample_without_replacement(memory, kb, temperature=t2, **kw)       # the cached step graph, other values
    a3 = eng.sample_without_replacement(memory, kb, temperature=t2, **dict(kw, seed=6))
    ref = new_engine(model, monkeypatch, MMT_NO_GRAPH="1")
    for got, (t, sd) in ((a1, (t1, 5)), (a2, (t2, 5)), (a3, (t2, 6))):
        want = ref.sample_without_replacement(memory, kb, temperature=t, **dict(kw, seed=sd))
        for x, y in zip(got[:5], want[:5]):
            assert torch.equal(x, y)
    assert not torch.equal(a1[0], a2[0]) and not torch.equal(a2[0], a3[0])


# ----------------------------------------------------------------------------- argument checks
def test_validation_errors():
    s = setup()
    M = s["M"]
    from multimodalspectraltransformer_b200 import engine as E
    from multimodalspectraltransformer_b200 import _lib
    cfg = config()
    torch.manual_seed(1)
    fresh = M.MultimodalTransformer(cfg)
    mem = torch.zeros(582, 2, 128, device="cuda")
    msk = torch.zeros(2, 582, dtype=torch.bool, device="cuda")
    for kw, msg in ((dict(n_candidates=0), "n_candidates"), (dict(n_candidates=129), "n_candidates"),
                    (dict(n_candidates=2.0), "n_candidates"), (dict(n_candidates=4, seq_index_base=6), "seq_index_base"),
                    (dict(n_candidates=4, temperature=0.0), "temperature"), (dict(n_candidates=4, temperature=float("nan")), "temperature"),
                    (dict(n_candidates=4, temperature=[1.0, -1.0]), "temperature"), (dict(n_candidates=4, n_total=6), "n_total")):
        with pytest.raises(ValueError, match=msg):
            M.sample_without_replacement(fresh, STOI, mem, msk, cfg, **kw)
    with pytest.raises(ValueError, match="EOS"):
        M.sample_without_replacement(fresh, {k: v for k, v in STOI.items() if k != "<EOS>"}, mem, msk, cfg, n_candidates=4)
    assert fresh not in E._ENGINES
    # C ABI checks
    eng = E.engine_for(s["model"], cfg)
    L = eng.L
    out = [torch.empty(130 * 4, dtype=torch.float64, device="cuda") for _ in range(5)]
    temp = np.ones(2, np.float32)

    def call(temp_arr=temp, eos=EOS, **over):
        a, keep = eng._decode_args(mem, torch.zeros(2, 582, device="cuda"), over.pop("n_cand", 4), over.pop("max_len", 8), 1.0,
                                   1, False, over.pop("precision", "fp32"))
        for f, v in over.items():
            setattr(a, f, v)
        rc = L.mmt_sample_without_replacement(eng.h, C.byref(a), temp_arr.ctypes.data if temp_arr is not None else None, eos,
                                              *[o.data_ptr() for o in out], None, eng._stream())
        return rc, L.mmt_last_error().decode()

    for over, msg in ((dict(n_cand=0), "n_cand"), (dict(n_cand=129), "n_cand"), (dict(max_len=129), "max_len"),
                      (dict(eos=43), "eos"), (dict(eos=-1), "eos"), (dict(seq_index_base=3), "seq_index_base"),
                      (dict(N_total=6), "N_total"), (dict(precision="fp32", stride_s=6), "aligned"),
                      (dict(temp_arr=np.array([1.0, 0.0], np.float32)), "temperature"),
                      (dict(temp_arr=np.array([1.0, np.inf], np.float32)), "temperature"),
                      (dict(temp_arr=None, temperature=-1.0), "temperature")):
        eos = over.pop("eos", EOS)
        ta = over.pop("temp_arr", temp)
        rc, err = call(ta, eos, **over)
        assert rc != 0 and msg in err, (over, err)
    a, _ = eng._decode_args(mem, torch.zeros(2, 582, device="cuda"), 4, 8, 1.0, 1, False, "fp32")
    a.precision = 7
    assert L.mmt_sample_without_replacement(eng.h, C.byref(a), temp.ctypes.data, EOS, *[o.data_ptr() for o in out], None, eng._stream()) != 0
    assert "precision" in L.mmt_last_error().decode()
