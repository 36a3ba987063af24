"""The reference's generation entry points, same names / arguments / return layouts,
running on the B200 engine.

    run_model                    validate_generate_MMT_v15_4.py:95-267
    greedy_sequence              validate_generate_MMT_v15_4.py:723-775
    multinomial_sequence         validate_generate_MMT_v15_4.py:841-880
    multinomial_sequence_multi   run_batch_gen_val_MMT_v15_4.py:121-158
    duplicate_tensor / _dict     run_batch_gen_val_MMT_v15_4.py:93-107
    greedy_sequence_2            mmt_result_test_functions_15_4.py:984-1032
    multinomial_sequence_multi_2 mmt_result_test_functions_15_4.py:791-829
    beam_search                  validate_generate_MMT_v15_4.py:995-1086
    sample_without_replacement   (extension) k distinct candidates per spectrum by stochastic beam search
    predict_prop_correct_max_sequence(_2)   validate_generate_MMT_v15_4.py:309-509
    predict_prop_correct_max_sequence_3     mmt_result_test_functions_15_4.py:340-400

``model`` may be this package's ``MultimodalTransformer`` or the reference's own
instance: only its ``state_dict()`` is read.  Runtime knobs (``device``,
``training_mode``, ``max_len``, ``temperature``, optional ``precision``) are read
from ``config`` at call time, never cached (callers mutate it mid-run,
mmt_result_test_functions_15_4.py:547).

Extensions (keyword-only, default = reference behaviour):
  n_candidates=k   decode k sequences per memory column without materialising the
                   reference's 128x tensor duplication (cross-attention K/V shared);
  seq_index_base / n_total  place the call inside a larger logical batch so sharded
                   runs draw the Philox numbers of the unsharded run.
  per_memory_rng=True  the n_candidates rows of each memory column draw what a separate
                   torch.multinomial((n_candidates, V), 1) per step would, the columns'
                   calls in order: one call over many spectra draws the ids of the
                   reference's per-spectrum loop (seq_index_base must be a multiple of
                   n_candidates; n_total is then the whole call's sequence count).
  stop_at_eos=True  stop computing a sequence once it has emitted stoi["<EOS>"]: ids and
                   probabilities equal the default's up to and including that <EOS> and are
                   <PAD> / 0 after it; shapes and generator advance are unchanged (greedy
                   also stops once every sequence has finished).  Every consumer of the ids
                   (tensor_to_smiles*, distinct_smiles) ignores what follows <EOS>.
  temperature=None, top_k=0, top_p=1.0  multinomial sampling controls per spectrum, each a
                   scalar or one value per spectrum (a spectrum's candidates share them):
                   softmax(logits / temperature) (None: config.temperature at call time), then
                   the draw restricted to the top_k most probable tokens (0 or vocab: off) and,
                   of those, the nucleus of mass top_p (1: off), HF order.  A draw the default
                   call makes inside the kept set is unchanged; the reported probability is the
                   chosen token's softmax(logits / temperature), not renormalised.  Neutral
                   controls run the default call; greedy sampling refuses any other.
"""
from __future__ import annotations

import torch

from . import engine as _engine

SOS_KEY, PAD = "<SOS>", 0


# ------------------------------------------------------------------ helpers
def _mask_to_bias(mask: torch.Tensor) -> torch.Tensor:
    """Key-padding mask -> additive attention bias, torch semantics: bool True -> -inf;
    floating masks are added as they are (SURVEY.md B.2).  Integer masks, which
    torch >= 2 rejects and the reference's collate_fn produces for mask_MF, are read
    as bool (non-zero = pad) -- SURVEY.md B.1."""
    if mask.is_floating_point():
        return mask.to(torch.float32)
    pad = mask if mask.dtype == torch.bool else (mask != 0)
    return torch.zeros(pad.shape, dtype=torch.float32, device=pad.device).masked_fill_(pad, float("-inf"))


def _encode(eng, data, config, want_embedding_src=False, reuse=False):
    prec = _engine.default_precision(config)
    memory, pad, key_bias, fp, avg, emb = eng.encode(data, config.training_mode, prec, want_embedding_src, reuse=reuse)
    from . import _lib
    if _lib.lib().mmt_mask_is_float(_lib.mode_bits(config.training_mode)):
        mask = pad.to(torch.float32)       # torch.cat promoted the reference's mask to float 0/1
    else:
        mask = pad.to(torch.bool)
    return memory, mask, fp, avg, emb


def _check_sos(stoi):
    sos = stoi[SOS_KEY]
    if sos != 3:
        raise ValueError("the engine hard-codes <SOS> = 3 (stoi.json)")
    return sos


def _eos_id(stoi):
    if "<EOS>" not in stoi:
        raise ValueError("stop_at_eos needs an <EOS> entry in stoi")
    return int(stoi["<EOS>"])


def _philox_state(dev_index):
    g = torch.cuda.default_generators[dev_index]
    return g, int(g.initial_seed()), int(g.get_offset())


# ------------------------------------------------------------------- encoder
def run_model(model, data_dict, config):
    """-> (memory (S,B,128), src_padding_mask (B,S), trg_enc_SMI, fingerprint (B,512), src_HSQC, src_COSY)."""
    eng = _engine.engine_for(model, config)
    x = data_dict
    dev = config.device
    distinct = x._distinct() if isinstance(x, _DuplicatedDict) else None
    if distinct is not None and distinct[1] > 1:
        # copies made by duplicate_dict: encode the distinct spectra, tile the results in tensor.repeat's order
        base, n = distinct
        memory, mask, fingerprint, _, _ = _encode(eng, base, config)
        memory, mask, fingerprint = memory.repeat(1, n, 1), mask.repeat(n, 1), fingerprint.repeat(n, 1)
    else:
        memory, mask, fingerprint, _, _ = _encode(eng, x, config)
    src_HSQC = x["src_HSQC"].to(dev) if "HSQC" in config.training_mode else x["src_HSQC_"].to(dev)
    src_COSY = x["src_COSY"].to(dev) if "COSY" in config.training_mode else x["src_COSY_"].to(dev)
    return memory, mask, x["trg_enc_SMI"].to(dev), fingerprint, src_HSQC, src_COSY


def duplicate_tensor(tensor, n_times):
    repeat_dims = [n_times] + [1] * (tensor.dim() - 1)
    return tensor.repeat(*repeat_dims).to("cuda")


class _DuplicatedDict(dict):
    """What ``duplicate_dict`` returns: the reference's materialised copies (a plain dict for every caller), plus a note
    of what they are copies of.  ``run_model`` uses the note to encode each distinct spectrum once and repeat the result
    -- the reference's flow (run_batch_gen_val_MMT_v15_4.py:93-158) sends 128 identical spectra through the six encoder
    stacks.  The note is ignored as soon as any entry has been replaced or written to."""

    def _distinct(self):
        base, n, marks = self._mmt_base, self._mmt_n, self._mmt_marks
        if set(self.keys()) != set(marks):
            return None
        for k, (ident, version) in marks.items():
            v = dict.__getitem__(self, k)
            if id(v) != ident or v._version != version:
                return None
        return base, n


def duplicate_dict(data_dict, n_times):
    out = _DuplicatedDict({k: duplicate_tensor(v, n_times) for k, v in data_dict.items()})
    out._mmt_base = {k: v.detach().clone() for k, v in data_dict.items()}
    out._mmt_n = int(n_times)
    out._mmt_marks = {k: (id(v), v._version) for k, v in out.items()}
    return out


# ------------------------------------------------------------------- decoder
def _philox_advance(eng, n_candidates, n_total, max_len, per_memory_rng):
    """Generator offset consumed by one call: max_len torch.multinomial calls over all n_total sequences, or -- per-memory
    streams -- max_len calls over n_candidates rows for each of the n_total / n_candidates columns."""
    if per_memory_rng:
        return (n_total // n_candidates) * max_len * eng.philox_increment(n_candidates)
    return eng.philox_increment(n_total) * max_len


def _vocab(model, config):
    return _engine._desc_from(getattr(model, "config", config), _engine._normalize_state_dict(model.state_dict())).vocab


def _controls(model, config, n_cols, sampling, temperature, top_k, top_p):
    """Checked sampling controls for n_cols spectra (engine.sampling_controls), before any engine exists."""
    if temperature is None:
        temperature = float(config.temperature)
    return _engine.sampling_controls(n_cols, _vocab(model, config), temperature, top_k, top_p, sampling=sampling)


def _decode(model, memory, src_padding_mask, config, sampling, stop_on_all_pad, n_candidates, seq_index_base, n_total,
            per_memory_rng=False, eos=None, temperature=None, top_k=0, top_p=1.0):
    """eos: None, or the id at which a sequence stops being computed (Engine.decode_until_eos).  temperature / top_k /
    top_p: sampling controls per memory column (module docstring)."""
    if per_memory_rng and (sampling != "multinomial" or seq_index_base % n_candidates):
        raise ValueError("per_memory_rng needs multinomial sampling and seq_index_base a multiple of n_candidates")
    temperature, ctl = _controls(model, config, memory.size(1), sampling, temperature, top_k, top_p)
    if ctl is not None:
        temperature, top_k, top_p = ctl
    model.eval()                                    # the reference flips eval() and leaves it
    eng = _engine.engine_for(model, config)
    prec = _engine.default_precision(config)
    bias = _mask_to_bias(src_padding_mask.to(eng.device))
    N = memory.size(1) * n_candidates
    kw = {}
    gen = None
    if sampling == "multinomial":
        gen, seed, offset = _philox_state(eng.dev_index)
        kw = dict(seed=seed, offset=offset)
    if eos is not None:
        kw["eos"] = eos
    run = eng.decode if eos is None else eng.decode_until_eos
    if ctl is not None:
        kw.update(top_k=top_k, top_p=top_p)
    tokens, probs, steps = run(memory, bias, n_cand=n_candidates, max_len=int(config.max_len),
                               temperature=temperature, sampling=sampling,
                               stop_on_all_pad=stop_on_all_pad, precision=prec,
                               seq_index_base=seq_index_base, n_total=n_total, per_memory_rng=per_memory_rng, **kw)[:3]
    if gen is not None:   # consume exactly what the torch.multinomial calls would have
        gen.set_offset(offset + _philox_advance(eng, n_candidates, n_total if n_total else N, int(config.max_len), per_memory_rng))
    return tokens, probs, steps


def greedy_sequence(model, stoi, itos, memory, src_padding_mask, config, *, n_candidates=1, stop_at_eos=False):
    """-> ((T,N) i64 tokens without <SOS>, (T-1,N) f32 probs).  T < max_len only when one
    step emitted <PAD> for every sequence (stop_at_eos: or every sequence had emitted <EOS>).  NB the reference
    fails for N == 1 (SURVEY.md B.6); this returns the shapes its N > 1 code path would."""
    _check_sos(stoi)
    eos = _eos_id(stoi) if stop_at_eos else None
    tokens, probs, steps = _decode(model, memory, src_padding_mask, config, "greedy", True, n_candidates, 0, 0, eos=eos)
    return tokens[:steps], probs[1:steps]


def greedy_sequence_2(model, stoi, itos, memory, src_padding_mask, config, *, n_candidates=1, stop_at_eos=False):
    """mrtf variant: probabilities are NOT sliced -> ((T,N), (T,N))."""
    _check_sos(stoi)
    eos = _eos_id(stoi) if stop_at_eos else None
    tokens, probs, steps = _decode(model, memory, src_padding_mask, config, "greedy", True, n_candidates, 0, 0, eos=eos)
    return tokens[:steps], probs[:steps]


def multinomial_sequence(model, stoi, memory, src_padding_mask, config, *, n_candidates=1, seq_index_base=0, n_total=0,
                         per_memory_rng=False, stop_at_eos=False, temperature=None, top_k=0, top_p=1.0):
    """-> ((T,N) i64, (N,T) f32): probabilities transposed, always max_len steps."""
    _check_sos(stoi)
    eos = _eos_id(stoi) if stop_at_eos else None
    tokens, probs, _ = _decode(model, memory, src_padding_mask, config, "multinomial", False, n_candidates, seq_index_base, n_total,
                               per_memory_rng, eos=eos, temperature=temperature, top_k=top_k, top_p=top_p)
    return tokens, probs.transpose(0, 1)


def multinomial_sequence_multi(model, memory, src_padding_mask, stoi, config, *, n_candidates=1, seq_index_base=0, n_total=0,
                               per_memory_rng=False, stop_at_eos=False, temperature=None, top_k=0, top_p=1.0):
    """-> ((T,N) i64, (T,N) f32); the reference's .squeeze() drops the N axis of the
    probabilities when N == 1 (run_batch_gen_val_MMT_v15_4.py:149)."""
    _check_sos(stoi)
    eos = _eos_id(stoi) if stop_at_eos else None
    tokens, probs, _ = _decode(model, memory, src_padding_mask, config, "multinomial", False, n_candidates, seq_index_base, n_total,
                               per_memory_rng, eos=eos, temperature=temperature, top_k=top_k, top_p=top_p)
    if probs.shape[1] == 1:
        probs = probs.squeeze(1)
    return tokens, probs


def multinomial_sequence_multi_2(model, memory, src_padding_mask, stoi, config, *, n_candidates=1, seq_index_base=0, n_total=0,
                                 per_memory_rng=False, stop_at_eos=False, temperature=None, top_k=0, top_p=1.0):
    """mrtf variant: probabilities lose their first row -> ((T,N), (T-1,N))."""
    tokens, probs = multinomial_sequence_multi(model, memory, src_padding_mask, stoi, config, n_candidates=n_candidates,
                                               seq_index_base=seq_index_base, n_total=n_total, per_memory_rng=per_memory_rng,
                                               stop_at_eos=stop_at_eos, temperature=temperature, top_k=top_k, top_p=top_p)
    return tokens, probs[1:]


def teacher_forced_logits(model, memory, src_padding_mask, trg_SMI_input, config, *, n_candidates=1):
    """Decoder tail of forward(..., trg) (models_MMT_v15_4.py:955-976): (T,N) ids -> (T,N,V) logits."""
    eng = _engine.engine_for(model, config)
    bias = _mask_to_bias(src_padding_mask.to(eng.device))
    return eng.teacher_forced(memory, bias, trg_SMI_input, n_cand=n_candidates, precision=_engine.default_precision(config))


def beam_search(model, stoi, memory, src_padding_mask, config, beam_size):
    """validate_generate_MMT_v15_4.py:1058-1086: -> beams[item] = [(score, sequence, prob_sequence), ...] best first,
    ``config.gen_len`` steps from [<SOS>]; sequences keep their <SOS> and stop growing at <EOS>; score is the double
    product of the float32 probabilities under softmax(logits) (no temperature, :1038).  All items and beams advance
    together on the KV-cached decoder (the reference re-runs every beam's whole prefix, one item at a time)."""
    model.eval()
    sos = _check_sos(stoi)
    gen_len = int(config.gen_len)
    N = memory.size(1)
    if gen_len <= 0:
        return [[(1, [sos], [])] for _ in range(N)]
    eng = _engine.engine_for(model, config)
    bias = torch.zeros(N, memory.size(0), device=eng.device) if src_padding_mask is None else _mask_to_bias(src_padding_mask.to(eng.device))
    seq, ln, score, probs, _ = eng.beam_search(memory, bias, beam_size=int(beam_size), gen_len=gen_len, eos=int(stoi["<EOS>"]),
                                               precision=_engine.default_precision(config))
    seq, ln, score, probs = seq.cpu().tolist(), ln.cpu().tolist(), score.cpu().tolist(), probs.cpu().tolist()
    return [[(score[i][k], seq[i][k][:ln[i][k]], probs[i][k][:ln[i][k] - 1]) for k in range(len(seq[i]))] for i in range(N)]


def sample_without_replacement(model, stoi, memory, src_padding_mask, config, *, n_candidates, temperature=None,
                               seq_index_base=0, n_total=0):
    """``n_candidates`` DISTINCT sequences per spectrum in one call: stochastic beam search (Kool, van Hoof & Welling,
    ICML 2019) on the KV-cached decoder, an exact sample without replacement from the sequences ``multinomial_sequence``
    draws (cut at <EOS>) at ``temperature`` (a scalar or one per spectrum; None: config.temperature at call time), for
    ``config.max_len`` steps.  Candidate n = spectrum * n_candidates + slot; within a spectrum the slots are ordered by
    their Gumbel key, so slot 0 is an ordinary sample and slot j a sample from what slots 0..j-1 left.
    -> (tokens (T,N) i64 without <SOS>, <PAD> after <EOS>; probs (T,N) f32 of each chosen token, 0 after <EOS>;
        log_prob (N,) f64 = sum of log(probs); key (N,) f64, descending per spectrum).  Fewer than n_candidates
    possible sequences (tiny max_len): the remaining slots are empty (<PAD> only, log_prob = key = -inf).
    The noise follows torch's CUDA generator in per-memory streams (``per_memory_rng``): seq_index_base (a multiple of
    n_candidates) / n_total place the call inside a larger logical batch; the generator advances by
    (n_total or N) / n_candidates * max_len exponential_ calls of n_candidates x vocab elements."""
    _check_sos(stoi)
    if "<EOS>" not in stoi:
        raise ValueError("sample_without_replacement needs an <EOS> entry in stoi")
    eos = int(stoi["<EOS>"])
    if isinstance(n_candidates, bool) or not isinstance(n_candidates, int) or not 1 <= n_candidates <= 128:
        raise ValueError(f"n_candidates must be an integer in [1, 128], got {n_candidates!r}")
    k = n_candidates
    Bm = memory.size(1)
    if not isinstance(seq_index_base, int) or seq_index_base < 0 or seq_index_base % k:
        raise ValueError("seq_index_base must be a non-negative multiple of n_candidates")
    if n_total and (n_total % k or n_total < seq_index_base + Bm * k):
        raise ValueError("n_total must be a multiple of n_candidates covering seq_index_base + the call's sequences")
    if temperature is None:
        temperature = float(config.temperature)
    temperature = _engine.control_arrays(Bm, _vocab(model, config), temperature)[0]
    max_len = int(config.max_len)
    model.eval()
    eng = _engine.engine_for(model, config)
    bias = _mask_to_bias(src_padding_mask.to(eng.device))
    gen, seed, offset = _philox_state(eng.dev_index)
    tokens, probs, _, log_prob, key, _ = eng.sample_without_replacement(
        memory, bias, n_cand=k, max_len=max_len, temperature=temperature, eos=eos, seed=seed, offset=offset,
        seq_index_base=seq_index_base, n_total=n_total, precision=_engine.default_precision(config))
    gen.set_offset(offset + _philox_advance(eng, k, n_total if n_total else Bm * k, max_len, True))
    return tokens, probs, log_prob, key


# ------------------------------------------------------------- teacher-forced scorers
def _scorer_inputs(stoi, trg_enc_SMI, device):
    """real_trg = trg_enc_SMI^T[1:] (validate_generate_MMT_v15_4.py:336-338); the decoder sees [<SOS>, real_trg[:-1]]."""
    sos = _check_sos(stoi)
    real_trg = trg_enc_SMI.to(device).transpose(0, 1)[1:, :].contiguous()
    trg_in = torch.cat([torch.full((1, real_trg.shape[1]), sos, dtype=torch.long, device=device), real_trg[:-1]], dim=0)
    return real_trg, trg_in


def predict_prop_correct_max_sequence_2(model, stoi, memory, src_padding_mask, trg_enc_SMI, config):
    """-> (trg_tensor (N,L) i64, corr_token_prob (L,N), trg_tensor_max (N,L) i64, max_token_prob (L,N)): at every position
    of the teacher-forced target the probability of the correct token, the arg-max token and its probability under
    softmax(logits / config.temperature).  One KV-cached pass; the reference re-runs the decoder on every prefix.  Like
    the reference's .squeeze(), the probability tensors lose their N axis when N == 1."""
    model.eval()
    eng = _engine.engine_for(model, config)
    real_trg, trg_in = _scorer_inputs(stoi, trg_enc_SMI, eng.device)
    bias = _mask_to_bias(src_padding_mask.to(eng.device))
    pick, pick_prob, corr = eng.teacher_forced_scores(memory, bias, trg_in, real_trg, temperature=float(config.temperature),
                                                      precision=_engine.default_precision(config))
    if real_trg.shape[1] == 1:
        corr, pick_prob = corr.squeeze(1), pick_prob.squeeze(1)
    return real_trg.transpose(0, 1), corr, pick.transpose(0, 1), pick_prob


predict_prop_correct_max_sequence_3 = predict_prop_correct_max_sequence_2      # identical bodies in the reference


def predict_prop_correct_max_sequence(model, stoi, memory, src_padding_mask, trg_enc_SMI, gen_num, config):
    """The five-output variant (validate_generate_MMT_v15_4.py:309-432): additionally the probability of one multinomial
    draw per position under the teacher-forced context, flattened to (L*N,) like the reference's .view(1,-1).squeeze(0)
    (gen_num is overwritten with 1 there, :386).  Draws follow torch.multinomial's CUDA Philox stream: L calls."""
    if memory.size(1) != 1:    # the reference only runs for N == 1: torch.tensor(list of (N,) tensors) raises at :415
        raise ValueError("only one element tensors can be converted to Python scalars")
    out = predict_prop_correct_max_sequence_2(model, stoi, memory, src_padding_mask, trg_enc_SMI, config)
    eng = _engine.engine_for(model, config)
    real_trg, trg_in = _scorer_inputs(stoi, trg_enc_SMI, eng.device)
    bias = _mask_to_bias(src_padding_mask.to(eng.device))
    gen, seed, offset = _philox_state(eng.dev_index)
    _, mprob, _ = eng.teacher_forced_scores(memory, bias, trg_in, None, temperature=float(config.temperature), sampling="multinomial",
                                            precision=_engine.default_precision(config), seed=seed, offset=offset)
    gen.set_offset(offset + eng.philox_increment(real_trg.shape[1]) * real_trg.shape[0])
    return out + (mprob.reshape(-1),)
