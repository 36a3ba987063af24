"""CPU restatement of the MMT candidate-generation path.  TEST INFRASTRUCTURE.

This module is the *checker* for the CUDA engine: a plain-PyTorch (fp32)
restatement of the reference's encoder and SMILES decode loops, written out
op by op (explicit projections, softmax, layer norm) instead of through
``nn.Transformer*``.  Only ``tests/``, ``__graft_entry__.smoke()`` and
``bench.py``'s CPU-baseline legs may import it; the product package never does.

Parity status: the reference ships no tests or golden vectors for this path
(SURVEY.md 8c), so the restatement is pinned against the reference's own code
executed in the build container on seeded random-init weights and synthetic
spectra -- ``oracle/make_golden.py`` generates ``tests/golden/*.npz`` from the
shimmed reference and ``tests/test_oracle_golden.py`` checks this file against
them.

Citations are relative to /root/reference/utils_MMT/.  The attention math the
reference executes lives in PyTorch (third-party, pinned torch==1.9.1+cu111 in
installs.sh:21; torch 2.11 here): nn.TransformerEncoderLayer/DecoderLayer with
batch_first=False, norm_first=False, ReLU, eps=1e-5, i.e. torch's
``_sa_block/_mha_block/_ff_block`` -> ``F.multi_head_attention_forward`` ->
``scaled_dot_product_attention`` with key-padding and causal masks merged by
addition.
"""
from __future__ import annotations

import math
from types import SimpleNamespace

import torch
import torch.nn as nn
import torch.nn.functional as F

D = 128
FUSED_SDPA = True   # False: spelled-out softmax(QK^T/sqrt(dh)+bias)V, same math (tests check both)
MODALITIES = ("1H", "13C", "HSQC", "COSY", "IR")
_EMBED_KEYS = {
    "1H": "linear_spec_embedding_1H.point_embedding_layer_1H.fc_H",
    "13C": "linear_spec_embedding_13C.point_embedding_layer_13C.fc_C",
    "HSQC": "linear_spec_embedding_HSQC.point_embedding_layer_HSQC.fc_HSQC",
    "COSY": "linear_spec_embedding_COSY.point_embedding_layer_COSY.fc_COSY",
    "IR": "linear_spec_embedding_IR.linear_spec_embedding_IR",
}


def default_config(**over):
    """The hot-path subset of config_V8.json (utils_MMT/config_V8.json:1)."""
    c = dict(hidden_size=128, num_heads=16, num_encoder_layers=6, num_decoder_layers=6,
             in_size=43, out_size=43, max_len=128, drop_out=0.1, fingerprint_size=512,
             input_dim_1H=2, input_dim_13C=1, input_dim_HSQC=2, input_dim_COSY=2,
             input_dim_IR=1000, MF_vocab_size=212, MS_vocab_size=43,
             training_mode="1H_13C_HSQC_COSY_IR_MF_MW", temperature=1, use_real_data=False,
             device="cpu")
    c.update(over)
    return SimpleNamespace(**c)


def random_init_state_dict(config, seed=0):
    """Seeded default-PyTorch init in the reference's construction order
    (models_MMT_v15_4.py:494-546), so that ``torch.manual_seed(seed)`` yields the
    same 25,566,294 parameters as ``MultimodalTransformer(config)``."""
    import warnings
    torch.manual_seed(seed)
    h = config.hidden_size
    mods = {}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        mods[_EMBED_KEYS["1H"]] = nn.Linear(config.input_dim_1H, h)
        mods[_EMBED_KEYS["13C"]] = nn.Linear(config.input_dim_13C, h)
        mods[_EMBED_KEYS["HSQC"]] = nn.Linear(config.input_dim_HSQC, h)
        mods[_EMBED_KEYS["COSY"]] = nn.Linear(config.input_dim_COSY, h)
        mods[_EMBED_KEYS["IR"]] = nn.Linear(config.input_dim_IR, h)
        mods["linear_embedding_MF.embedding"] = nn.Embedding(config.MF_vocab_size, h, padding_idx=0)
        mods["linear_embedding_MS.embedding"] = nn.Embedding(config.MS_vocab_size, h, padding_idx=0)
        mods["linear_embedding_MW.linear_spec_embedding_MW"] = nn.Linear(1, h)
        mods["embed_trg"] = nn.Embedding(config.in_size, h)
        mods["pe_trg"] = nn.Embedding(config.max_len, h)
        for m in MODALITIES:
            mods[f"encoder_{m}"] = nn.TransformerEncoder(
                nn.TransformerEncoderLayer(d_model=h, nhead=config.num_heads),
                num_layers=config.num_encoder_layers)
        mods["encoder_cross"] = nn.TransformerEncoder(
            nn.TransformerEncoderLayer(d_model=h, nhead=int(config.num_heads / 4)),
            num_layers=config.num_encoder_layers)
        mods["decoder"] = nn.TransformerDecoder(
            nn.TransformerDecoderLayer(d_model=h, nhead=config.num_heads),
            num_layers=config.num_decoder_layers)
        mods["fp1"] = nn.Linear(h, config.fingerprint_size)
        mods["fc_out"] = nn.Linear(h, config.out_size)
        mods["real_data_linear"] = nn.Linear(h, config.out_size)
    sd = {}
    for prefix, mod in mods.items():
        for k, v in mod.state_dict().items():
            sd[f"{prefix}.{k}"] = v.detach().clone()
    return sd


# --------------------------------------------------------------------------
# building blocks
# --------------------------------------------------------------------------
def _mha(P, prefix, nhead, x_q, x_kv, attn_bias):
    """Multi-head attention, seq-first.  x_q (Tq,B,D), x_kv (Tk,B,D);
    ``attn_bias`` broadcastable to (B,1|H,Tq,Tk), added to the scaled scores
    (torch functional.py multi_head_attention_forward; scale 1/sqrt(dh) on QK^T,
    softmax in fp32; cross-attention takes Q from in_proj[:D], K,V from in_proj[D:])."""
    Tq, B, _ = x_q.shape
    Tk = x_kv.shape[0]
    W, b = P[f"{prefix}.in_proj_weight"], P[f"{prefix}.in_proj_bias"]
    q = F.linear(x_q, W[:D], b[:D])
    k = F.linear(x_kv, W[D:2 * D], b[D:2 * D])
    v = F.linear(x_kv, W[2 * D:], b[2 * D:])
    dh = D // nhead
    q = q.reshape(Tq, B, nhead, dh).permute(1, 2, 0, 3)
    k = k.reshape(Tk, B, nhead, dh).permute(1, 2, 0, 3)
    v = v.reshape(Tk, B, nhead, dh).permute(1, 2, 0, 3)
    if attn_bias is not None:
        # in q's dtype: torch's CPU SDPA returns wrong values, without an error, for float64 q/k/v with a float32 mask
        attn_bias = attn_bias.to(q.dtype)
        attn_bias = attn_bias.expand(B, nhead, Tq, Tk) if attn_bias.dim() == 4 else attn_bias
    if FUSED_SDPA:
        # what the reference executes: torch's fused scaled_dot_product_attention (float additive mask)
        o = F.scaled_dot_product_attention(q, k, v, attn_mask=attn_bias)
    else:
        s = torch.matmul(q, k.transpose(-1, -2)) * (1.0 / math.sqrt(dh))
        if attn_bias is not None:
            s = s + attn_bias
        o = torch.matmul(torch.softmax(s, dim=-1), v)
    o = o.permute(2, 0, 1, 3).reshape(Tq, B, D)
    return F.linear(o, P[f"{prefix}.out_proj.weight"], P[f"{prefix}.out_proj.bias"])


def _ln(P, prefix, x):
    return F.layer_norm(x, (D,), P[f"{prefix}.weight"], P[f"{prefix}.bias"], 1e-5)


def _ffn(P, prefix, x):
    return F.linear(F.relu(F.linear(x, P[f"{prefix}.linear1.weight"], P[f"{prefix}.linear1.bias"])),
                    P[f"{prefix}.linear2.weight"], P[f"{prefix}.linear2.bias"])


def key_padding_bias(mask):
    """(B,S) key-padding mask -> additive (B,1,1,S) float bias.  bool: True -> -inf.
    Float masks are ADDED as they are -- the reference's blank-modality branch
    builds float ``ones`` masks (models_MMT_v15_4.py:852-854) so that, after
    torch.cat promotes the whole mask to float, pads get +1.0 rather than -inf
    (SURVEY.md B.2)."""
    if mask.dtype == torch.bool:
        bias = torch.zeros(mask.shape, dtype=torch.float32, device=mask.device)
        bias = bias.masked_fill(mask, float("-inf"))
    elif mask.is_floating_point():
        bias = mask.to(torch.float32)
    else:
        raise AssertionError("only bool and floating types of key_padding_mask are supported")
    return bias[:, None, None, :]


def encoder_stack(P, name, nhead, x, mask, num_layers):
    """nn.TransformerEncoder of post-norm layers, no final norm
    (models_MMT_v15_4.py:510-533; torch transformer.py _sa_block/_ff_block)."""
    bias = key_padding_bias(mask)
    for l in range(num_layers):
        p = f"{name}.layers.{l}"
        x = _ln(P, f"{p}.norm1", x + _mha(P, f"{p}.self_attn", nhead, x, x, bias))
        x = _ln(P, f"{p}.norm2", x + _ffn(P, p, x))
    return x


def decoder_stack(P, nhead, x, memory, tgt_bias, mem_mask, num_layers):
    """nn.TransformerDecoder, post-norm: self-attn(causal) -> LN1 -> cross-attn
    (memory key padding) -> LN2 -> FFN -> LN3 (models_MMT_v15_4.py:539-541)."""
    mbias = key_padding_bias(mem_mask)
    for l in range(num_layers):
        p = f"decoder.layers.{l}"
        x = _ln(P, f"{p}.norm1", x + _mha(P, f"{p}.self_attn", nhead, x, x, tgt_bias))
        x = _ln(P, f"{p}.norm2", x + _mha(P, f"{p}.multihead_attn", nhead, x, memory, mbias))
        x = _ln(P, f"{p}.norm3", x + _ffn(P, p, x))
    return x


def causal_bias(T, device):
    """0 / -inf upper-triangular float mask (models_MMT_v15_4.py:794-800)."""
    m = torch.full((T, T), float("-inf"), device=device)
    return torch.triu(m, diagonal=1)


# --------------------------------------------------------------------------
# encoder  ==  vgmmt.run_model  ==  MultimodalTransformer.forward(trg=None)
# --------------------------------------------------------------------------
def encode(P, data, config):
    """validate_generate_MMT_v15_4.py:95-267 / models_MMT_v15_4.py:803-953.

    Computes in the dtype of the weights (fp32 as the reference; float64 weights give the fp64 oracle).
    Returns (memory (S,B,D), src_padding_mask (B,S) bool-or-float,
    fingerprint (B,512), embedding_src (S,B,D))."""
    mode = config.training_mode
    dev, dt = P["fc_out.weight"].device, P["fc_out.weight"].dtype
    g = lambda k: data[k].to(dev)
    nL, H = config.num_encoder_layers, config.num_heads
    B = None
    emb, msk = {}, {}
    for m in ("1H", "13C", "HSQC", "COSY"):
        if m in mode:                                                  # :733-759
            x = g(f"src_{m}").to(dt)
            if m == "13C":
                x = x.unsqueeze(-1)
            W, b = P[_EMBED_KEYS[m] + ".weight"], P[_EMBED_KEYS[m] + ".bias"]
            e = F.relu(F.relu(F.linear(x, W, b)))                      # ReLU twice (:401 + :735)
            emb[m] = e.permute(1, 0, 2)
            msk[m] = g(f"mask_{m}").to(torch.bool)
            B = e.shape[0]
    if "IR" in mode:                                                   # :761-767, :827-828
        x = g("src_IR").to(dt)
        e = F.relu(F.linear(x, P[_EMBED_KEYS["IR"] + ".weight"], P[_EMBED_KEYS["IR"] + ".bias"]))
        emb["IR"] = e.unsqueeze(0)
        msk["IR"] = torch.zeros(e.shape[0], 1, dtype=torch.bool, device=dev)
    extra = []
    if "MF" in mode:                                                   # :769-776 (mask passed through)
        e = F.relu(F.embedding(g("src_MF"), P["linear_embedding_MF.embedding.weight"]))
        extra.append((e.permute(1, 0, 2), g("mask_MF")))
    if "MS" in mode:                                                   # :778-785
        e = F.relu(F.embedding(g("src_MS"), P["linear_embedding_MS.embedding.weight"]))
        extra.append((e.permute(1, 0, 2), g("mask_MS")))
    if "MW" in mode:                                                   # :787-792, :804, :830-831
        mw = g("trg_MW").to(dt).unsqueeze(1)
        e = F.relu(F.linear(mw, P["linear_embedding_MW.linear_spec_embedding_MW.weight"],
                            P["linear_embedding_MW.linear_spec_embedding_MW.bias"]))
        extra.append((e.unsqueeze(0), torch.zeros(mw.shape[0], 1, dtype=torch.bool, device=dev)))

    fdim = 193 if "MS" in mode else 129
    fdim_ir = 130 if "MS" in mode else 66
    mems, embs, masks = [], [], []
    for m in MODALITIES:
        if m in emb:                                                   # :549-731 cat order X|MF|MS|MW
            x = torch.cat([emb[m]] + [e for e, _ in extra], dim=0)
            k = torch.cat([msk[m]] + [mm for _, mm in extra], dim=1)
            mems.append(encoder_stack(P, f"encoder_{m}", H, x, k, nL))
            embs.append(x)
            masks.append(k)
        else:                                                          # :850-858 ... :931-939
            n = {"COSY": 65, "IR": fdim_ir}.get(m, fdim)
            mems.append(torch.zeros(n, B, D, device=dev, dtype=dt))
            embs.append(torch.zeros(n, B, D, device=dev, dtype=dt))
            if m == "IR":
                masks.append(torch.zeros(B, n, dtype=torch.bool, device=dev))
            else:
                masks.append(torch.ones(B, n, device=dev))             # float "mask"
    memory = torch.cat(mems, dim=0)                                    # :941
    embedding_src = torch.cat(embs, dim=0)
    mask = torch.cat(masks, dim=1)                                     # dtype promotion bool->float
    memory = encoder_stack(P, "encoder_cross", int(H / 4), memory, mask, nL)   # :944
    fingerprint = F.linear(memory.mean(dim=0), P["fp1.weight"], P["fp1.bias"])  # :946-948
    return memory, mask, fingerprint, embedding_src


# --------------------------------------------------------------------------
# decoder loops
# --------------------------------------------------------------------------
def _embed_target(P, tokens):
    T = tokens.shape[0]
    pos = torch.arange(T, device=tokens.device).unsqueeze(1).expand_as(tokens)
    return F.embedding(tokens, P["embed_trg.weight"]) + F.embedding(pos, P["pe_trg.weight"])


def teacher_forced_logits(P, memory, mask, tokens, config):
    """forward(..., trg_SMI_input) tail: models_MMT_v15_4.py:955-976 (use_real_data False).
    tokens (T,N) i64 -> logits (T,N,V)."""
    x = _embed_target(P, tokens)                     # dropout2 is identity in eval
    out = decoder_stack(P, config.num_heads, x, memory, causal_bias(tokens.shape[0], tokens.device),
                        mask, config.num_decoder_layers)
    return F.linear(out, P["fc_out.weight"], P["fc_out.bias"])


def _decode_loop(P, memory, mask, config, pick, stop_on_all_pad, sos=3, max_len=None, margins=None):
    """Shared body of greedy_sequence / multinomial_sequence(_multi): every step
    re-runs the decoder on the whole prefix and samples from position -1
    (validate_generate_MMT_v15_4.py:744-764, 861-875).  ``margins`` (a list) receives, per step, the (N,) top-2 logit
    margin of position -1 relative to the row's max |logit| (test bookkeeping for the near-tie rules; not reference code)."""
    N = memory.shape[1]
    dev = memory.device
    tokens = torch.full((1, N), sos, dtype=torch.long, device=dev)
    probs = []
    for _ in range(max_len or config.max_len):
        logits = teacher_forced_logits(P, memory, mask, tokens, config)
        if margins is not None:
            top2 = torch.topk(logits[-1], 2, dim=1).values
            margins.append((top2[:, 0] - top2[:, 1]) / logits[-1].abs().amax(dim=1))
        p = torch.softmax(logits[-1] / config.temperature, dim=1)
        nxt = pick(p)
        probs.append(p.gather(1, nxt.unsqueeze(1)).squeeze(1))
        tokens = torch.cat([tokens, nxt.unsqueeze(0)], dim=0)
        if stop_on_all_pad and bool((nxt == 0).all()):
            break
    return tokens[1:], torch.stack(probs)


def greedy_sequence(P, memory, mask, config, max_len=None):
    """validate_generate_MMT_v15_4.py:723-775 -> ((T,N) i64, (T-1,N) f32)."""
    tok, pr = _decode_loop(P, memory, mask, config, lambda p: torch.argmax(p, dim=1), True, max_len=max_len)
    return tok, pr[1:]


def greedy_sequence_with_margins(P, memory, mask, config, max_len=None):
    """greedy_sequence plus the relative top-2 logit margin of every pick: ((T,N) i64, (T-1,N) f32, (T,N) f32)."""
    m = []
    tok, pr = _decode_loop(P, memory, mask, config, lambda p: torch.argmax(p, dim=1), True, max_len=max_len, margins=m)
    return tok, pr[1:], torch.stack(m)


def multinomial_sequence(P, memory, mask, config, generator=None, max_len=None):
    """validate_generate_MMT_v15_4.py:841-880 -> ((T,N) i64, (N,T) f32)."""
    pick = lambda p: torch.multinomial(p, 1, generator=generator).squeeze(1)
    tok, pr = _decode_loop(P, memory, mask, config, pick, False, max_len=max_len)
    return tok, pr.transpose(0, 1)


def multinomial_sequence_multi(P, memory, mask, config, generator=None, max_len=None):
    """run_batch_gen_val_MMT_v15_4.py:121-158 -> ((T,N) i64, (T,N) f32)."""
    pick = lambda p: torch.multinomial(p, 1, generator=generator).squeeze(1)
    return _decode_loop(P, memory, mask, config, pick, False, max_len=max_len)


# --------------------------------------------------------------------------
# sampling RNG restatement (SURVEY.md appendix D) -- numpy, bit-exact integers
# --------------------------------------------------------------------------
def predict_prop_correct_max_sequence_2(P, memory, mask, trg_enc_SMI, config, sos=3):
    """validate_generate_MMT_v15_4.py:434-509 (= mmt_result_test_functions_15_4.py:340-400), with the reference's
    full-prefix decoder run per position.  -> (trg (N,L), corr_prob (L,N), trg_max (N,L), max_prob (L,N))."""
    N = memory.size(1)
    real_trg = trg_enc_SMI.transpose(0, 1)[1:, :]
    trg = torch.full((1, N), sos, dtype=torch.long)
    trg_max = torch.full((1, N), sos, dtype=torch.long)
    corr, mx = [], []
    for idx in range(real_trg.shape[0]):
        logits = teacher_forced_logits(P, memory, mask, trg, config)
        probs = torch.softmax(logits / config.temperature, dim=2)
        nxt = torch.argmax(probs[-1], dim=1)
        mx.append(probs[-1].gather(1, nxt.unsqueeze(-1)).squeeze())
        trg_max = torch.cat((trg_max, nxt.unsqueeze(0)), dim=0)
        corr.append(probs[-1].gather(1, real_trg[idx].unsqueeze(-1)).squeeze())
        trg = torch.cat((trg, real_trg[idx].unsqueeze(0)), dim=0)
    return trg.transpose(0, 1)[:, 1:], torch.stack(corr), trg_max.transpose(0, 1)[:, 1:], torch.stack(mx)


def beam_search(P, memory, mask, config, beam_size, gen_len, sos=3, eos=2):
    """validate_generate_MMT_v15_4.py:995-1086 (beam_search_step + beam_search), per item, full-prefix decoder runs.
    Returns beams[item] = [(score, sequence, prob_sequence), ...] sorted by score, like the reference.
    NB the reference ranks with softmax(logits) WITHOUT the temperature (:1038) and multiplies Python floats (double)."""
    N = memory.size(1)
    beams = [[(1, [sos], [])] for _ in range(N)]
    for _ in range(gen_len):
        new_beams = []
        for i in range(N):
            mem_i, mask_i = memory[:, i:i + 1, :], mask[i:i + 1]
            new_beam, seen = [], set()
            for score, seq, pseq in beams[i]:
                if tuple(seq) in seen:
                    continue
                seen.add(tuple(seq))
                if seq[-1] == eos:
                    new_beam.append((score, seq, pseq))
                    continue
                trg = torch.tensor(seq, dtype=torch.long).unsqueeze(1)
                logits = teacher_forced_logits(P, mem_i, mask_i, trg, config)
                probs = torch.softmax(logits[-1, :, :], dim=-1)
                top_p, top_i = torch.topk(probs, beam_size, dim=-1)
                for k in range(beam_size):
                    ns = seq + [top_i[0, k].item()]
                    if tuple(ns) in seen:
                        continue
                    seen.add(tuple(ns))
                    new_beam.append((score * top_p[0, k].item(), ns, pseq + [top_p[0, k].item()]))
            new_beam.sort(key=lambda x: x[0], reverse=True)
            new_beams.append(new_beam[:beam_size])
        beams = new_beams
    return beams


def philox4x32_10(counter, key):
    """Philox4x32-10 (Salmon et al., Random123) as used by curand's
    curandStatePhilox4_32_10: counter (..,4) uint32, key (..,2) uint32 -> (..,4)."""
    import numpy as np
    c = [np.asarray(counter[..., i], dtype=np.uint64) for i in range(4)]
    k0 = np.asarray(key[..., 0], dtype=np.uint64)
    k1 = np.asarray(key[..., 1], dtype=np.uint64)
    M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    W0, W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = M0 * c[0]
        p1 = M1 * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & mask
        hi1, lo1 = p1 >> np.uint64(32), p1 & mask
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + W0) & mask
        k1 = (k1 + W1) & mask
    return np.stack([x.astype(np.uint32) for x in c], axis=-1)


def cuda_exponential_like(numel, seed, offset, sm_count=148, max_threads_per_sm=2048):
    """What ``torch.empty(numel, device='cuda').exponential_(1)`` writes for Philox
    state (seed, offset): torch DistributionTemplates.h distribution_nullary_kernel
    (block 256, grid capped at SMs*(maxThreadsPerSM/256), unroll 4, curand_uniform4,
    transform -log(u) with the u~1 guard of TransformationHelper.h).  The device
    evaluates the log with the fast __logf (ATen/NumericUtils.h:150-160); numpy's log
    is correctly rounded, so values agree to a few ulp, not bit for bit.  Returns
    (float32[numel], counter_offset_increment)."""
    import numpy as np
    block = 256
    grid = min(sm_count * (max_threads_per_sm // block), (numel + block - 1) // block)
    threads = block * grid
    inc = ((numel - 1) // (threads * 4) + 1) * 4
    li = np.arange(numel, dtype=np.int64)
    it = li // (threads * 4)
    comp = (li % (threads * 4)) // threads
    idx = li % threads
    off4 = (offset // 4) + it
    ctr = np.stack([off4 & 0xFFFFFFFF, off4 >> 32, idx & 0xFFFFFFFF, idx >> 32], axis=-1).astype(np.uint32)
    key = np.broadcast_to(np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32), (numel, 2))
    r = philox4x32_10(ctr, key)
    x = r[np.arange(numel), comp]
    u = x.astype(np.float32) * np.float32(2.3283064365386963e-10) + np.float32(2.3283064365386963e-10 / 2.0)
    eps = np.float32(np.finfo(np.float32).eps)
    lg = np.where(u >= np.float32(1.0) - eps / np.float32(2), -eps / np.float32(2), np.log(u, dtype=np.float32))
    return (np.float32(-1.0) * lg).astype(np.float32), inc


def cuda_multinomial_like(p, seed, offset, sm_count=148, max_threads_per_sm=2048):
    """torch.multinomial(p, 1) on CUDA == argmax(p / Exp(1)) with first-index ties
    (torch Distributions multinomial fast path).  p (N,V) float32 numpy."""
    import numpy as np
    q, inc = cuda_exponential_like(p.size, seed, offset, sm_count, max_threads_per_sm)
    r = p.astype(np.float32) / q.reshape(p.shape)
    return np.argmax(r, axis=1), inc
