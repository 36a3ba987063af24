"""The engine against fp64 references on trained-like weights.

PyTorch's default init leaves 276 of the 562 state-dict tensors constant: every attention in_proj_bias / out_proj.bias
and LayerNorm bias is 0, every LayerNorm weight is 1.  With those weights a bias dropped or taken from another block, or a
LayerNorm affine read from the wrong slot or layer, gives bit-identical output.  A trained checkpoint has distinct values
in all of them, so these tests draw them (`trained_state_dict`): in_proj_bias / out_proj.bias 0.1 N(0,1), norm weight
1 + 0.2 N(0,1), norm bias 0.1 N(0,1), every tensor independently; everything else keeps the seed-0 init.  Test files that
take a `weights` parameter ("init" / "trained") get their weights and engines from `state_dict_for` / `engine_with`.

CPU (no GPU needed):
(a) the oracle's encoder and decoder stacks equal torch's nn.TransformerEncoder / nn.TransformerDecoder in fp64 on these
    weights, with the fused SDPA and with the spelled-out softmax;
(b) every numeric-only fault of a bias or LayerNorm parameter that the GPU tests are meant to see leaves their bound:
    decoder faults move the teacher-forced logits past 1e-2 of the row scale on > 90 % of rows, encoder faults move the
    fp64 bf16 contract past 3e-3 (rms error / rms) for every spectrum.  The K bias is left out: it adds q.b_k to every
    score of a row, and softmax does not change when every score shifts by the same amount.
GPU:
(c) teacher-forced logits, all 128 positions, at the small-wave geometries (fused decode_attn with the norm3 fold, bf16 and
    fp32; the cluster FFN) -- the large-wave geometries run in test_gpu_large_wave with both weight sets;
(d) beam search in fp32 against oracle.beam_search, fused and un-fused kernels;
(e) the decode layer tail (`mmt_decode_layer_tail`: out-proj + norm1, cross-attention query, cross out-proj + norm2,
    FFN + norm3) element by element against an fp64 evaluation of the bf16 contract, every variant of the un-fused step."""
import copy

import pytest
import torch
import torch.nn.functional as F

D = 128


# --------------------------------------------------------------------------------------------------------- weights
_W = {}


def trained_state_dict():
    """fp64 state dict (CPU): the seed-0 init with every attention bias and LayerNorm affine drawn independently from a
    fixed generator.  Values are fp32-representable, so the engine's fp32 copy holds them exactly."""
    if "P64" not in _W:
        from oracle import mmt_oracle as O
        sd = O.random_init_state_dict(O.default_config(), seed=0)
        g = torch.Generator().manual_seed(0)
        for k in sd:                      # state-dict order
            v = sd[k]
            if k.endswith(("in_proj_bias", "out_proj.bias")):
                sd[k] = 0.1 * torch.randn(v.shape, generator=g)
            elif ".norm" in k and k.endswith(".weight"):
                sd[k] = 1 + 0.2 * torch.randn(v.shape, generator=g)
            elif ".norm" in k and k.endswith(".bias"):
                sd[k] = 0.1 * torch.randn(v.shape, generator=g)
        _W["P64"] = {k: v.float().double() for k, v in sd.items()}
    return _W["P64"]


def state_dict_for(weights, dtype=torch.float32, device="cuda"):
    """State dict of the weight set "init" (the model every GPU test builds, torch.manual_seed(0)) or "trained"."""
    if weights == "init":
        from test_gpu_parity import setup
        sd = setup()["model"].state_dict()
    else:
        sd = trained_state_dict()
    return {k: v.detach().to(device, dtype) for k, v in sd.items()}


def engine_with(weights, **env):
    """A new Engine on the weight set, created with the engine knobs `env` (read at creation).  Not cached: an engine
    keeps the arena of the largest wave it ran, tens of GB for the bench wave."""
    import os
    from test_gpu_parity import setup
    from multimodalspectraltransformer_b200.engine import Engine
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        return Engine(state_dict_for(weights), setup()["cfg"], "cuda")
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


def trained_model():
    """The test model (test_gpu_parity.setup) with the trained-like weights loaded: public calls (run_model,
    teacher_forced_logits, beam_search) reach it through engine_for."""
    if "model" not in _W:
        from test_gpu_parity import setup
        m = copy.deepcopy(setup()["model"])
        m.load_state_dict(state_dict_for("trained"))
        m.eval()
        _W["model"] = m
    return _W["model"]


def with_weights(values):
    """Parameters (value, weights) for a test's innermost parametrization: each value with the init weights under its
    own id, and with the trained-like weights as "<value>-trained"."""
    return ([pytest.param(v, "init", id=str(v)) for v in values] +
            [pytest.param(v, "trained", id=f"{v}-trained") for v in values])


def test_trained_weights_have_no_constant_vector():
    """No 1-D parameter is constant (under the init, 276 tensors are), and the drawn ones differ between layers."""
    P = trained_state_dict()
    const = [k for k, v in P.items() if v.dim() == 1 and v.numel() > 1 and bool((v == v[0]).all())]
    assert not const, const[:10]
    assert not torch.equal(P["decoder.layers.0.norm3.weight"], P["decoder.layers.1.norm3.weight"])
    assert not torch.equal(P["decoder.layers.2.norm2.bias"], P["decoder.layers.2.norm3.bias"])
    assert float(P["encoder_cross.layers.5.norm1.weight"].std()) > 0.1


# --------------------------------------------------------------------------------------------------------- faults
def with_fault(P, prefix, kind):
    """Copy of the state dict P with one fault in the layer `prefix` (e.g. "decoder.layers.3"):
    swap_n2n3 / swap_n1n2: the two LayerNorms exchanged;
    drop_n2_beta; drop_out_bias / drop_ca_out_bias: self / cross out_proj.bias zero; drop_v_bias / drop_ca_v_bias,
    drop_q_bias / drop_ca_q_bias: that third of in_proj_bias zero; ca_q_from_self: the cross query bias taken from the
    self-attention's."""
    P = dict(P)
    z = lambda k: P.__setitem__(k, torch.zeros_like(P[k]))

    def part(k, lo, hi, src=None):
        t = P[k].clone()
        t[lo:hi] = 0 if src is None else src[lo:hi]
        P[k] = t
    sa, ca = f"{prefix}.self_attn", f"{prefix}.multihead_attn"
    if kind in ("swap_n2n3", "swap_n1n2"):
        a, b = ("norm2", "norm3") if kind == "swap_n2n3" else ("norm1", "norm2")
        for t in ("weight", "bias"):
            P[f"{prefix}.{a}.{t}"], P[f"{prefix}.{b}.{t}"] = P[f"{prefix}.{b}.{t}"], P[f"{prefix}.{a}.{t}"]
    elif kind == "drop_n2_beta":
        z(f"{prefix}.norm2.bias")
    elif kind == "drop_out_bias":
        z(f"{sa}.out_proj.bias")
    elif kind == "drop_ca_out_bias":
        z(f"{ca}.out_proj.bias")
    elif kind in ("drop_q_bias", "drop_ca_q_bias", "drop_v_bias", "drop_ca_v_bias"):
        lo = 0 if "_q_" in kind else 2 * D
        part(f"{ca if '_ca_' in kind else sa}.in_proj_bias", lo, lo + D)
    elif kind == "ca_q_from_self":
        part(f"{ca}.in_proj_bias", 0, D, P[f"{sa}.in_proj_bias"])
    else:
        raise ValueError(kind)
    return P


def other_layer_gamma(P, prefix, norm, layer):
    """Copy of P whose `prefix`.`norm`.weight is layer `layer`'s."""
    P = dict(P)
    stack = prefix.rsplit(".", 1)[0]
    P[f"{prefix}.{norm}.weight"] = P[f"{stack}.{layer}.{norm}.weight"]
    return P


# decoder faults that move > 90 % of the teacher-forced rows past the bound (fault, layer)
DECODER_FAULTS = [(k, l) for l in (0, 3, 5) for k in ("n3_from_other", "n1_from_other", "swap_n2n3", "drop_n2_beta",
                                                      "drop_out_bias", "drop_ca_out_bias", "drop_v_bias", "drop_ca_v_bias")]
ENCODER_FAULTS = ("swap_n1n2", "drop_out_bias", "drop_n2_beta", "drop_v_bias")


def decoder_fault(P, kind, layer):
    prefix = f"decoder.layers.{layer}"
    if kind in ("n3_from_other", "n1_from_other"):
        return other_layer_gamma(P, prefix, "norm3" if kind == "n3_from_other" else "norm1", (layer + 1) % 6)
    return with_fault(P, prefix, kind)


# --------------------------------------------------------------------------------------------------------- (a) CPU
def _torch_layers(cls, layer_cls, P, stack, nhead, num_layers):
    layer = layer_cls(d_model=D, nhead=nhead, dim_feedforward=P[f"{stack}.layers.0.linear1.weight"].shape[0], dropout=0.0,
                      dtype=torch.float64)
    kw = dict(enable_nested_tensor=False) if cls is torch.nn.TransformerEncoder else {}
    mod = cls(layer, num_layers=num_layers, **kw).eval()
    mod.load_state_dict({k[len(stack) + 1:]: v for k, v in P.items() if k.startswith(stack + ".")})
    return mod


@pytest.mark.parametrize("fused", [True, False])
def test_oracle_stacks_equal_torch_modules_on_trained_weights(fused, monkeypatch):
    """O.encoder_stack (a modality stack, 16 heads; encoder_cross, 4 heads; bool and float key masks) and O.decoder_stack
    (causal mask, memory padding mask) against nn.TransformerEncoder / nn.TransformerDecoder in fp64, to 1e-12."""
    from oracle import mmt_oracle as O
    monkeypatch.setattr(O, "FUSED_SDPA", fused)
    P = trained_state_dict()
    g = torch.Generator().manual_seed(3)
    S, B = 37, 3
    x = torch.randn(S, B, D, generator=g, dtype=torch.float64)
    bool_mask = torch.rand(B, S, generator=g) < 0.3
    bool_mask[:, 0] = False
    float_mask = (torch.rand(B, S, generator=g) < 0.4).double()
    prev = torch.backends.mha.get_fastpath_enabled()
    torch.backends.mha.set_fastpath_enabled(False)
    try:
        with torch.no_grad():
            for stack, nhead in (("encoder_HSQC", 16), ("encoder_cross", 4)):
                mod = _torch_layers(torch.nn.TransformerEncoder, torch.nn.TransformerEncoderLayer, P, stack, nhead, 6)
                for mask in (bool_mask, float_mask):
                    want = mod(x, src_key_padding_mask=mask)
                    got = O.encoder_stack(P, stack, nhead, x, mask, 6)
                    torch.testing.assert_close(got, want, atol=1e-12, rtol=0, msg=f"{stack} {mask.dtype}")
            T = 21
            tgt = torch.randn(T, B, D, generator=g, dtype=torch.float64)
            mod = _torch_layers(torch.nn.TransformerDecoder, torch.nn.TransformerDecoderLayer, P, "decoder", 16, 6)
            causal = O.causal_bias(T, "cpu").double()
            want = mod(tgt, x, tgt_mask=causal, memory_key_padding_mask=bool_mask)
            got = O.decoder_stack(P, 16, tgt, x, causal, bool_mask, 6)
            torch.testing.assert_close(got, want, atol=1e-12, rtol=0)
    finally:
        torch.backends.mha.set_fastpath_enabled(prev)


# --------------------------------------------------------------------------------------------------------- (b) CPU
REL_TOL = 1e-2                 # the teacher-forced bound: |logit error| / max |logit| of the row
ENC_CONTRACT_REL = 3e-3        # the encoder bound against the fp64 bf16 contract: rms error / rms per spectrum


def _cpu_memory():
    if "mem" not in _W:
        from multimodalspectraltransformer_b200 import synthetic
        from oracle import mmt_oracle as O
        data = synthetic.make_spectra(4, seed=77)
        with torch.no_grad():
            mem, mask, _, _ = O.encode(trained_state_dict(), data, O.default_config())
        _W["mem"], _W["mask"], _W["data"] = mem, mask, data
    return _W["mem"], _W["mask"], _W["data"]


def _teacher_forced_cpu(P, T=48, K=4):
    from oracle import mmt_oracle as O
    mem, mask, _ = _cpu_memory()
    B = mem.shape[1]
    g = torch.Generator().manual_seed(5)
    trg = torch.randint(4, 43, (T, B * K), generator=g)
    trg[0] = 3
    with torch.no_grad():
        return O.teacher_forced_logits(P, mem.repeat_interleave(K, dim=1), mask.repeat_interleave(K, dim=0), trg, O.default_config())


@pytest.mark.parametrize("kind,layer", DECODER_FAULTS)
def test_decoder_faults_leave_the_teacher_forced_bound(kind, layer, monkeypatch):
    """4 spectra x 4 candidates x 48 positions of the fp64 oracle: each fault moves > 90 % of the rows past 1e-2 of the
    row scale -- the bound of the teacher-forced tests, which therefore fail on such a fault in the engine."""
    from oracle import mmt_oracle as O
    monkeypatch.setattr(O, "FUSED_SDPA", False)
    P = trained_state_dict()
    if "tf_ref" not in _W:
        _W["tf_ref"] = _teacher_forced_cpu(P)
    ref = _W["tf_ref"]
    wrong = _teacher_forced_cpu(decoder_fault(P, kind, layer))
    rel = (wrong - ref).abs().amax(-1) / ref.abs().amax(-1)
    frac = float((rel > REL_TOL).double().mean())
    assert frac > 0.9, (kind, layer, frac, float(rel.max()))


def _contract_encode(P):
    from oracle import mmt_oracle as O
    from test_gpu_encoder_fp64 import _contract_stack
    _, _, data = _cpu_memory()
    fused, stack = O.FUSED_SDPA, O.encoder_stack
    try:
        O.FUSED_SDPA, O.encoder_stack = False, _contract_stack
        with torch.no_grad():
            return O.encode(P, data, O.default_config())[0]
    finally:
        O.FUSED_SDPA, O.encoder_stack = fused, stack


@pytest.mark.parametrize("stack,layer", [("encoder_13C", 2), ("encoder_cross", 4)])
def test_encoder_faults_leave_the_contract_bound(stack, layer):
    """Each encoder fault, run through the fp64 bf16 contract of the whole encoder, moves every spectrum's memory past
    the 3e-3 (rms error / rms) bound the GPU encoder is held to against that contract."""
    P = trained_state_dict()
    if "enc_ref" not in _W:
        _W["enc_ref"] = _contract_encode(P)
    ref = _W["enc_ref"]
    for kind in ENCODER_FAULTS:
        wrong = _contract_encode(with_fault(P, f"{stack}.layers.{layer}", kind))
        err = (wrong - ref).pow(2).mean(dim=(0, 2)).sqrt() / ref.pow(2).mean(dim=(0, 2)).sqrt()
        assert bool((err > ENC_CONTRACT_REL).all()), (stack, layer, kind, err.tolist())


# --------------------------------------------------------------------------------------------------------- (c) GPU
SMALL_GEOMETRIES = {          # spectra, candidates, engine knobs, precisions: waves of the fused decode_attn path
    "fused_6x16": (6, 16, {}, ("bf16", "fp32")),
    "cluster_ffn_6x16": (6, 16, {"MMT_CLUSTER_FFN": "1"}, ("bf16",)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("weights", ["init", "trained"])
@pytest.mark.parametrize("geometry", list(SMALL_GEOMETRIES))
def test_fused_step_teacher_forced_logits_vs_fp64_oracle(geometry, weights, monkeypatch):
    """The small-wave step (decode_attn with the previous layer's FFN partials and norm3 folded into its prologue and the
    last layer's into the sampler; the cluster FFN applying norm3 itself), all 128 positions, against the fp64 oracle,
    with the bounds and fault guard of test_gpu_large_wave's teacher-forced test."""
    from test_gpu_large_wave import check_teacher_forced
    check_teacher_forced(*SMALL_GEOMETRIES[geometry], weights, geometry, monkeypatch)


# --------------------------------------------------------------------------------------------------------- (d) GPU
@pytest.mark.gpu
@pytest.mark.parametrize("unfused", [False, True])
def test_beam_search_fp32_vs_oracle_on_trained_weights(unfused):
    """3 items x 4 beams x 20 steps in the fp32 check mode against oracle.beam_search: identical sequences, scores to
    5e-4, probabilities to 5e-6.  unfused: the engine with MMT_FUSED_DECODE_ROWS=0 (the large-wave kernels)."""
    from test_gpu_beam import MODE, STOI, compare, run
    from oracle import mmt_oracle as O
    from multimodalspectraltransformer_b200 import synthetic
    from multimodalspectraltransformer_b200.generate import _mask_to_bias
    model = trained_model()
    data = synthetic.make_spectra(3, seed=21)
    got, memory, mask = run(model, data, 4, 20)
    if unfused:
        eng = engine_with("trained", MMT_FUSED_DECODE_ROWS="0")
        seq, ln, score, probs, _ = eng.beam_search(memory, _mask_to_bias(mask), beam_size=4, gen_len=20, eos=STOI["<EOS>"])
        got = [[(score[i, k].item(), seq[i, k, :ln[i, k]].tolist(), probs[i, k, :ln[i, k] - 1].tolist()) for k in range(4)]
               for i in range(3)]
    P = state_dict_for("trained", device="cpu")
    with torch.no_grad():
        want = O.beam_search(P, memory.cpu(), mask.cpu(), O.default_config(training_mode=MODE), 4, 20)
    compare(got, want)


# --------------------------------------------------------------------------------------------------------- (e) GPU
def layer_tail_ref(x, att_s, att_c, P, layer, mode, proj_terms=1, ffn_terms=1):
    """fp64 evaluation of the decode layer tail's contract on rows x / att_s / att_c (R,128): mode "bf16": the attention
    outputs and every GEMM operand rounded to bf16, times the hi weight terms (proj_terms / ffn_terms = 2: hi + lo), the
    FFN hidden activation rounded to bf16, residual and LayerNorm exact; "fp32": exact.  -> x1, qc, x2, out."""
    from test_gpu_encoder_fp64 import two_term
    from test_gpu_large_wave import bf16
    p = f"decoder.layers.{layer}."
    b = lambda n: P[p + n].double()
    if mode == "fp32":
        W = lambda n, t: P[p + n].double()
        rnd = lambda t: t.double()
    else:
        W = lambda n, t: two_term(P[p + n], t)
        rnd = bf16
    ln = lambda t, n: F.layer_norm(t, (D,), b(n + ".weight"), b(n + ".bias"), 1e-5)
    x = x.double()
    x1 = ln(x + F.linear(rnd(att_s), W("self_attn.out_proj.weight", proj_terms), b("self_attn.out_proj.bias")), "norm1")
    qc = F.linear(rnd(x1), W("multihead_attn.in_proj_weight", proj_terms)[:D], b("multihead_attn.in_proj_bias")[:D])
    x2 = ln(x1 + F.linear(rnd(att_c), W("multihead_attn.out_proj.weight", proj_terms), b("multihead_attn.out_proj.bias")), "norm2")
    h = rnd(torch.relu(F.linear(rnd(x2), W("linear1.weight", ffn_terms), b("linear1.bias"))))
    out = ln(x2 + F.linear(h, W("linear2.weight", ffn_terms), b("linear2.bias")), "norm3")
    return x1, qc, x2, out


TAIL_VARIANTS = {   # engine knobs, precision, weight terms of the projections / the FFN
    "default": ({}, "bf16", 1, 1),
    "no_chain": ({"MMT_NO_GEMM_CHAIN": "1"}, "bf16", 1, 1),
    "no_prologue": ({"MMT_NO_FFN_PROLOGUE": "1"}, "bf16", 1, 1),
    "proj_two_term": ({"MMT_DEC_PROJ_TWO_TERM": "1"}, "bf16", 2, 1),
    "ffn_two_term": ({"MMT_DEC_FFN_TWO_TERM": "1"}, "bf16", 1, 2),
    "fp32": ({}, "fp32", 1, 1),
}
# per element |err| <= atol + rtol |ref| and mean |err| <= mean, on every output of the tail.  Measured on an NVIDIA B200
# (1000 W power limit) over every case: bf16 max |err| 1.9e-3 (a bf16 operand rounded the other way where the fp32
# accumulator sits at a midpoint), mean 1.6e-5 (hi weight terms) / 2.4e-5 (two-term projections); fp32 max 2.2e-6, mean
# 1.4e-7.  bf16 keeps the fused-FFN test's per-element bound; the means and the fp32 bound keep 2.5x to 7x headroom.
TAIL_TOL = {"bf16": (3e-3, 1e-3, 6e-5), "fp32": (1e-5, 0.0, 1e-6)}
TAIL_ROWS = (1, 5, 129, 2047, 2048, 4099, 24576, 24577, 131072)


def _tail_violation(got, ref, tol):
    """(fraction of rows with an element outside the bound, mean |err|)."""
    atol, rtol, _ = tol
    err = (got.double() - ref).abs()
    return float((err > atol + rtol * ref.abs()).any(-1).double().mean()), float(err.mean())


@pytest.mark.gpu
@pytest.mark.parametrize("weights", ["init", "trained"])
@pytest.mark.parametrize("R", TAIL_ROWS)
@pytest.mark.parametrize("variant", list(TAIL_VARIANTS))
def test_decode_layer_tail_vs_fp64_contract(variant, R, weights):
    """x1, qc, x2 (where stored) and the layer output of layers 0 and 5, element by element against `layer_tail_ref`:
    the chained out-proj + norm1 + query projection (R <= 24,576), the separate launches above it or with
    MMT_NO_GEMM_CHAIN, the FFN prologue (cross out-proj + norm2 inside the FFN kernel, R >= 2048), the LN-epilogue GEMM
    with the split-F FFN below 2048 rows or with MMT_NO_FFN_PROLOGUE, two-term weights, and the fp32 mode.  Rows checked:
    all up to 4,099, else both edges of every 128-row tile and 256 random rows.  Sharpness guard (trained weights):
    references with another layer's norm3, norm2 and norm3 exchanged, or the cross query bias taken from the self
    attention's leave the bound on > 90 % of the rows."""
    from test_gpu_large_wave import _check_rows
    env, prec, pt, ft = TAIL_VARIANTS[variant]
    tol = TAIL_TOL[prec]
    eng = engine_with(weights, **env)
    P = state_dict_for(weights, torch.float64)
    g = torch.Generator(device="cuda").manual_seed(R + 7)
    x = torch.randn(R, D, device="cuda", generator=g)
    att_s = 0.5 * torch.randn(R, D, device="cuda", generator=g)
    att_c = 0.5 * torch.randn(R, D, device="cuda", generator=g)
    rows = _check_rows(R, R)
    stored_x2 = prec == "fp32" or R < 2048 or variant == "no_prologue"
    for layer in (0, 5):
        outs = eng.decode_layer_tail(layer, x, att_s, att_c, precision=prec)
        assert (outs[2] is not None) == stored_x2, (variant, R)
        refs = layer_tail_ref(x[rows], att_s[rows], att_c[rows], P, layer, prec, pt, ft)
        stats = []
        for name, got, ref in zip(("x1", "qc", "x2", "out"), outs, refs):
            if got is None:
                continue
            frac, mean = _tail_violation(got[rows], ref, tol)
            stats.append(f"{name} max {float((got[rows].double() - ref).abs().max()):.2e} mean {mean:.2e}")
            assert frac == 0 and mean <= tol[2], (variant, R, weights, layer, name, frac, mean)
        print(f"layer tail {variant} R={R} {weights} layer {layer}: " + ", ".join(stats))
        if weights != "trained":
            continue
        got_out, got_qc = outs[3][rows], outs[1][rows]
        for kind, which, Pw in (("norm3 of another layer", 3, other_layer_gamma(P, f"decoder.layers.{layer}", "norm3", (layer + 1) % 6)),
                                ("norm2 <-> norm3", 3, with_fault(P, f"decoder.layers.{layer}", "swap_n2n3")),
                                ("cross q bias from self attention", 1, with_fault(P, f"decoder.layers.{layer}", "ca_q_from_self"))):
            wrong = layer_tail_ref(x[rows], att_s[rows], att_c[rows], Pw, layer, prec, pt, ft)[which]
            frac, _ = _tail_violation(got_out if which == 3 else got_qc, wrong, tol)
            assert frac > 0.9, (kind, variant, R, layer, frac)
