"""The encoder against fp64 references, kernel by kernel and for every spectrum of the bench batch.

(a) the encoder attention kernels (attn_encoder_tc8 for the 8-wide heads of the five modality stacks, attn_encoder_tc and
    the opt-in attn_encoder_tc5 for the 32-wide heads of encoder_cross, attn_encoder_f32 in both widths), driven through
    `mmt_encoder_layer` (the encoder's own layer code), element by element against softmax(q k^T / sqrt(dh) + bias) v in
    fp64 on the QKV projection the kernel read: key counts at the 16-key block and 16-row tile edges, more than 768 keys
    (the 32-wide kernels walk them in chunks), dense and ragged layouts, bool and float (+1.0) key masks;
(b) one encoder layer, row by row, against an fp64 evaluation of the bf16 mode's contract (bf16(x) times the two-term
    weights, attention output and FFN hidden activation rounded to bf16, residual and LayerNorm exact) and of the fp32 mode;
(c) the whole encoder at the bench batch (1024 spectra: four chunks of 256) and at 257 / 600 spectra, a float-mask mode
    and an MS mode (902 memory rows), every spectrum against oracle.encode in fp64 on the device, and in the bf16 mode
    against the contract of (b) run through all 12 layers;
(d) CPU: the fp64 oracle encoder is the same function with torch's fused SDPA and with the spelled-out softmax.

Every bound carries a sharpness guard: references with one deliberate fault (a key dropped, a key read from the
neighbouring row, the +1.0 float-mask bias ignored, the lo weight term dropped, the neighbouring spectrum, a chunk shifted
by one spectrum) must fall outside it."""
import math

import pytest
import torch
import torch.nn.functional as F

from test_gpu_large_wave import SCALE as SCALE8, U16, _tolerance, bf16, outside
from test_gpu_trained_weights import with_weights

D = 128
LAYER = {0: 1, 1: 4, 2: 2, 3: 5, 4: 3, 5: 3}      # which layer of each stack the kernel tests use
STACKS = ("encoder_1H", "encoder_13C", "encoder_HSQC", "encoder_COSY", "encoder_IR", "encoder_cross")


def _heads(stack):
    return 4 if stack == 5 else 16


def _engine(weights, **env):
    from test_gpu_trained_weights import engine_with
    return engine_with(weights, **env)


def _layer_params(stack, layer, weights):
    from test_gpu_trained_weights import state_dict_for
    sd = state_dict_for(weights)
    p = f"{STACKS[stack]}.layers.{layer}."
    names = ("self_attn.in_proj_weight", "self_attn.in_proj_bias", "self_attn.out_proj.weight", "self_attn.out_proj.bias",
             "linear1.weight", "linear1.bias", "linear2.weight", "linear2.bias", "norm1.weight", "norm1.bias",
             "norm2.weight", "norm2.bias")
    return {n: sd[p + n] for n in names}


# --------------------------------------------------------------------------------------------------------- references
def attend(qkv, qrows, krows, kbias, nh, scale):
    """fp64 attention of B sequences: qkv (R,384) rows; qrows (B,Tq) / krows (B,Tk) row numbers (padding: any valid row);
    kbias (B,Tk) additive (-inf: key padding).  -> o (B,H,Tq,dh), p (B,H,Tq,Tk), q, k, v."""
    dh = D // nh
    t = qkv.double()
    B, Tq = qrows.shape
    Tk = krows.shape[1]
    q = t[qrows][..., :D].reshape(B, Tq, nh, dh).transpose(1, 2)
    k = t[krows][..., D:2 * D].reshape(B, Tk, nh, dh).transpose(1, 2)
    v = t[krows][..., 2 * D:].reshape(B, Tk, nh, dh).transpose(1, 2)
    s = q @ k.transpose(-1, -2) * scale + kbias.double()[:, None, None, :]
    p = torch.softmax(s, dim=-1)
    return p @ v, p, q, k, v


def attention_bound(o, p, q, k, v, scale, split, rounded):
    """Per-element bound of |kernel - fp64| (`_tolerance` of the decode tests; q rescaled because it applies 1/sqrt(8)).
    split: the tensor-core kernels' two-term bf16 operands (the dropped lo.lo products and the residuals' own rounding:
    ~3 * 2^-18 of |q||k| and of p|v|, inside its 2^-16 terms) with ex2.approx; else the fp32 SIMT kernel.  rounded: the
    output is stored as bf16 (2^-8 |o|)."""
    qs = q * (scale / SCALE8)
    if split:
        z = torch.zeros_like(k)
        t = _tolerance(o, p, qs, k, v, True, z, z)
        return t if rounded else t - (U16 - 2.0 ** -20) * o.abs()
    t = _tolerance(o, p, qs, k, v, False)
    return t + U16 * o.abs() if rounded else t


def two_term(w, terms=2):
    hi = w.float().bfloat16()
    return hi.double() + ((w.float() - hi.float()).bfloat16().double() if terms == 2 else 0.0)


def layer_ref(x, qrows, krows, kbias, prm, nh, mode):
    """One post-norm encoder layer in fp64 on the rows x (R,128) (sequences as in `attend`; only the query rows of the
    result are meaningful).  mode "fp32": exact arithmetic; "bf16": the tensor-core contract -- bf16(x) times W_hi + W_lo
    (QKV, out_proj, linear1, linear2), attention output and FFN hidden activation rounded to bf16, residual and LayerNorm
    exact; "bf16_hi": the same with the hi weight terms alone (a fault the bounds must see)."""
    x = x.double()
    if mode == "fp32":
        W, xin, rnd = (lambda n: prm[n].double()), x, (lambda t: t)
    else:
        terms = 1 if mode == "bf16_hi" else 2
        W, xin, rnd = (lambda n: two_term(prm[n], terms)), bf16(x), bf16
    b = lambda n: prm[n].double()
    qkv = F.linear(xin, W("self_attn.in_proj_weight"), b("self_attn.in_proj_bias"))
    o = attend(qkv, qrows, krows, kbias, nh, 1.0 / math.sqrt(D // nh))[0]
    att = torch.zeros_like(x)
    B, Tq = qrows.shape
    att[qrows.reshape(-1)] = o.transpose(1, 2).reshape(B * Tq, D)            # padding query rows repeat a real row
    att = rnd(att)
    x1 = F.layer_norm(x + F.linear(att, W("self_attn.out_proj.weight"), b("self_attn.out_proj.bias")), (D,),
                      b("norm1.weight"), b("norm1.bias"), 1e-5)
    h = rnd(torch.relu(F.linear(rnd(x1), W("linear1.weight"), b("linear1.bias"))))
    return F.layer_norm(x1 + F.linear(h, W("linear2.weight"), b("linear2.bias")), (D,), b("norm2.weight"), b("norm2.bias"), 1e-5)


# --------------------------------------------------------------------------------------------------------- cases
NK8 = (1, 15, 16, 17, 31, 32, 33, 63, 64, 65, 128, 129, 193)
NK32 = (1, 15, 16, 17, 31, 32, 33, 63, 64, 65, 128, 129, 582, 767, 768, 769, 902)
DOM = (None, 0, "last", 15, 16, 31, 32, 767, 768)        # the key a sequence's aimed queries score highest
CASES = {   # stack, S, spectra, layout, key counts
    "dh8_S66_bool_B256": (0, 66, 256, "bool", NK8),
    "dh8_S129_bool": (2, 129, 64, "bool", NK8),
    "dh8_S193_float": (1, 193, 24, "float", None),
    "dh8_S193_ragged": (4, 193, 96, "ragged", NK8),
    "dh32_S582_bool": (5, 582, 24, "bool", NK32),
    "dh32_S902_float": (5, 902, 6, "float", None),
    "dh32_S902_bool": (5, 902, 17, "bool", NK32),
    "dh32_S902_ragged": (5, 902, 17, "ragged", NK32),
}


def make_case(name, prm):
    """Rows x, the layout arguments of `Engine.encoder_layer` and the fp64 view of the sequences (qrows, krows, kbias).
    Sequence b has nk = NK[b % len] keys (at random positions; ragged: cnt >= nk rows, kidx a random subset, three unused
    rows between sequences, kstride = S + 5 with the unused kidx slots pointing at row 0); float masks attend every row, +1.0 on a
    block of a third of them.  Every third query row of a sequence is aimed at its dominant key DOM[b % len] (scaled score
    ~ +10 in every head), so the running maximum moves when that key's block is reached."""
    stack, S, B, layout, nks = CASES[name]
    nh = _heads(stack)
    dh = D // nh
    g = torch.Generator().manual_seed(sum(name.encode()) * 7 + S)
    qrows, keys, biases, cnts, starts, kidx = [], [], [], [], [], []
    row = 0
    for bb in range(B):
        nk = S if nks is None else min(nks[bb % len(nks)], S)
        cnt = S if layout != "ragged" else int(torch.randint(nk, S + 1, (1,), generator=g))
        kk = torch.sort(torch.randperm(cnt, generator=g)[:nk]).values
        bias = torch.zeros(nk, dtype=torch.float64)
        if layout == "float":
            lo = int(torch.randint(0, S - S // 3, (1,), generator=g))
            bias[lo:lo + S // 3] = 1.0
        starts.append(row); cnts.append(cnt)
        qrows.append(row + torch.arange(cnt)); keys.append(row + kk); biases.append(bias)
        kidx.append(torch.cat([kk, torch.zeros(S + 5 - nk, dtype=torch.long)]))
        row += cnt + (3 if layout == "ragged" else 0)
    R = row
    x = torch.randn(R, D, generator=g, dtype=torch.float64)
    # aim: x_i = alpha * sum_h Wq_h^T k_h / |k_h| for the dominant key's k (the per-head directions are nearly orthogonal)
    Wq, Wk = prm["self_attn.in_proj_weight"][:D].double().cpu(), prm["self_attn.in_proj_weight"][D:2 * D].double().cpu()
    bq, bk = prm["self_attn.in_proj_bias"][:D].double().cpu(), prm["self_attn.in_proj_bias"][D:2 * D].double().cpu()
    dom = []
    for bb in range(B):
        sel = DOM[bb % len(DOM)]
        nk = len(keys[bb])
        j = None if sel is None else (nk - 1 if sel == "last" else sel)
        if j is not None and j >= nk:
            j = None
        dom.append(j)
        if j is None:
            continue
        kj = (F.linear(x[keys[bb][j]], Wk, bk)).reshape(nh, dh)
        kh = kj / kj.norm(dim=-1, keepdim=True)
        u = torch.einsum("hdc,hd->c", Wq.reshape(nh, dh, D), kh)
        a = (F.linear(u, Wq).reshape(nh, dh) * kj).sum(-1).mean() / math.sqrt(dh)
        c = (bq.reshape(nh, dh) * kj).sum(-1).mean() / math.sqrt(dh)
        aimed = qrows[bb][::3]
        aimed = aimed[aimed != keys[bb][j]]
        x[aimed] = ((10 - c) / a) * u
    Tq, Tk = max(cnts), max(len(k) for k in keys)
    pad_to = lambda t, n: torch.cat([t, t[:1].expand(n - len(t))])
    view = dict(qrows=torch.stack([pad_to(q, Tq) for q in qrows]).cuda(),
                krows=torch.stack([pad_to(k, Tk) for k in keys]).cuda(),
                kbias=torch.stack([torch.cat([b, torch.full((Tk - len(b),), float("-inf"), dtype=torch.float64)]) for b in biases]).cuda(),
                qmask=torch.stack([torch.arange(Tq) < c for c in cnts]).cuda(), dom=dom, keys=keys, nh=nh, S=S)
    if layout == "ragged":
        args = dict(row_start=torch.tensor(starts), cnt=torch.tensor(cnts), nk=torch.tensor([len(k) for k in keys]),
                    kidx=torch.stack(kidx), S=S)
    else:
        kb = torch.full((B, S), float("-inf"))
        for bb in range(B):
            kb[bb, keys[bb] - starts[bb]] = biases[bb].float()
        args = dict(key_bias=kb)
    return x.float().cuda(), args, view


def _faulty(view, kind):
    """krows / kbias of a reference with one fault in every sequence: "drop" (the dominant key, else the last one, left
    out), "neighbour" (that key read from the next row: the previous one for the last row), "bias" (+1.0 read as 0)."""
    krows, kbias = view["krows"].clone(), view["kbias"].clone()
    for bb, keys in enumerate(view["keys"]):
        j = view["dom"][bb] if view["dom"][bb] is not None else len(keys) - 1
        if kind == "drop":
            kbias[bb, j] = float("-inf")
        elif kind == "neighbour":
            r = int(keys[j])
            last = int(view["qrows"][bb][view["qmask"][bb]].max())
            krows[bb, j] = r + 1 if r < last else r - 1
    if kind == "bias":
        kbias = torch.where(kbias == 1.0, torch.zeros_like(kbias), kbias)
    return krows, kbias


# --------------------------------------------------------------------------------------------------------- (a)
VARIANTS = {   # engine knobs (read at creation), precision, two-term tensor-core numerics, output stored as bf16
    "tc_bf16": ({}, "bf16", True, True),                                          # attn_encoder_tc8 / attn_encoder_tc
    "tc_fp32": ({"MMT_TC_ATTENTION_FP32": "1"}, "fp32", True, False),
    "tc5_bf16": ({"MMT_TC5_ATTENTION": "1"}, "bf16", True, True),                 # attn_encoder_tc5 (32-wide heads)
    "tc5_fp32": ({"MMT_TC5_ATTENTION": "1", "MMT_TC_ATTENTION_FP32": "1"}, "fp32", True, False),
    "simt_bf16": ({"MMT_NO_TC_ATTENTION": "1"}, "bf16", False, True),             # attn_encoder_f32<8 / 32>
    "simt_fp32": ({}, "fp32", False, False),
}


def _seq_rows(view, t):
    """(B,Tq,...) per-query view of the rows t (R,...)."""
    return t[view["qrows"]]


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("variant,weights", with_weights(list(VARIANTS)))
def test_encoder_attention_vs_fp64(variant, case, weights):
    """Every query row of every sequence, element by element: |kernel - fp64| within `attention_bound`.  Sharpness
    guard: the references with the dominant (else last) key dropped or read from the neighbouring row leave the bound on
    > 90 % of the aimed rows, the one with the +1.0 biases ignored on > 75 % of the rows of the float-mask cases.
    weights: the init or the trained-like weights (non-zero Q / K / V biases)."""
    env, prec, split, rounded = VARIANTS[variant]
    stack = CASES[case][0]
    if variant.startswith("tc5") and stack != 5:
        pytest.skip("attn_encoder_tc5 serves the 32-wide heads only")
    layer = LAYER[stack]
    prm = _layer_params(stack, layer, weights)
    x, args, view = make_case(case, prm)
    qkv, att, _ = _engine(weights, **env).encoder_layer(stack, layer, x, precision=prec, **args)
    nh = view["nh"]
    scale = 1.0 / math.sqrt(D // nh)
    qm = view["qmask"]
    got = _seq_rows(view, att).double()                                      # (B,Tq,128)
    back = lambda z: z.transpose(1, 2).reshape(z.shape[0], z.shape[2], D)
    worst, B = 0.0, got.shape[0]
    refs, tols = [], []
    for b0 in range(0, B, 32):
        sl = slice(b0, b0 + 32)
        o, p, q, k, v = attend(qkv, view["qrows"][sl], view["krows"][sl], view["kbias"][sl], nh, scale)
        tol = attention_bound(o, p, q, k, v, scale, split, rounded)
        o, tol = back(o), back(tol)
        bad = outside(got[sl], o, tol) & qm[sl]
        worst = max(worst, float((((got[sl] - o).abs() / tol).amax(-1))[qm[sl]].max()))
        assert not bool(bad.any()), (variant, case, torch.nonzero(bad)[:5].tolist(), worst)
        refs.append(o); tols.append(tol)
    ref, tol = torch.cat(refs), torch.cat(tols)
    print(f"encoder attention {variant} {case} {weights}: max |err| / bound = {worst:.3f}")
    # sharpness guards
    aimed = torch.zeros_like(qm)
    for bb in range(B):
        if view["dom"][bb] is not None:
            aimed[bb, ::3] = True
    aimed &= qm
    for kind in ("drop", "neighbour") + (("bias",) if CASES[case][3] == "float" else ()):
        krows, kbias = _faulty(view, kind)
        wrong = torch.cat([back(attend(qkv, view["qrows"][b0:b0 + 32], krows[b0:b0 + 32], kbias[b0:b0 + 32], nh, scale)[0])
                           for b0 in range(0, B, 32)])
        sel = aimed if kind != "bias" else qm
        if not bool(sel.any()):
            continue
        frac = float(outside(wrong, ref, tol)[sel].double().mean())
        assert frac > (0.9 if kind != "bias" else 0.75), (kind, variant, case, frac)


# --------------------------------------------------------------------------------------------------------- (b)
LAYER_CASES = ("dh8_S66_bool_B256", "dh8_S193_ragged", "dh32_S582_bool", "dh32_S902_float", "dh32_S902_ragged")
# |err| of the layer output (unit-scale LayerNorm rows), max and mean over the checked rows.  Measured on an NVIDIA B200
# (1000 W power limit): bf16 max 3.1e-3 .. 5.3e-3, mean 2.1e-5 .. 3.1e-5; fp32 max 2.5e-6 .. 1.3e-5, mean 1.9e-7 .. 9.8e-7.
LAYER_TOL = {"bf16": (1e-2, 8e-5), "fp32": (5e-5, 5e-6)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", LAYER_CASES)
@pytest.mark.parametrize("prec,weights", with_weights(["bf16", "fp32"]))
def test_encoder_layer_vs_fp64_contract(prec, case, weights):
    """The whole layer (QKV projection, attention, out_proj + LN1, fused FFN + LN2), every query row, against
    `layer_ref` in fp64: max |err| and mean |err| bounds (LAYER_TOL, like the fused-FFN test: a handful of bf16 values
    round the other way where the fp32 accumulator sits at a midpoint).  Sharpness guard (bf16): the contract with the hi
    weight terms alone exceeds the mean bound.  weights: the init or the trained-like weights; with the trained ones,
    references with norm1 and norm2 exchanged, the out_proj bias, the V bias or the Q bias dropped each leave the max or
    the mean bound."""
    from test_gpu_trained_weights import with_fault
    stack = CASES[case][0]
    layer = LAYER[stack]
    prm = _layer_params(stack, layer, weights)
    x, args, view = make_case(case, prm)
    _, _, out = _engine(weights).encoder_layer(stack, layer, x, precision=prec, **args)
    qm = view["qmask"]
    ref = layer_ref(x, view["qrows"], view["krows"], view["kbias"], prm, view["nh"], prec)
    err = (_seq_rows(view, out).double() - _seq_rows(view, ref))[qm].abs()
    mx, mean = float(err.max()), float(err.mean())
    mean_hi = None
    if prec == "bf16":
        hi = layer_ref(x, view["qrows"], view["krows"], view["kbias"], prm, view["nh"], "bf16_hi")
        mean_hi = float((_seq_rows(view, hi) - _seq_rows(view, ref))[qm].abs().mean())
    print(f"encoder layer {prec} {case} {weights}: max |err| {mx:.3e} mean {mean:.3e} (bounds {LAYER_TOL[prec]}; hi terms "
          f"only: mean {mean_hi})")
    assert mx < LAYER_TOL[prec][0] and mean < LAYER_TOL[prec][1], (prec, case, mx, mean)
    if prec == "bf16":
        assert mean_hi > 2 * LAYER_TOL[prec][1], (case, mean_hi)
    if weights == "trained":
        got = _seq_rows(view, out).double()[qm]
        for kind in ("swap_n1n2", "drop_out_bias", "drop_v_bias", "drop_q_bias"):
            faulty = {k[2:]: v for k, v in with_fault({"x." + k: v for k, v in prm.items()}, "x", kind).items()}
            wrong = layer_ref(x, view["qrows"], view["krows"], view["kbias"], faulty, view["nh"], prec)
            e = (got - _seq_rows(view, wrong)[qm]).abs()
            assert float(e.max()) >= LAYER_TOL[prec][0] or float(e.mean()) >= LAYER_TOL[prec][1], (kind, prec, case, float(e.max()), float(e.mean()))


# --------------------------------------------------------------------------------------------------------- (c)
FULL = "1H_13C_HSQC_COSY_IR_MF_MW"
ENCODES = {   # spectra, seed, peaks, training_mode
    "bench_1024": (1024, 1000, "realistic", FULL),
    "max_257": (257, 257, "max", FULL),
    "realistic_600": (600, 600, "realistic", FULL),
    "float_mask_300": (300, 300, "realistic", "1H_13C_HSQC_IR_MF_MW"),     # COSY blank: +1.0 biases
    "ms_max_260": (260, 260, "max", "1H_13C_HSQC_COSY_IR_MF_MS_MW"),        # 902 memory rows
}
# Per spectrum, measured on an NVIDIA B200 (1000 W power limit) over the 2,441 spectra of ENCODES: fp32 max |memory - fp64|
# 1.1e-5 .. 3.3e-5 (the fp32 oracle is 1.35e-5 from fp64 on the CPU), mean / fingerprint <= 1.8e-5; bf16 rms error / rms
# 5.1e-3 .. 7.5e-3 against fp64 (the contract itself is ~5e-3 from fp64), 1.5e-3 .. 2.2e-3 (mean 1.26e-3 .. 1.82e-3) against
# the fp64 contract -- a tenth of the 1.5e-2 the golden tests allow.
FP32_ABS = 5e-5          # fp32 mode: max |memory - fp64|
BF16_REL = 1e-2          # bf16 mode: rms(memory - fp64) / rms(fp64)
BF16_CONTRACT_REL = 3e-3  # bf16 mode: rms(memory - fp64 contract) / rms
_REFS = {}


def _contract_stack(P, name, nhead, x, mask, num_layers):
    """oracle.encoder_stack with `layer_ref`'s bf16 rounding points (x (S,B,128) fp64, mask (B,S))."""
    S, B, _ = x.shape
    bias = mask.double().masked_fill(mask.bool(), float("-inf")) if mask.dtype == torch.bool else mask.double()
    rows = torch.arange(S * B, device=x.device).reshape(B, S)                # row b*S + s of x.transpose(0, 1)
    xr = x.transpose(0, 1).reshape(B * S, D)
    for l in range(num_layers):
        prm = {n[len(f"{name}.layers.{l}."):]: v for n, v in P.items() if n.startswith(f"{name}.layers.{l}.")}
        xr = layer_ref(xr, rows, rows, bias, prm, nhead, "bf16")
    return xr.reshape(B, S, D).transpose(0, 1)


def _references(name, weights):
    """fp64 oracle (and bf16 contract) outputs of case `name`, in blocks of 128 spectra, kept for the precisions."""
    if (name, weights) in _REFS:
        return _REFS[name, weights]
    from multimodalspectraltransformer_b200 import synthetic
    from oracle import mmt_oracle as O
    from test_gpu_trained_weights import state_dict_for
    B, seed, peaks, mode = ENCODES[name]
    data = {k: v.cuda() for k, v in synthetic.make_spectra(B, seed=seed, peaks=peaks).items()}
    P64 = state_dict_for(weights, torch.float64)
    cfg = O.default_config(training_mode=mode)
    out = {"data": data, "mem": [], "mask": [], "fp": [], "emb": [], "contract": []}
    fused, stack = O.FUSED_SDPA, O.encoder_stack
    try:
        O.FUSED_SDPA = False
        with torch.no_grad():
            for b0 in range(0, B, 128):
                blk = {k: v[b0:b0 + 128] for k, v in data.items()}
                mem, mask, fp, emb = O.encode(P64, blk, cfg)
                out["mem"].append(mem); out["mask"].append(mask); out["fp"].append(fp); out["emb"].append(emb)
                O.encoder_stack = _contract_stack
                out["contract"].append(O.encode(P64, blk, cfg)[0])
                O.encoder_stack = stack
    finally:
        O.FUSED_SDPA, O.encoder_stack = fused, stack
    for k in ("mem", "emb", "contract"):
        out[k] = torch.cat(out[k], dim=1)
    out["mask"], out["fp"] = torch.cat(out["mask"]), torch.cat(out["fp"])
    out["avg"] = out["mem"].mean(dim=0)
    _REFS.clear()              # one case at a time: the references of 1024 spectra are large
    _REFS[name, weights] = out
    return out


def _per_spectrum(got, ref, rel):
    """(S,B,D) -> (B,): max |err| (rel False) or rms(err) / rms(ref) (rel True) of each spectrum."""
    e = got.double() - ref
    if not rel:
        return e.abs().amax(dim=(0, 2))
    return e.pow(2).mean(dim=(0, 2)).sqrt() / ref.pow(2).mean(dim=(0, 2)).sqrt()


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("name,weights", with_weights(list(ENCODES)))
def test_encoder_every_spectrum_vs_fp64(weights, name, prec):
    """Memory, avg_memory and fingerprint of every spectrum against oracle.encode in fp64 (fp32 mode: max |err| <
    FP32_ABS; bf16: rms error / rms < BF16_REL, and < BF16_CONTRACT_REL against the fp64 contract run through all 12
    layers); key_bias and pad_mask bit for bit from the oracle's mask; embedding_src against fp64 and bit for bit
    against an encode of the same spectra one batch position further on.  Sharpness guards: every spectrum fails against
    the neighbouring spectrum's reference, and the spectra of a chunk shifted by one fail.  weights: the init or the
    trained-like weights (the bias and LayerNorm faults this bound sees on the latter: test_gpu_trained_weights)."""
    eng = _engine(weights)
    r = _references(name, weights)
    data = r["data"]
    B, _, _, mode = ENCODES[name]
    memory, pad, kb, fp, avg, emb = eng.encode(data, mode, prec, want_embedding_src=True)
    # masks and embeddings: exact
    omask = r["mask"]
    opad = omask if omask.dtype == torch.bool else omask != 0
    assert torch.equal(pad, opad.to(torch.uint8))
    okb = omask.float() if omask.dtype != torch.bool else torch.zeros_like(kb).masked_fill(omask, float("-inf"))
    assert torch.equal(kb, okb)
    e_emb = (emb.double() - r["emb"]).abs() / (1 + r["emb"].abs())
    assert float(e_emb.max()) < 1e-5, float(e_emb.max())
    rolled = {k: torch.roll(v, 1, dims=0) for k, v in data.items()}
    _, pad2, kb2, _, _, emb2 = eng.encode(rolled, mode, prec, want_embedding_src=True)
    assert torch.equal(torch.roll(pad2, -1, 0), pad) and torch.equal(torch.roll(kb2, -1, 0), kb)
    assert torch.equal(torch.roll(emb2, -1, 1), emb)
    # memory, mean and fingerprint of every spectrum
    rel = prec == "bf16"
    bound = BF16_REL if rel else FP32_ABS
    err = _per_spectrum(memory, r["mem"], rel)
    err_avg = _per_spectrum(avg[None], r["avg"][None], rel)
    err_fp = _per_spectrum(fp[None], r["fp"][None], rel)
    worst = {"memory": float(err.max()), "avg": float(err_avg.max()), "fingerprint": float(err_fp.max())}
    if rel:
        err_c = _per_spectrum(memory, r["contract"], True)
        worst["contract"] = float(err_c.max())
        print(f"encoder {name} {weights} bf16 on {torch.cuda.get_device_name()}: rms err / rms vs fp64 contract max "
              f"{worst['contract']:.3e} mean {float(err_c.mean()):.3e}")
        assert bool((err_c < BF16_CONTRACT_REL).all()), (name, torch.nonzero(err_c >= BF16_CONTRACT_REL)[:8].flatten().tolist(), worst)
    print(f"encoder {name} {weights} {prec}: worst spectrum {worst} (bound {bound})")
    assert bool((err < bound).all()), (name, prec, torch.nonzero(err >= bound)[:8].flatten().tolist(), worst)
    assert bool((err_avg < bound).all()) and bool((err_fp < bound).all()), (name, prec, worst)
    # sharpness: the neighbouring spectrum's reference fails for every spectrum; so does a chunk shifted by one
    assert bool((_per_spectrum(memory, torch.roll(r["mem"], 1, dims=1), rel) >= bound).all())
    c0 = 256 * (min(B, 1024) // 256 - 1) if B > 256 else 0
    shifted = r["mem"].clone()
    shifted[:, c0:c0 + 256] = torch.roll(r["mem"][:, c0:c0 + 256], 1, dims=1)
    e_shift = _per_spectrum(memory[:, c0:c0 + 256], shifted[:, c0:c0 + 256], rel)
    assert bool((e_shift >= bound).all()), (name, prec, float(e_shift.min()))


# --------------------------------------------------------------------------------------------------------- (d) CPU
@pytest.mark.parametrize("case", ["full_b2", "mode_hsqc_b2", "mode_ms_b2", "blank_1h13c_b2"])
def test_oracle_fp64_encode_fused_equals_spelled_out(case, monkeypatch):
    """oracle.encode with float64 weights computes in fp64 throughout (inputs, blank-modality zeros, key biases: torch's
    CPU SDPA gives wrong values without an error for float64 q/k/v and a float32 mask), and is the same function through
    the fused SDPA and the spelled-out softmax, to 1e-12: bool masks, float-mask modes, an MS mode."""
    from golden_util import load_case
    from oracle import mmt_oracle as O
    c, data, _ = load_case(case)
    cfg = O.default_config(training_mode=c["mode"])
    P = {k: v.double() for k, v in O.random_init_state_dict(O.default_config(), seed=0).items()}
    outs = []
    for fused in (True, False):
        monkeypatch.setattr(O, "FUSED_SDPA", fused)
        with torch.no_grad():
            outs.append(O.encode(P, data, cfg))
    (m1, k1, f1, e1), (m2, k2, f2, e2) = outs
    assert m1.dtype == torch.float64 and f1.dtype == torch.float64 and e1.dtype == torch.float64
    assert torch.equal(k1, k2) and torch.equal(e1, e2)
    torch.testing.assert_close(m1, m2, atol=1e-12, rtol=0)
    torch.testing.assert_close(f1, f2, atol=1e-12, rtol=0)
    # and it is the fp32 oracle's function: within fp32 round-off of it
    P32 = O.random_init_state_dict(O.default_config(), seed=0)
    with torch.no_grad():
        m32 = O.encode(P32, data, cfg)[0]
    assert float((m32.double() - m1).abs().max()) < 5e-5
