"""Python handle on one libmmt_b200 engine (weights resident on one B200).

PyTorch is plumbing here: it owns the input/output tensors and the CUDA stream;
all arithmetic of the path runs in the hand-written kernels behind the C ABI.
"""
from __future__ import annotations

import ctypes as C
import weakref

import numpy as np
import torch

from . import _lib
from ._lib import DecodeArgs, ModelDesc, Spectra

_PREC = {"fp32": _lib.PREC_FP32, "bf16": _lib.PREC_BF16}


def _desc_from(config, state_dict=None) -> ModelDesc:
    """Hyper-parameters of the model.  Every size a weight shape determines is read from the state_dict, not from
    ``config``: callers mutate ``config`` (e.g. ``max_len``) long after the model was built from it
    (mmt_result_test_functions_15_4.py:547), and the model -- not the namespace -- is what the engine must match."""
    g = lambda k, dflt: int(getattr(config, k, dflt))
    sd = state_dict or {}

    def rows(key, dflt, axis=0):
        return int(sd[key].shape[axis]) if key in sd else dflt

    def layers(prefix, dflt):
        idx = [int(k[len(prefix):].split(".")[0]) for k in sd if k.startswith(prefix)]
        return max(idx) + 1 if idx else dflt

    return ModelDesc(
        d_model=rows("embed_trg.weight", g("hidden_size", 128), 1), n_heads=g("num_heads", 16), n_heads_cross=int(g("num_heads", 16) / 4),
        d_ff=rows("decoder.layers.0.linear1.weight", 2048),      # torch default dim_feedforward; the reference never overrides it
        n_enc_layers=layers("encoder_cross.layers.", g("num_encoder_layers", 6)),
        n_dec_layers=layers("decoder.layers.", g("num_decoder_layers", 6)),
        vocab=rows("fc_out.weight", g("out_size", 43)), max_len=rows("pe_trg.weight", g("max_len", 128)),
        mf_vocab=rows("linear_embedding_MF.embedding.weight", g("MF_vocab_size", 212)),
        ms_vocab=rows("linear_embedding_MS.embedding.weight", g("MS_vocab_size", 43)),
        ir_bins=rows("linear_spec_embedding_IR.linear_spec_embedding_IR.weight", g("input_dim_IR", 1000), 1),
        fp_size=rows("fp1.weight", g("fingerprint_size", 512)),
        pad_points=g("padding_points_number", 64))


def _normalize_state_dict(state_dict):
    """Lightning checkpoints / the TransformerMultiGPU wrapper prefix every key with ``model.`` (models_MMT_v15_4.py:998);
    accept either form."""
    if "embed_trg.weight" not in state_dict and "model.embed_trg.weight" in state_dict:
        return {k[len("model."):]: v for k, v in state_dict.items() if k.startswith("model.")}
    return state_dict


def default_precision(config) -> str:
    """``config.precision`` ("fp32" check mode | "bf16" tensor-core mode); fp32 when unset."""
    return str(getattr(config, "precision", "fp32"))


def control_arrays(n_cols, vocab, temperature, top_k=0, top_p=1.0):
    """Per-column sampling controls for ``n_cols`` memory columns (spectra), each a scalar or a length-``n_cols``
    sequence / tensor, checked: temperature > 0 and finite, top_k an integer in [0, vocab] (0 or vocab: off), top_p in
    (0, 1] (1: off).  -> (temperature f32, top_k i32, top_p f32) numpy arrays of ``n_cols``; raises ValueError."""
    def column(name, v):
        a = np.asarray(v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else v)
        if a.ndim == 0:
            a = np.full(n_cols, a)
        if a.ndim != 1 or a.shape[0] != n_cols:
            raise ValueError(f"{name} must be a scalar or hold one value per spectrum ({n_cols}), got shape {a.shape}")
        if not (np.issubdtype(a.dtype, np.number) or a.dtype == np.bool_):
            raise ValueError(f"{name} must be numeric")
        return a
    t = column("temperature", temperature).astype(np.float32)
    if not bool(np.all(np.isfinite(t) & (t > 0))):
        raise ValueError("temperature must be > 0 and finite")
    k = column("top_k", top_k)
    if not np.issubdtype(k.dtype, np.integer):
        if not bool(np.all(np.isfinite(k) & (k == np.round(k)))):
            raise ValueError("top_k must be an integer")
    k = k.astype(np.float64)
    if not bool(np.all((k >= 0) & (k <= vocab))):
        raise ValueError(f"top_k must be in [0, {vocab}]")
    p = column("top_p", top_p).astype(np.float32)
    if not bool(np.all((p > 0) & (p <= 1))):
        raise ValueError("top_p must be in (0, 1]")
    return np.ascontiguousarray(t), np.ascontiguousarray(k.astype(np.int32)), np.ascontiguousarray(p)


def sampling_controls(n_cols, vocab, temperature, top_k=0, top_p=1.0, *, sampling="multinomial"):
    """``control_arrays``, then -> (temperature, None) when the controls are neutral -- one temperature for every column,
    top-k and top-p off: the plain decode call -- else (the first column's temperature, the arrays).  Controls that are not
    neutral need multinomial sampling (ValueError for greedy).  The defaults (a scalar temperature, top_k=0, top_p=1.0)
    return at once: the plain call checks its temperature as it always has."""
    if isinstance(temperature, (int, float)) and isinstance(top_k, int) and isinstance(top_p, (int, float)) and top_k == 0 and top_p == 1:
        return float(temperature), None
    t, k, p = control_arrays(n_cols, vocab, temperature, top_k, top_p)
    if bool(np.all(t == t[0])) and bool(np.all((k == 0) | (k == vocab))) and bool(np.all(p == 1)):
        return float(t[0]), None
    if sampling != "multinomial":
        raise ValueError("temperature per spectrum, top_k and top_p need multinomial sampling")
    return float(t[0]), (t, k, p)


def _controls_struct(ctl):
    t, k, p = ctl
    return _lib.SamplingControls(count=len(t), h_temperature=t.ctypes.data, h_top_k=k.ctypes.data, h_top_p=p.ctypes.data)


class Engine:
    """Weights of one MultimodalTransformer packed on ``device`` + the kernel drivers."""

    def __init__(self, state_dict, config, device):
        if not torch.cuda.is_available():
            raise RuntimeError("mmt_b200 needs a CUDA (sm_100a) device; there is no CPU fallback")
        self.L = _lib.lib()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError(f"mmt_b200 engine cannot run on device {device!r}; there is no CPU fallback")
        self.dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        state_dict = _normalize_state_dict(state_dict)
        self.desc = _desc_from(config, state_dict)
        L, d = self.L, C.byref(self.desc)
        n = L.mmt_weight_count(d)
        if n < 0:
            _lib.check(1)
        total = L.mmt_weight_total(d)
        blob = torch.zeros(total, dtype=torch.float32)
        for i in range(n):
            name = L.mmt_weight_name(d, i).decode()
            numel, off = L.mmt_weight_numel(d, i), L.mmt_weight_offset(d, i)
            if name not in state_dict:
                if name.startswith("real_data_linear"):
                    continue
                raise KeyError(f"state_dict lacks {name}")
            t = state_dict[name].detach().to("cpu", torch.float32).reshape(-1)
            if t.numel() != numel:
                raise ValueError(f"{name}: {t.numel()} elements, engine expects {numel}")
            blob[off:off + numel] = t
        h = C.c_void_p()
        _lib.check(L.mmt_create(d, blob.data_ptr(), total, self.dev_index, C.byref(h)))
        self.h = h
        self._finalizer = weakref.finalize(self, L.mmt_destroy, h)
        props = torch.cuda.get_device_properties(self.dev_index)
        self.sm_count = props.multi_processor_count
        self.max_threads_per_sm = props.max_threads_per_multi_processor
        self.vocab = self.desc.vocab
        import os
        self._enc_cache_on = not os.environ.get("MMT_NO_ENCODE_CACHE")
        self._enc_cache = None
        self.encode_cache_hits = 0

    # ------------------------------------------------------------------ util
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.dev_index).cuda_stream)

    def launch_count(self) -> int:
        return int(self.L.mmt_launch_count(self.h))

    def profile(self, on: bool):
        _lib.check(self.L.mmt_profile_enable(self.h, int(on)))

    def profile_report(self) -> dict:
        import json
        buf = C.create_string_buffer(1 << 16)
        _lib.check(self.L.mmt_profile_report(self.h, buf, len(buf)))
        return json.loads(buf.value.decode())

    def memory_len(self, training_mode: str) -> int:
        return int(self.L.mmt_memory_len(C.byref(self.desc), _lib.mode_bits(training_mode)))

    def philox_increment(self, n_total: int) -> int:
        return int(self.L.mmt_philox_increment(n_total * self.vocab, self.sm_count, self.max_threads_per_sm))

    # ---------------------------------------------------------------- encode
    def encode(self, data, training_mode: str, precision="fp32", want_embedding_src=False, reuse=False):
        """data: dict of CUDA tensors in the collate contract. Returns
        (memory (S,B,128), pad_mask u8 (B,S), key_bias (B,S), fingerprint (B,fp), avg (B,128), embedding_src|None).

        The engine remembers the inputs and outputs of its last encode (references, no copies).  With ``reuse=True``
        (``MultimodalTransformer.forward``: CLIP's second encode of a batch ``run_model`` has just encoded, SURVEY 8 f4)
        a call whose inputs are bit-identical to the remembered ones (device-side comparison, ``mmt_spectra_equal``)
        returns copies of the remembered outputs instead of encoding again.  ``MMT_NO_ENCODE_CACHE=1`` disables."""
        bits = _lib.mode_bits(training_mode)
        dev = self.device
        keep = []

        def f32(k):
            t = data[k].to(dev, torch.float32).contiguous()
            keep.append(t)
            return t

        sp = Spectra()
        B = None
        for m in ("1H", "13C", "HSQC", "COSY"):
            if bits & _lib.MODE_BITS[m]:
                x, mk = f32(f"src_{m}"), f32(f"mask_{m}")
                setattr(sp, f"d_src_{m}", x.data_ptr()); setattr(sp, f"d_mask_{m}", mk.data_ptr())
                B = x.shape[0]
        if B is None:
            raise TypeError("training_mode needs at least one of 1H/13C/HSQC/COSY (the reference fails on "
                            "current_batch_size=False, validate_generate_MMT_v15_4.py:122-131,165)")
        if bits & _lib.MODE_BITS["IR"]:
            sp.d_src_IR = f32("src_IR").data_ptr()
        for m in ("MF", "MS"):
            if bits & _lib.MODE_BITS[m]:
                ids = data[f"src_{m}"].to(dev, torch.int64).contiguous()
                mk = (data[f"mask_{m}"].to(dev) != 0).to(torch.uint8).contiguous()
                keep += [ids, mk]
                setattr(sp, f"d_src_{m}", ids.data_ptr()); setattr(sp, f"d_mask_{m}", mk.data_ptr())
        if bits & _lib.MODE_BITS["MW"]:
            sp.d_trg_MW = f32("trg_MW").reshape(-1).data_ptr()
        else:
            raise AttributeError("training_mode needs MW (the reference fails at trg_MW.unsqueeze, "
                                 "validate_generate_MMT_v15_4.py:118)")
        S = self.memory_len(training_mode)
        D, FP = self.desc.d_model, self.desc.fp_size
        key = (B, bits, precision)
        c = self._enc_cache
        if reuse and c is not None and c["key"] == key and all(t._version == v for t, v in c["versions"]):
            eq = C.c_int32(0)
            _lib.check(self.L.mmt_spectra_equal(self.h, C.byref(sp), C.byref(c["sp"]), B, bits, C.byref(eq), self._stream()))
            if eq.value:
                self.encode_cache_hits += 1
                memory, pad, key_bias, fp, avg, emb = c["outs"]
                if want_embedding_src and emb is None:       # embedding-only pass: one embed kernel
                    emb = torch.empty(S, B, D, device=dev, dtype=torch.float32)
                    _lib.check(self.L.mmt_encode(self.h, C.byref(sp), B, bits, _PREC[precision], None, emb.data_ptr(),
                                                 None, None, None, None, self._stream()))
                    for t in keep:
                        t.record_stream(torch.cuda.current_stream(self.dev_index))
                    c["outs"] = (memory, pad, key_bias, fp, avg, emb)
                    c["versions"] = c["versions"] + [(emb, emb._version)]
                return (memory.clone(), pad.clone(), key_bias.clone(), fp.clone(), avg.clone(),
                        emb.clone() if want_embedding_src else None)
        memory = torch.empty(S, B, D, device=dev, dtype=torch.float32)
        emb = torch.empty(S, B, D, device=dev, dtype=torch.float32) if want_embedding_src else None
        key_bias = torch.empty(B, S, device=dev, dtype=torch.float32)
        pad = torch.empty(B, S, device=dev, dtype=torch.uint8)
        fp = torch.empty(B, FP, device=dev, dtype=torch.float32)
        avg = torch.empty(B, D, device=dev, dtype=torch.float32)
        _lib.check(self.L.mmt_encode(self.h, C.byref(sp), B, bits, _PREC[precision], memory.data_ptr(),
                                     emb.data_ptr() if emb is not None else None, key_bias.data_ptr(),
                                     pad.data_ptr(), fp.data_ptr(), avg.data_ptr(), self._stream()))
        for t in keep:   # the kernels read these on the current stream
            t.record_stream(torch.cuda.current_stream(self.dev_index))
        if self._enc_cache_on:
            outs = (memory, pad, key_bias, fp, avg, emb)
            held = list(keep) + [t for t in outs if t is not None]
            self._enc_cache = dict(key=key, sp=sp, keep=keep, outs=outs, versions=[(t, t._version) for t in held])
        return memory, pad, key_bias, fp, avg, emb

    # ---------------------------------------------------------------- decode
    def _decode_args(self, memory, key_bias, n_cand, max_len, temperature, sampling, stop_on_all_pad, precision,
                     seed=0, offset=0, seq_index_base=0, n_total=0):
        if memory.dim() != 3 or memory.shape[2] != self.desc.d_model:
            raise ValueError("memory must be (S, B, 128)")
        memory = memory.to(self.device, torch.float32)
        if memory.stride(2) != 1 or memory.stride(0) % 4 or memory.stride(1) % 4 or memory.data_ptr() % 16:
            memory = memory.contiguous()
        key_bias = key_bias.to(self.device, torch.float32).contiguous()
        S, Bm = memory.shape[0], memory.shape[1]
        if tuple(key_bias.shape) != (Bm, S):
            raise ValueError(f"mask shape {tuple(key_bias.shape)} does not match memory {(Bm, S)}")
        a = DecodeArgs(d_memory=memory.data_ptr(), stride_s=memory.stride(0), stride_b=memory.stride(1),
                       d_key_bias=key_bias.data_ptr(), S=S, Bm=Bm, n_cand=n_cand, max_len=max_len,
                       temperature=float(temperature), sampling=sampling, stop_on_all_pad=int(stop_on_all_pad),
                       precision=_PREC[precision], philox_seed=seed, philox_offset=offset,
                       seq_index_base=seq_index_base, N_total=n_total, rng_sm_count=0, rng_max_threads_per_sm=0)
        return a, (memory, key_bias)

    def decode(self, memory, key_bias, *, n_cand=1, max_len=128, temperature=1.0, sampling="greedy",
               stop_on_all_pad=False, precision="fp32", seed=0, offset=0, seq_index_base=0, n_total=0, per_memory_rng=False,
               top_k=0, top_p=1.0):
        """Returns (tokens (T,N) i64, probs (T,N) f32, steps) with T == max_len rows allocated.  ``per_memory_rng``: the
        n_cand candidates of each memory column draw as one torch.multinomial((n_cand, V), 1) call per step, the columns'
        calls in order (``mmt_decode_memory_streams``); multinomial only, seq_index_base a multiple of n_cand.
        ``temperature`` / ``top_k`` / ``top_p``: a scalar or one value per memory column (``control_arrays``); controls
        that are not neutral run ``decode_controlled``."""
        temperature, ctl = sampling_controls(memory.shape[1], self.vocab, temperature, top_k, top_p, sampling=sampling)
        if ctl is not None:
            return self.decode_controlled(memory, key_bias, n_cand=n_cand, max_len=max_len, temperature=ctl[0], top_k=ctl[1],
                                          top_p=ctl[2], precision=precision, seed=seed, offset=offset,
                                          seq_index_base=seq_index_base, n_total=n_total, per_memory_rng=per_memory_rng)[:3]
        smp = _lib.SAMPLE_GREEDY if sampling == "greedy" else _lib.SAMPLE_MULTINOMIAL
        if per_memory_rng and (smp != _lib.SAMPLE_MULTINOMIAL or seq_index_base % n_cand):
            raise ValueError("per_memory_rng needs multinomial sampling and seq_index_base a multiple of n_candidates")
        a, keep = self._decode_args(memory, key_bias, n_cand, max_len, temperature, smp, stop_on_all_pad, precision,
                                    seed, offset, seq_index_base, n_total)
        N = a.Bm * n_cand
        tokens = torch.empty(max_len, N, device=self.device, dtype=torch.int64)
        probs = torch.empty(max_len, N, device=self.device, dtype=torch.float32)
        steps = C.c_int32(max_len)
        fn = self.L.mmt_decode_memory_streams if per_memory_rng else self.L.mmt_decode
        _lib.check(fn(self.h, C.byref(a), tokens.data_ptr(), probs.data_ptr(), C.byref(steps), self._stream()))
        for t in keep:
            t.record_stream(torch.cuda.current_stream(self.dev_index))
        return tokens, probs, int(steps.value)

    def decode_until_eos(self, memory, key_bias, *, eos, n_cand=1, max_len=128, temperature=1.0, sampling="greedy",
                         stop_on_all_pad=False, precision="fp32", seed=0, offset=0, seq_index_base=0, n_total=0,
                         per_memory_rng=False, top_k=0, top_p=1.0):
        """``decode`` that stops computing a sequence once it has emitted ``eos`` (``mmt_decode_until_eos``).  Returns
        (tokens (T,N) i64, probs (T,N) f32, steps, lengths (N,) i32, rows (T,) i64 on the host): ids and probabilities
        equal ``decode``'s up to and including each sequence's first ``eos`` and are <PAD> / 0 after it (and from
        ``steps`` on); ``lengths`` = position of that first ``eos`` (max_len if none); ``rows`` = decode-step rows
        computed at each position.  Sampling controls as ``decode``."""
        temperature, ctl = sampling_controls(memory.shape[1], self.vocab, temperature, top_k, top_p, sampling=sampling)
        if ctl is not None:
            return self.decode_controlled(memory, key_bias, eos=eos, n_cand=n_cand, max_len=max_len, temperature=ctl[0],
                                          top_k=ctl[1], top_p=ctl[2], precision=precision, seed=seed, offset=offset,
                                          seq_index_base=seq_index_base, n_total=n_total, per_memory_rng=per_memory_rng)
        smp = _lib.SAMPLE_GREEDY if sampling == "greedy" else _lib.SAMPLE_MULTINOMIAL
        if per_memory_rng and (smp != _lib.SAMPLE_MULTINOMIAL or seq_index_base % n_cand):
            raise ValueError("per_memory_rng needs multinomial sampling and seq_index_base a multiple of n_candidates")
        a, keep = self._decode_args(memory, key_bias, n_cand, max_len, temperature, smp, stop_on_all_pad, precision,
                                    seed, offset, seq_index_base, n_total)
        N = a.Bm * n_cand
        tokens = torch.empty(max_len, N, device=self.device, dtype=torch.int64)
        probs = torch.empty(max_len, N, device=self.device, dtype=torch.float32)
        lengths = torch.empty(N, device=self.device, dtype=torch.int32)
        rows = torch.zeros(max_len, dtype=torch.int64)
        steps = C.c_int32(max_len)
        _lib.check(self.L.mmt_decode_until_eos(self.h, C.byref(a), int(per_memory_rng), int(eos), tokens.data_ptr(),
                                               probs.data_ptr(), lengths.data_ptr(), C.byref(steps), rows.data_ptr(),
                                               self._stream()))
        for t in keep:
            t.record_stream(torch.cuda.current_stream(self.dev_index))
        return tokens, probs, int(steps.value), lengths, rows

    def decode_controlled(self, memory, key_bias, *, n_cand=1, max_len=128, temperature=1.0, top_k=0, top_p=1.0, eos=None,
                          precision="fp32", seed=0, offset=0, seq_index_base=0, n_total=0, per_memory_rng=False):
        """Multinomial decode with per-column sampling controls (``mmt_decode_controlled``), also when they are neutral:
        at temperature[b] (a scalar or one per memory column), from the kept set of top_k[b] / top_p[b]
        (``mmt_sampling_controls``: HF order, ties by lower index).  The reported probabilities are softmax(logits /
        temperature[b]) of the chosen token, NOT renormalised over the kept set: where a draw equals the plain call's, so
        does its probability, and probabilities stay comparable across columns.  The generator advance is the plain
        call's.  -> (tokens, probs, steps), and with ``eos`` (``decode_until_eos``) also (lengths, rows)."""
        if per_memory_rng and seq_index_base % n_cand:
            raise ValueError("per_memory_rng needs seq_index_base a multiple of n_candidates")
        ctl = control_arrays(memory.shape[1], self.vocab, temperature, top_k, top_p)
        a, keep = self._decode_args(memory, key_bias, n_cand, max_len, float(ctl[0][0]), _lib.SAMPLE_MULTINOMIAL, False,
                                    precision, seed, offset, seq_index_base, n_total)
        N = a.Bm * n_cand
        tokens = torch.empty(max_len, N, device=self.device, dtype=torch.int64)
        probs = torch.empty(max_len, N, device=self.device, dtype=torch.float32)
        lengths = torch.empty(N, device=self.device, dtype=torch.int32) if eos is not None else None
        rows = torch.zeros(max_len, dtype=torch.int64)
        steps = C.c_int32(max_len)
        c = _controls_struct(ctl)
        _lib.check(self.L.mmt_decode_controlled(self.h, C.byref(a), int(per_memory_rng), -1 if eos is None else int(eos), C.byref(c),
                                                tokens.data_ptr(), probs.data_ptr(), lengths.data_ptr() if lengths is not None else None,
                                                C.byref(steps), rows.data_ptr(), self._stream()))
        for t in keep:
            t.record_stream(torch.cuda.current_stream(self.dev_index))
        if eos is None:
            return tokens, probs, int(steps.value)
        return tokens, probs, int(steps.value), lengths, rows

    def teacher_forced(self, memory, key_bias, trg, *, n_cand=1, precision="fp32"):
        """trg (T,N) i64 -> logits (T,N,V)."""
        trg = trg.to(self.device, torch.int64).contiguous()
        T, N = trg.shape
        a, keep = self._decode_args(memory, key_bias, n_cand, max(T, 1), 1.0, 0, False, precision)
        if a.Bm * n_cand != N:
            raise ValueError("target batch does not match memory batch")
        logits = torch.empty(T, N, self.vocab, device=self.device, dtype=torch.float32)
        _lib.check(self.L.mmt_teacher_forced(self.h, C.byref(a), trg.data_ptr(), T, logits.data_ptr(), self._stream()))
        for t in keep + (trg,):
            t.record_stream(torch.cuda.current_stream(self.dev_index))
        return logits

    def teacher_forced_scores(self, memory, key_bias, trg_in, target=None, *, n_cand=1, temperature=1.0, sampling="greedy",
                              precision="fp32", seed=0, offset=0):
        """trg_in (T,N) forced inputs -> (pick (T,N) i64, pick_prob (T,N) f32, target_prob (T,N) f32 | None)."""
        trg_in = trg_in.to(self.device, torch.int64).contiguous()
        T, N = trg_in.shape
        smp = _lib.SAMPLE_GREEDY if sampling == "greedy" else _lib.SAMPLE_MULTINOMIAL
        a, keep = self._decode_args(memory, key_bias, n_cand, max(T, 1), temperature, smp, False, precision, seed, offset)
        if a.Bm * n_cand != N:
            raise ValueError("target batch does not match memory batch")
        pick = torch.empty(T, N, device=self.device, dtype=torch.int64)
        pick_prob = torch.empty(T, N, device=self.device, dtype=torch.float32)
        tgt = tprob = None
        if target is not None:
            tgt = target.to(self.device, torch.int64).contiguous()
            if tuple(tgt.shape) != (T, N):
                raise ValueError("target must have the shape of trg_in")
            tprob = torch.empty(T, N, device=self.device, dtype=torch.float32)
        _lib.check(self.L.mmt_teacher_forced_scores(self.h, C.byref(a), trg_in.data_ptr(), tgt.data_ptr() if tgt is not None else None, T,
                                                    pick.data_ptr(), pick_prob.data_ptr(), tprob.data_ptr() if tprob is not None else None,
                                                    self._stream()))
        for t in keep + (trg_in,) + ((tgt,) if tgt is not None else ()):
            t.record_stream(torch.cuda.current_stream(self.dev_index))
        return pick, pick_prob, tprob

    def beam_search(self, memory, key_bias, *, beam_size, gen_len, eos=2, precision="fp32"):
        """-> (seq (Bm,K,gen_len+1) i64, len (Bm,K) i32, score (Bm,K) f64, probs (Bm,K,gen_len) f32, steps)."""
        a, keep = self._decode_args(memory, key_bias, beam_size, gen_len, 1.0, 0, False, precision)
        Bm, K, T = a.Bm, beam_size, gen_len
        seq = torch.empty(Bm, K, T + 1, device=self.device, dtype=torch.int64)
        ln = torch.empty(Bm, K, device=self.device, dtype=torch.int32)
        score = torch.empty(Bm, K, device=self.device, dtype=torch.float64)
        probs = torch.empty(Bm, K, T, device=self.device, dtype=torch.float32)
        steps = C.c_int32(T)
        _lib.check(self.L.mmt_beam_search(self.h, C.byref(a), K, T, eos, seq.data_ptr(), ln.data_ptr(), score.data_ptr(),
                                          probs.data_ptr(), C.byref(steps), self._stream()))
        for t in keep:
            t.record_stream(torch.cuda.current_stream(self.dev_index))
        return seq, ln, score, probs, int(steps.value)

    def sample_without_replacement(self, memory, key_bias, *, n_cand, max_len, temperature=1.0, eos=2, seed=0, offset=0,
                                   seq_index_base=0, n_total=0, precision="fp32"):
        """Stochastic beam search (``mmt_sample_without_replacement``): ``n_cand`` distinct sequences per memory column,
        an exact sample without replacement from the decoder's sampling distribution at ``temperature`` (a scalar or one
        per memory column), slot 0 first.  The generator state (seed, offset) is read, not advanced.
        -> (tokens (T,N) i64, probs (T,N) f32, lengths (N,) i32, log_prob (N,) f64, key (N,) f64, steps)."""
        temp = control_arrays(memory.shape[1], self.vocab, temperature)[0]
        a, keep = self._decode_args(memory, key_bias, n_cand, max_len, float(temp[0]), _lib.SAMPLE_MULTINOMIAL, False,
                                    precision, seed, offset, seq_index_base, n_total)
        N = a.Bm * n_cand
        tokens = torch.empty(max_len, N, device=self.device, dtype=torch.int64)
        probs = torch.empty(max_len, N, device=self.device, dtype=torch.float32)
        lengths = torch.empty(N, device=self.device, dtype=torch.int32)
        log_prob = torch.empty(N, device=self.device, dtype=torch.float64)
        key = torch.empty(N, device=self.device, dtype=torch.float64)
        steps = C.c_int32(max_len)
        _lib.check(self.L.mmt_sample_without_replacement(self.h, C.byref(a), temp.ctypes.data, int(eos), tokens.data_ptr(),
                                                         probs.data_ptr(), lengths.data_ptr(), log_prob.data_ptr(),
                                                         key.data_ptr(), C.byref(steps), self._stream()))
        for t in keep:
            t.record_stream(torch.cuda.current_stream(self.dev_index))
        return tokens, probs, lengths, log_prob, key, int(steps.value)

    # ------------------------------------------------------------ unit hooks
    def sbs_select_step(self, logits, phi, key, lengths, hist, probs, *, k, step, eos, temperature, seed, offset,
                        seq_index_base=0):
        """One selection step of ``sample_without_replacement`` on given logits (Bm*k, V) and slot state: phi / key
        (Bm*k,) f64 (-inf: empty slot), lengths (Bm*k,) i32, hist (Bm*k, T) u8 ids, probs (Bm*k, T) f32
        (``mmt_sbs_select_step``, test hook).  -> the new (phi, key, lengths, hist, probs) and p (Bm*k, V) f32, the
        softmax the step computed for every live, unfinished slot (0 in other rows)."""
        dev = self.device
        lg = logits.to(dev, torch.float32).contiguous()
        N, V = lg.shape
        st = [phi.to(dev, torch.float64).contiguous(), key.to(dev, torch.float64).contiguous(),
              lengths.to(dev, torch.int32).contiguous(), hist.to(dev, torch.uint8).contiguous(),
              probs.to(dev, torch.float32).contiguous()]
        T = st[3].shape[1]
        temp = control_arrays(N // k, V, temperature)[0]
        out = [torch.empty_like(t) for t in st]
        p = torch.zeros(N, V, device=dev, dtype=torch.float32)
        _lib.check(self.L.mmt_sbs_select_step(self.h, lg.data_ptr(), N // k, k, V, T, step, eos, temp.ctypes.data, seed, offset,
                                              seq_index_base, 0, 0, *[t.data_ptr() for t in st], *[t.data_ptr() for t in out],
                                              p.data_ptr(), self._stream()))
        for t in st + [lg]:
            t.record_stream(torch.cuda.current_stream(self.dev_index))
        return tuple(out) + (p,)

    def sample(self, x, temperature=1.0, sampling="greedy", seed=0, offset=0, seq_index_base=0, n_total=0,
               want_logits=False):
        x = x.to(self.device, torch.float32).contiguous()
        N = x.shape[0]
        tok = torch.empty(N, device=self.device, dtype=torch.int64)
        pr = torch.empty(N, device=self.device, dtype=torch.float32)
        lg = torch.empty(N, self.vocab, device=self.device, dtype=torch.float32) if want_logits else None
        smp = _lib.SAMPLE_GREEDY if sampling == "greedy" else _lib.SAMPLE_MULTINOMIAL
        _lib.check(self.L.mmt_sample(self.h, x.data_ptr(), N, float(temperature), smp, seed, offset, seq_index_base,
                                     n_total, 0, 0, tok.data_ptr(), pr.data_ptr(),
                                     lg.data_ptr() if lg is not None else None, self._stream()))
        return tok, pr, lg

    def exponential(self, n, *, seed, offset, elem_base=0, numel_total=0):
        """The Exp(1) variates torch.empty(numel_total).exponential_() holds at [elem_base, elem_base + n) (test hook)."""
        q = torch.empty(n, device=self.device, dtype=torch.float32)
        _lib.check(self.L.mmt_exponential(seed, offset, elem_base, n, numel_total or n, self.sm_count, self.max_threads_per_sm,
                                          q.data_ptr(), self._stream()))
        return q

    def sample_probs(self, p, *, seed, offset, seq_index_base=0, n_total=0):
        """torch.multinomial(p, 1) on given probabilities p (N,V) under generator state (seed, offset) (test hook)."""
        p = p.to(self.device, torch.float32).contiguous()
        N, V = p.shape
        tok = torch.empty(N, device=self.device, dtype=torch.int64)
        _lib.check(self.L.mmt_sample_probs(p.data_ptr(), N, V, seed, offset, seq_index_base, n_total, self.sm_count,
                                           self.max_threads_per_sm, tok.data_ptr(), self._stream()))
        return tok

    def sample_memory_streams(self, *, x=None, p=None, n_cand, max_len, step=0, temperature=1.0, seed, offset,
                              seq_index_base=0):
        """Per-memory RNG streams at one step (test hook): from hidden states x (N,128) through the fused sampler ->
        (ids, probabilities), or from probabilities p (N,V) -> (ids, None)."""
        src = (x if p is None else p).to(self.device, torch.float32).contiguous()
        N = src.shape[0]
        tok = torch.empty(N, device=self.device, dtype=torch.int64)
        pr = torch.empty(N, device=self.device, dtype=torch.float32) if p is None else None
        _lib.check(self.L.mmt_sample_memory_streams(self.h, src.data_ptr() if p is None else None, src.data_ptr() if p is not None else None,
                                                    N, n_cand, max_len, step, float(temperature), seed, offset, seq_index_base,
                                                    0, 0, tok.data_ptr(), pr.data_ptr() if pr is not None else None, self._stream()))
        return tok, pr

    def sample_controlled(self, *, x=None, p=None, n_cand=1, temperature=1.0, top_k=0, top_p=1.0, per_memory_rng=False,
                          max_len=1, step=0, seed=0, offset=0, seq_index_base=0, n_total=0, want_logits=False, want_kept=False):
        """The controlled pick at one step (``mmt_sample_controlled``, test hook): rows n of x (N,128) hidden states or
        of p (N,V) probabilities, control column n // n_cand (controls: a scalar or one per column).
        -> (ids (N,), probabilities (N,) of the chosen token, logits (N,V) | None, kept (N,V) u8 | None)."""
        src = (x if p is None else p).to(self.device, torch.float32).contiguous()
        N = src.shape[0]
        ctl = control_arrays((N + n_cand - 1) // n_cand, self.vocab, temperature, top_k, top_p)
        tok = torch.empty(N, device=self.device, dtype=torch.int64)
        pr = torch.empty(N, device=self.device, dtype=torch.float32)
        lg = torch.empty(N, self.vocab, device=self.device, dtype=torch.float32) if want_logits and p is None else None
        kept = torch.empty(N, self.vocab, device=self.device, dtype=torch.uint8) if want_kept else None
        c = _controls_struct(ctl)
        _lib.check(self.L.mmt_sample_controlled(self.h, src.data_ptr() if p is None else None, src.data_ptr() if p is not None else None,
                                                N, n_cand, C.byref(c), int(per_memory_rng), max_len, step, seed, offset, seq_index_base,
                                                n_total, 0, 0, tok.data_ptr(), pr.data_ptr(), lg.data_ptr() if lg is not None else None,
                                                kept.data_ptr() if kept is not None else None, self._stream()))
        return tok, pr, lg, kept

    def linear(self, A, W, bias=None, act=0, precision="fp32"):
        A = A.to(self.device, torch.float32).contiguous()
        W = W.to(self.device, torch.float32).contiguous()
        b = bias.to(self.device, torch.float32).contiguous() if bias is not None else None
        M, K = A.shape
        N = W.shape[0]
        out = torch.empty(M, N, device=self.device, dtype=torch.float32)
        _lib.check(self.L.mmt_linear(self.h, A.data_ptr(), W.data_ptr(), b.data_ptr() if b is not None else None,
                                     out.data_ptr(), M, N, K, act, _PREC[precision], self._stream()))
        return out

    def ffn(self, x, w1, b1, w2, b2, gamma, beta, splits=1, weight_terms=2):
        """LN(x + W2 relu(W1 bf16(x) + b1) + b2): the fused tensor-core FFN block, stand-alone (weight_terms: 2 = hi + lo
        bf16 terms, 1 = hi term only, the decoder's variant)."""
        t = [v.to(self.device, torch.float32).contiguous() for v in (x, w1, b1, w2, b2, gamma, beta)]
        M, F = t[0].shape[0], t[1].shape[0]
        out = torch.empty_like(t[0])
        _lib.check(self.L.mmt_ffn(self.h, *[v.data_ptr() for v in t], out.data_ptr(), M, F, splits, weight_terms, self._stream()))
        return out

    def decode_self_attention(self, layer, x, precision="bf16"):
        """x (T,N,128): input rows of decoder layer ``layer`` at positions 0..T-1 -> (T,N,128) f32 self-attention output
        (before out_proj) of every position over keys 0..t, through the un-fused decode step's QKV projection, paged KV
        cache and attention kernel (test hook)."""
        x = x.to(self.device, torch.float32).contiguous()
        T, N, _ = x.shape
        out = torch.empty_like(x)
        _lib.check(self.L.mmt_decode_self_attention(self.h, layer, x.data_ptr(), N, T, _PREC[precision], out.data_ptr(),
                                                    self._stream()))
        return out

    def decode_cross_attention(self, layer, memory, key_bias, q, *, n_cand=1, precision="bf16"):
        """q (Bm*n_cand,128) queries of decoder layer ``layer`` over memory (S,Bm,128) with the additive key_bias (Bm,S)
        -> (Bm*n_cand,128) f32 cross-attention output (before out_proj), through the un-fused decode step's memory
        preparation and attention kernel (test hook)."""
        a, keep = self._decode_args(memory, key_bias, n_cand, 1, 1.0, 0, False, precision)
        q = q.to(self.device, torch.float32).contiguous()
        if tuple(q.shape) != (a.Bm * n_cand, self.desc.d_model):
            raise ValueError("q must be (Bm * n_cand, 128)")
        out = torch.empty_like(q)
        _lib.check(self.L.mmt_decode_cross_attention(self.h, C.byref(a), layer, q.data_ptr(), out.data_ptr(), self._stream()))
        for t in keep:
            t.record_stream(torch.cuda.current_stream(self.dev_index))
        return out

    def decode_layer_tail(self, layer, x, att_self, att_cross, precision="bf16"):
        """The rest of decoder layer ``layer`` of the un-fused decode step after its attentions, on R rows (test hook):
        x, att_self, att_cross (R,128) -> (x1, qc, x2, out), f32 (R,128): x1 = norm1(x + out_proj(att_self)), qc its
        cross-attention query, x2 = norm2(x1 + ca_out_proj(att_cross)), out = norm3(x2 + FFN(x2)).  x2 is None where the
        step keeps it inside the FFN kernel (bf16, R >= 2048, FFN prologue on)."""
        t = [v.to(self.device, torch.float32).contiguous() for v in (x, att_self, att_cross)]
        R = t[0].shape[0]
        if any(tuple(v.shape) != (R, self.desc.d_model) for v in t):
            raise ValueError("x, att_self and att_cross must be (R, 128)")
        x1, qc, out = (torch.empty_like(t[0]) for _ in range(3))
        x2 = torch.full_like(t[0], float("nan"))
        _lib.check(self.L.mmt_decode_layer_tail(self.h, layer, *[v.data_ptr() for v in t], R, _PREC[precision], x1.data_ptr(),
                                                qc.data_ptr(), x2.data_ptr(), out.data_ptr(), self._stream()))
        for v in t:
            v.record_stream(torch.cuda.current_stream(self.dev_index))
        if bool(torch.isnan(x2).all()):
            x2 = None
        return x1, qc, x2, out

    def encoder_layer(self, stack, layer, x, *, key_bias=None, row_start=None, cnt=None, kidx=None, nk=None, S=None,
                      precision="bf16"):
        """Layer ``layer`` of encoder stack ``stack`` (0-4 the modality stacks, 5 encoder_cross) on the rows x (R,128),
        through the encoder's own layer code and attention kernel (test hook).  Dense layout: key_bias (B,S) additive, x
        holds B*S rows.  Ragged layout: row_start / cnt / nk (B,) and kidx (B,kstride) int, sequence b owns rows
        row_start[b] .. + cnt[b] - 1 and attends rows row_start[b] + kidx[b, :nk[b]] (S: bound of cnt, default max cnt).
        -> (qkv (R,384), attention output before out_proj (R,128), layer output after norm2 (R,128)), f32."""
        x = x.to(self.device, torch.float32).contiguous()
        R = x.shape[0]
        keep = [x]
        if key_bias is not None:
            key_bias = key_bias.to(self.device, torch.float32).contiguous()
            B, S = key_bias.shape
            ptrs, kstride = [key_bias.data_ptr(), None, None, None, None], 0
            keep.append(key_bias)
        else:
            ints = [t.to(self.device, torch.int32).contiguous() for t in (row_start, cnt, kidx, nk)]
            keep += ints
            B, kstride = ints[2].shape
            S = S or int(ints[1].max())
            ptrs = [None] + [t.data_ptr() for t in ints]
        qkv = torch.empty(R, 3 * self.desc.d_model, device=self.device, dtype=torch.float32)
        att, out = torch.empty_like(x), torch.empty_like(x)
        _lib.check(self.L.mmt_encoder_layer(self.h, stack, layer, x.data_ptr(), R, B, S, *ptrs, kstride, _PREC[precision],
                                            qkv.data_ptr(), att.data_ptr(), out.data_ptr(), self._stream()))
        for t in keep:
            t.record_stream(torch.cuda.current_stream(self.dev_index))
        return qkv, att, out

    def pack_tokens(self, tokens):
        tokens = tokens.contiguous()
        out = torch.empty(tokens.shape, device=self.device, dtype=torch.uint8)
        _lib.check(self.L.mmt_pack_tokens_u8(tokens.data_ptr(), tokens.numel(), out.data_ptr(), self._stream()))
        return out

    def pack_tokens_seqmajor(self, tokens, out=None):
        """(T,N) i64 ids -> (N,T) u8 (the scheduler's all-gather payload: rank blocks land in their final order)."""
        tokens = tokens.contiguous()
        T, N = tokens.shape
        if out is None:
            out = torch.empty(N, T, device=self.device, dtype=torch.uint8)
        _lib.check(self.L.mmt_pack_tokens_u8_seqmajor(tokens.data_ptr(), T, N, out.data_ptr(), self._stream()))
        return out

    def unpack_tokens_seqmajor(self, packed, n):
        """First ``n`` rows of a (>= n, T) u8 buffer -> (T,n) i64."""
        packed = packed.contiguous()
        T = packed.shape[1]
        out = torch.empty(T, n, device=self.device, dtype=torch.int64)
        _lib.check(self.L.mmt_unpack_tokens_u8_seqmajor(packed.data_ptr(), T, n, out.data_ptr(), self._stream()))
        return out

    def unpack_tokens(self, packed):
        packed = packed.contiguous()
        out = torch.empty(packed.shape, device=self.device, dtype=torch.int64)
        _lib.check(self.L.mmt_unpack_tokens_u8(packed.data_ptr(), packed.numel(), out.data_ptr(), self._stream()))
        return out


# one engine per (model object, parameter version): callers pass a live nn.Module every
# call, exactly like the reference's functions (SURVEY.md 8b), never weights.
_ENGINES = weakref.WeakKeyDictionary()


def _param_version(model):
    return tuple((p.data_ptr(), p._version) for p in model.parameters())


def engine_for(model, config) -> Engine:
    dev = torch.device(getattr(config, "device", "cuda"))
    if dev.type != "cuda":
        raise RuntimeError(f"config.device={dev} - the B200 engine has no CPU path")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    ver = (_param_version(model), str(dev))
    hit = _ENGINES.get(model)
    if hit is not None and hit[0] == ver:
        return hit[1]
    eng = Engine(model.state_dict(), getattr(model, "config", config), dev)
    _ENGINES[model] = (ver, eng)
    return eng
