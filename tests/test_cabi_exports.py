"""CPU-side checks of the boundary: the shared library builds, loads and exports every
symbol include/mmt_b200.h declares; weight table matches the reference state_dict."""
import ctypes
import json
import os
import re
import subprocess

from multimodalspectraltransformer_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_all_exported():
    hdr = open(os.path.join(ROOT, "include", "mmt_b200.h")).read()
    declared = set(re.findall(r"\b(mmt_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    path = _lib.build()
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True).stdout
    for s in declared:
        assert f" T {s}" in out, s


def test_library_loads_and_weight_table_matches_reference_state_dict():
    L = _lib.lib()
    assert L.mmt_abi_version() == 2
    from multimodalspectraltransformer_b200.engine import _desc_from
    from multimodalspectraltransformer_b200.config import default_config
    d = _desc_from(default_config())
    meta = json.load(open(os.path.join(ROOT, "tests", "golden", "weights_meta.json")))
    n = L.mmt_weight_count(ctypes.byref(d))
    names = [L.mmt_weight_name(ctypes.byref(d), i).decode() for i in range(n)]
    assert set(names) == set(meta["keys"])
    for i, name in enumerate(names):
        shape = meta["shapes"][name]
        numel = 1
        for s in shape:
            numel *= s
        assert L.mmt_weight_numel(ctypes.byref(d), i) == numel
        assert L.mmt_weight_offset(ctypes.byref(d), i) % 64 == 0
    # every weight has its own slot: sorted by offset, each ends before the next begins, the last within the total
    slots = sorted((L.mmt_weight_offset(ctypes.byref(d), i), L.mmt_weight_numel(ctypes.byref(d), i), names[i]) for i in range(n))
    for (o0, n0, a), (o1, _, b) in zip(slots, slots[1:]):
        assert o0 >= 0 and o0 + n0 <= o1, (a, b)
    assert slots[-1][0] + slots[-1][1] <= L.mmt_weight_total(ctypes.byref(d))
    assert L.mmt_memory_len(ctypes.byref(d), _lib.mode_bits("1H_13C_HSQC_COSY_IR_MF_MW")) == 582
    assert L.mmt_memory_len(ctypes.byref(d), _lib.mode_bits("HSQC_MF_MW")) == 518
    assert L.mmt_mask_is_float(_lib.mode_bits("HSQC_MF_MW")) == 1
    assert L.mmt_mask_is_float(_lib.mode_bits("1H_13C_HSQC_COSY_MF_MW")) == 0
    # torch's Philox offset policy (DistributionTemplates.h calc_execution_policy)
    assert L.mmt_philox_increment(128 * 43, 148, 2048) == 4
    assert L.mmt_philox_increment(131072 * 43, 148, 2048) == 20


def test_no_cpu_fallback():
    import pytest
    import torch
    import multimodalspectraltransformer_b200 as M
    from multimodalspectraltransformer_b200 import synthetic
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    cfg = M.default_config(device="cuda", num_encoder_layers=1, num_decoder_layers=1)
    model = M.MultimodalTransformer(cfg)
    with pytest.raises(RuntimeError):
        M.run_model(model, synthetic.make_spectra(2), cfg)


def test_model_desc_follows_the_weights_not_the_mutable_config():
    """Callers lower config.max_len mid-run (mmt_result_test_functions_15_4.py:547) on the very namespace the model was
    built from; the engine's hyper-parameters must keep describing the model (pe_trg rows, layer counts, vocab sizes)."""
    import multimodalspectraltransformer_b200 as M
    from multimodalspectraltransformer_b200.engine import _desc_from
    cfg = M.default_config(device="cpu")
    model = M.MultimodalTransformer(cfg)
    cfg.max_len, cfg.num_decoder_layers, cfg.out_size, cfg.input_dim_IR = 12, 2, 7, 10
    d = _desc_from(cfg, model.state_dict())
    assert (d.max_len, d.n_dec_layers, d.n_enc_layers, d.vocab, d.ir_bins, d.mf_vocab, d.fp_size, d.d_ff, d.d_model) == \
        (128, 6, 6, 43, 1000, 212, 512, 2048, 128)
    d0 = _desc_from(M.default_config(device="cpu"))
    assert (d0.max_len, d0.n_dec_layers, d0.vocab) == (128, 6, 43)


def test_lightning_prefixed_state_dict_is_accepted():
    import multimodalspectraltransformer_b200 as M
    from multimodalspectraltransformer_b200.engine import _desc_from, _normalize_state_dict
    model = M.MultimodalTransformer(M.default_config(device="cpu"))
    sd = model.state_dict()
    wrapped = {"model." + k: v for k, v in sd.items()}
    un = _normalize_state_dict(wrapped)
    assert list(un.keys()) == list(sd.keys()) and _normalize_state_dict(sd) is sd
    assert _desc_from(M.default_config(device="cpu"), un).max_len == 128
