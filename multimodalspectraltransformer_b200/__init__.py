"""B200-native engine for the MMT candidate-generation hot path.

Mirrors the reference's Python interface for that path (same names, arguments and
return layouts); everything behind it is hand-written sm_100a CUDA reached through
the C ABI in include/mmt_b200.h.  No CPU fallback.
"""
from .model import MultimodalTransformer  # noqa: F401
from .generate import (run_model, greedy_sequence, greedy_sequence_2, multinomial_sequence,  # noqa: F401
                       multinomial_sequence_multi, multinomial_sequence_multi_2, duplicate_tensor,
                       duplicate_dict, teacher_forced_logits, beam_search, predict_prop_correct_max_sequence,
                       predict_prop_correct_max_sequence_2, predict_prop_correct_max_sequence_3, sample_without_replacement)
from .smiles import tensor_to_smiles, tensor_to_smiles_and_prob, tensor_to_smiles_and_prob_2, distinct_smiles  # noqa: F401
from .config import load_config, default_config  # noqa: F401

__all__ = ["MultimodalTransformer", "run_model", "greedy_sequence", "greedy_sequence_2", "multinomial_sequence",
           "multinomial_sequence_multi", "multinomial_sequence_multi_2", "duplicate_tensor", "duplicate_dict",
           "teacher_forced_logits", "beam_search", "predict_prop_correct_max_sequence", "predict_prop_correct_max_sequence_2",
           "predict_prop_correct_max_sequence_3", "sample_without_replacement", "tensor_to_smiles", "tensor_to_smiles_and_prob", "tensor_to_smiles_and_prob_2", "distinct_smiles",
           "load_config", "default_config"]
