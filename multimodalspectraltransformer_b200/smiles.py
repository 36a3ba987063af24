"""ids -> SMILES strings + truncated token probabilities, the reference's post-processing of the
generated tensors (reference utils_MMT/helper_functions_pl_v15_4.py):

    tensor_to_smiles              :247-269
    tensor_to_smiles_and_prob     :272-301
    tensor_to_smiles_and_prob_2   :390-419

The reference walks the tensors element by element with ``.item()`` (one device-to-host sync per
token).  Here the first-<EOS> scan runs on the device (``mmt_first_eos``), the ids cross to the
host once as bytes, and only the string join and the probability slicing remain in Python.  Same
arguments, same return layouts.

``distinct_smiles`` goes further for candidate generation: the distinct strings of every memory column, with their
first candidate and multiplicity, deduplicated on the device (``mmt_distinct_smiles``) so that the host only decodes
the strings that survive.
"""
from __future__ import annotations

import ctypes as C
from typing import NamedTuple, Optional

import torch

from . import _lib


def _eos_id(itos) -> int:
    for k, v in itos.items():
        if v == "<EOS>":
            return int(k)
    raise KeyError("<EOS> not in itos")


def _lengths_and_ids(tensor, eos):
    """(T,N) ids on a CUDA device -> (first-EOS position per column as list, ids as a CPU uint8/int64 array)."""
    t = tensor if tensor.dim() == 2 else tensor.unsqueeze(1)
    t = t.to(torch.int64).contiguous()
    T, N = t.shape
    if not t.is_cuda:
        # ids the caller already moved to the host (the reference's helpers take either, helper_functions_pl_v15_4.py:247-301):
        # the scan is a host-side index computation on data that is already there -- no kernel, nothing copied back and forth
        is_eos = (t == eos)
        first = torch.where(is_eos.any(dim=0), is_eos.to(torch.uint8).argmax(dim=0), torch.full((N,), T, dtype=torch.int64))
        return first.tolist(), t.numpy()
    lens = torch.empty(N, dtype=torch.int32, device=t.device)
    stream = C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)
    _lib.check(_lib.lib().mmt_first_eos(t.data_ptr(), T, N, eos, lens.data_ptr(), stream))
    ids = t.to(torch.uint8) if int(T) and eos < 256 else t
    return lens.cpu().tolist(), ids.cpu().numpy()


def tensor_to_smiles(tensor, itos):
    """(T,N) -> list of N strings; (T,) -> one string."""
    lens, ids = _lengths_and_ids(tensor, _eos_id(itos))
    out = ["".join(itos[str(int(v))] for v in ids[:lens[i], i]) for i in range(ids.shape[1])]
    return out if tensor.dim() > 1 else out[0]


def tensor_to_smiles_and_prob(tensor, token_prob, itos):
    """tensor (T,N), token_prob (N,T') -> (strings, [token_prob[i, :eos_i]]); 1-D input -> (string, prob[:eos])."""
    lens, ids = _lengths_and_ids(tensor, _eos_id(itos))
    if tensor.dim() > 1:
        seqs = ["".join(itos[str(int(v))] for v in ids[:lens[i], i]) for i in range(ids.shape[1])]
        return seqs, [token_prob[i, :lens[i]] for i in range(ids.shape[1])]
    smi = "".join(itos[str(int(v))] for v in ids[:lens[0], 0])
    return smi, torch.stack(list(token_prob[:lens[0]]))


def tensor_to_smiles_and_prob_2(tensor, token_prob, itos):
    """tensor (T,N), token_prob (T',N) -> (strings, [token_prob[:len_i, i]]); 1-D input -> (string, prob[:len])."""
    lens, ids = _lengths_and_ids(tensor, _eos_id(itos))
    if tensor.dim() > 1 and token_prob.dim() > 1:
        seqs = ["".join(itos[str(int(v))] for v in ids[:lens[i], i]) for i in range(ids.shape[1])]
        return seqs, [token_prob[:lens[i], i] for i in range(ids.shape[1])]
    smi = "".join(itos[str(int(v))] for v in ids[:lens[0], 0])
    return smi, torch.stack(list(token_prob[:lens[0]]))


class DistinctSmiles(NamedTuple):
    """One distinct string of a memory column: ``index`` is its first candidate inside the column, ``count`` how many
    candidates spell it, ``prob`` the first candidate's ``token_prob[:len, i]`` (None without token_prob)."""
    smiles: str
    index: int
    count: int
    prob: Optional[torch.Tensor]


_ITOS_TABLES = {}


def _itos_table(itos, device):
    """itos as the device table of mmt_distinct_smiles, uploaded once per content and device: (entries (n,2) i32
    {byte start, byte length or -1}, UTF-8 bytes u8, longest entry in bytes).  Only the keys str(i), i >= 0, can match an
    id (the host path looks ids up as itos[str(int(v))])."""
    key = (str(device), tuple(sorted((str(k), str(v)) for k, v in itos.items())))
    hit = _ITOS_TABLES.get(key)
    if hit is not None:
        return hit
    ids = {int(k): v for k, v in itos.items() if isinstance(k, str) and k.isdigit() and str(int(k)) == k}
    n = max(ids) + 1 if ids else 0
    ent = torch.full((max(n, 1), 2), -1, dtype=torch.int32)
    blob = bytearray()
    for i, v in sorted(ids.items()):
        b = v.encode("utf-8")
        ent[i, 0], ent[i, 1] = len(blob), len(b)
        blob += b
    data = torch.tensor(list(blob) or [0], dtype=torch.uint8)
    longest = max((len(v.encode("utf-8")) for v in ids.values()), default=0)
    hit = (ent.to(device), data.to(device), n, longest)
    _ITOS_TABLES[key] = hit
    return hit


def distinct_smiles(tokens, itos, n_candidates, token_prob=None):
    """Distinct SMILES of every memory column of generated ids, computed on the device (``mmt_distinct_smiles``).

    tokens (T, N) i64 on a CUDA device, N = Bm * n_candidates; column b owns tokens[:, b*n_candidates:(b+1)*n_candidates].
    Returns Bm lists of :class:`DistinctSmiles`; list b holds ``dict.fromkeys(tensor_to_smiles(column b, itos))`` in that
    order.  Strings are compared as bytes, so ids that spell the same string count once.  ``token_prob`` (T', N), the
    ``tensor_to_smiles_and_prob_2`` layout, adds each string's probability slice.  An id before <EOS> that itos lacks
    raises KeyError, as tensor_to_smiles does."""
    if tokens.dim() != 2 or not tokens.is_cuda:
        raise ValueError("tokens must be a (T, N) tensor on a CUDA device")
    k = int(n_candidates)
    T, N = tokens.shape
    if k < 1 or N % k or N == 0 or T == 0:
        raise ValueError(f"N = {N} is not a positive multiple of n_candidates = {k} (or T = {T} is 0)")
    t = tokens.to(torch.int64).contiguous()
    dev = t.device
    ent, data, n_tab, longest = _itos_table(itos, dev)
    L = _lib.lib()
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    need = C.c_int64(0)
    res = (C.c_int64 * 6)()
    args = (t.data_ptr(), T, N, k, _eos_id(itos), data.data_ptr(), ent.data_ptr(), n_tab, longest)
    _lib.check(L.mmt_distinct_smiles(*args, None, C.byref(need), res, stream))
    work = torch.empty(int(need.value), dtype=torch.uint8, device=dev)
    _lib.check(L.mmt_distinct_smiles(*args, work.data_ptr(), C.byref(need), res, stream))
    if res[4]:
        raise KeyError(str(int(res[5])))
    n_dist, off, size = int(res[0]), int(res[2]), int(res[3])
    out = work[off:off + size].cpu().numpy()               # the one copy of metadata and bytes
    Bm = N // k
    meta = out[:8 * (Bm + 1 + 4 * n_dist + 1)].view("<i8")
    col_off = meta[:Bm + 1].tolist()
    first, count, ntok, boff = (meta[Bm + 1 + j * n_dist:Bm + 1 + (j + 1) * n_dist + (j == 3)].tolist() for j in range(4))
    blob = out[8 * len(meta):].tobytes()
    res_cols = []
    for b in range(Bm):
        col = []
        for d in range(col_off[b], col_off[b + 1]):
            prob = token_prob[:ntok[d], b * k + first[d]] if token_prob is not None else None
            col.append(DistinctSmiles(blob[boff[d]:boff[d + 1]].decode("utf-8"), first[d], count[d], prob))
        res_cols.append(col)
    return res_cols
