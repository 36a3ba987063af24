"""Data-parallel batch scheduler: shard spectra across ranks, decode locally,
all-gather only the generated token ids.

Every spectrum (and every candidate of a spectrum) is independent on this path
(SURVEY.md 8e), so ranks own contiguous blocks of spectra, keep a full replica of
the 25.6 M-parameter model, and exchange nothing until the end: one NCCL
all-gather of the ids as bytes (vocab 43 < 256), optionally the chosen-token
probabilities.  The reference has no multi-GPU inference; the oracle for the
sharded run is the single-GPU run (shard-invariant Philox indexing, see
generate.multinomial_sequence_multi's seq_index_base / n_total).

The ids travel SEQUENCE-MAJOR, (N_local, T) bytes per rank: rank blocks are then
contiguous in the gathered (N_total, T) buffer, i.e. the collective writes the
final order and no permute / contiguous copy follows it.  The collective is issued
on a side stream behind an event recorded after the rank's last sampler kernel, so
a caller that keeps generating (``async_gather=True``) overlaps it -- and the
per-call rendezvous with the slowest rank -- with its next batch's encode.
"""
from __future__ import annotations

import torch
import torch.distributed as dist


def shard_bounds(n_items: int, world: int, rank: int):
    """Contiguous block [lo, hi) of ``n_items`` for ``rank``: ceil-sized blocks, the tail ranks may be short or empty."""
    per = (n_items + world - 1) // world
    lo = min(rank * per, n_items)
    hi = min(lo + per, n_items)
    return lo, hi


def shard_dict(data_dict, world: int, rank: int):
    n = next(iter(data_dict.values())).shape[0]
    lo, hi = shard_bounds(n, world, rank)
    return {k: v[lo:hi] for k, v in data_dict.items()}, lo, hi


def gather_rows(local: torch.Tensor, rows_per_rank: int, group=None) -> torch.Tensor:
    """All-gather row blocks: every rank holds ``local`` (<= rows_per_rank, ...) and receives
    (world * rows_per_rank, ...), rank r's rows at [r * rows_per_rank, ...).  Short tail shards are zero-padded for
    the collective; with ceil-sized contiguous shards the first n_total rows of the result are the unsharded order.
    Works for any dtype / backend (NCCL on GPUs, gloo in the CPU tests)."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    send = local
    if local.shape[0] != rows_per_rank:
        send = torch.zeros((rows_per_rank,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
        send[:local.shape[0]] = local
    send = send.contiguous()
    if world == 1:
        return send
    recv = torch.empty((world * rows_per_rank,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(recv, send, group=group)
    return recv


def gather_columns(local: torch.Tensor, n_cols_total: int, cols_per_rank: int, group=None) -> torch.Tensor:
    """All-gather column blocks of a time-major tensor: every rank holds ``local`` (T, <=cols_per_rank) and
    receives (T, n_cols_total).  The collective concatenates along dim 0, so this form pays a transpose on both
    sides; the scheduler itself gathers ids sequence-major (``gather_rows``) and keeps this for small float
    tensors (probabilities) and as a utility."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return local
    out = gather_rows(local.transpose(0, 1), cols_per_rank, group)          # (world * per, T)
    return out[:n_cols_total].transpose(0, 1).contiguous()


_SIDE = {}


def _side_stream(device):
    key = (device.type, device.index)
    if key not in _SIDE:
        _SIDE[key] = torch.cuda.Stream(device=device)
    return _SIDE[key]


class PendingTokens:
    """Result of a sharded generation whose id all-gather is (possibly still) in flight on the side stream."""

    def __init__(self, eng, packed, event, n_total, T, probs=None, local=(0, 0)):
        self._eng, self._packed, self._event, self.n_total, self.T, self._probs, self.local = eng, packed, event, n_total, T, probs, local

    def _sync(self):
        if self._event is not None:
            cur = torch.cuda.current_stream(self._packed.device)
            cur.wait_event(self._event)
            for t in (self._packed, self._probs):        # allocated on the side stream, read on the caller's from here on
                if t is not None:
                    t.record_stream(cur)
            self._event = None

    def packed(self) -> torch.Tensor:
        """(n_total, T) u8 ids, sequence-major (the gathered buffer itself, no copy)."""
        self._sync()
        return self._packed[:self.n_total]

    def tokens(self) -> torch.Tensor:
        """(T, n_total) i64 ids, the reference's layout."""
        self._sync()
        if self._packed.is_cuda:
            return self._eng.unpack_tokens_seqmajor(self._packed, self.n_total)
        return self._packed[:self.n_total].transpose(0, 1).to(torch.int64).contiguous()

    def probs(self):
        self._sync()
        return self._probs


def generate_sharded(model, data_dict, config, stoi, *, n_candidates=1, sampling="multinomial", gather_probs=False,
                     group=None, async_gather=False, per_memory_rng=False, stop_at_eos=False):
    """Encode + decode this rank's spectra and all-gather the ids.

    Returns (tokens (T, B*n_candidates) i64 -- identical on every rank and identical to the single-GPU run --, probs or
    None, local (lo, hi)); with ``async_gather=True`` a :class:`PendingTokens` instead, whose collective overlaps
    whatever the caller launches next (greedy early-exit trimming is then the caller's business).  ``per_memory_rng``:
    every spectrum's candidates draw in their own stream (generate.multinomial_sequence_multi), so the result also
    equals the reference's per-spectrum loop.  ``stop_at_eos``: sequences stop being computed at stoi["<EOS>"]
    (generate.multinomial_sequence_multi); retirement is per sequence, so the result is still shard invariant."""
    from . import generate as G
    from .engine import engine_for
    if per_memory_rng and sampling == "greedy":
        raise ValueError("per_memory_rng needs multinomial sampling")
    eos = G._eos_id(stoi) if stop_at_eos else None
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    B = next(iter(data_dict.values())).shape[0]
    local, lo, hi = shard_dict(data_dict, world, rank)
    per = (B + world - 1) // world
    T = int(config.max_len)
    eng = engine_for(model, config)
    if hi > lo:
        # host buffers: move this rank's shard with asynchronous copies (pinned memory makes them truly asynchronous), so the
        # host keeps launching instead of draining the stream at every tensor the way a blocking .to(device) does
        local = {k: (v if v.is_cuda else v.to(eng.device, non_blocking=True)) for k, v in local.items()}
        memory, mask, *_ = G.run_model(model, local, config)
        if sampling == "greedy":
            # stop_on_all_pad is a whole-batch property: decide it after the gather
            tok, pr, _ = G._decode(model, memory, mask, config, "greedy", False, n_candidates, 0, 0, eos=eos)
        else:
            tok, pr, _ = G._decode(model, memory, mask, config, "multinomial", False, n_candidates,
                                   lo * n_candidates, B * n_candidates, per_memory_rng, eos=eos)
        packed = eng.pack_tokens_seqmajor(tok)                                   # (n_local, T) u8
    else:
        packed = torch.zeros(0, T, dtype=torch.uint8, device=eng.device)
        pr = torch.zeros(T, 0, dtype=torch.float32, device=eng.device)
        if sampling != "greedy":
            # an empty shard draws nothing, but the unsharded run's T multinomial calls would have advanced this device's
            # generator: keep every rank's Philox offset in step so later sharded calls still reproduce the 1-GPU draws
            gen = torch.cuda.default_generators[eng.dev_index]
            gen.set_offset(int(gen.get_offset()) + G._philox_advance(eng, n_candidates, B * n_candidates, T, per_memory_rng))
    n_total = B * n_candidates
    cur = torch.cuda.current_stream(eng.device)
    if world > 1:
        side = _side_stream(eng.device)
        ready = torch.cuda.Event()
        ready.record(cur)
        with torch.cuda.stream(side):
            side.wait_event(ready)
            all_u8 = gather_rows(packed, per * n_candidates, group)              # (world * per * k, T): final order
            probs = gather_columns(pr, n_total, per * n_candidates, group) if gather_probs else None
            done = torch.cuda.Event()
            done.record(side)
        for t in (packed, pr, all_u8) + ((probs,) if probs is not None else ()):
            t.record_stream(side)
    else:
        all_u8, probs, done = packed, (pr if gather_probs else None), None
    pending = PendingTokens(eng, all_u8, done, n_total, T, probs, (lo, hi))
    if async_gather:
        return pending
    tokens, probs = pending.tokens(), pending.probs()
    if sampling == "greedy":
        allpad = (tokens == 0).all(dim=1)
        if bool(allpad.any()):
            steps = int(torch.nonzero(allpad)[0]) + 1
            tokens = tokens[:steps]
            probs = probs[:steps] if probs is not None else None
    return tokens, probs, (lo, hi)
