"""Utterance sharding across the GPUs of one box + the single N-best all-gather.

The reference parallelises decode only by fanning single utterances out to
joblib worker processes (``bin/test_asr.py:108-109,138-139``).  The recursion
does not shard inside an utterance (sequential in T, beam coupled every step),
so here whole utterances are dealt to ranks (one process per GPU), every rank
decodes its shard with the batched device beam search, and ONE all-gather of a
packed int32 N-best buffer (NCCL over NVLink/NVSwitch; gloo in the CPU tests)
gives every rank the full result in the original utterance order.  Nothing else
crosses GPUs.  The buffer is RAGGED (every rank derives the same layout from the
length list: no ids travel, nothing is padded to the set's longest utterance; ~4.5x
smaller than rectangular rows for a dev-clean-like set) and is packed ON THE DEVICE
from the finalize kernel's outputs (RaggedPacker -> e2e_nbest_pack_ragged), gathered
where it lies and read back once into pinned host memory.  pack_nbest_ragged (the same
layout packed on the CPU) remains for the gloo tests and as the cross-check of the kernel.
"""
import numpy as np
import torch
import torch.distributed as dist


def utterance_cost(n_frames, max_len_ratio=0.2):
    """Relative decode cost of an utterance: steps x encoder frames ~ L^2 (SURVEY.md §8e)."""
    n = np.asarray(n_frames, dtype=np.float64)
    return np.ceil(n * max_len_ratio) * (n / 4.0) + 50.0 * n


def plan_shards(lengths, world_size, max_len_ratio=0.2):
    """Longest-processing-time greedy: returns ``world_size`` index arrays (each sorted by
    descending length) whose summed costs are balanced.  Deterministic, so every rank
    computes the same plan from the same length list."""
    lengths = np.asarray(lengths)
    cost = utterance_cost(lengths, max_len_ratio)
    order = np.lexsort((np.arange(len(lengths)), -cost))          # cost desc, index asc
    load = np.zeros(world_size)
    shards = [[] for _ in range(world_size)]
    for i in order:
        r = int(np.argmin(load))                                    # ties -> lowest rank
        shards[r].append(int(i))
        load[r] += cost[i]
    return [np.array(s, dtype=np.int64) for s in shards]


def estimate_decode_bytes(n_utts, l_max, vocab, beam, n_cand, feat_dim=160, enc_dim=640, att_dim=300,
                          lm_dim=1024, lm_layers=4, encoder_chunk=128, num_head=1, v_proj=False, time_reduction=4,
                          front_reduction=4):
    """Upper estimate of the HBM ``BeamDecoder.decode_batch`` needs at its peak for ``n_utts`` utterances padded
    to ``l_max`` input frames (DESIGN.md §3: every buffer is sized by the LONGEST utterance of the batch).
    Dominant terms: the frame-major posteriors together with the CTC logits they are made from
    (2 x U x Tmax x Vp fp32 — 170 GB for 2620 utterances with a 10k subword vocabulary), the two prefix-state
    buffers, the encoder output and the attention keys; the encoder's chunk temporaries are a constant.  With
    ``num_head`` heads the keys and alignments are H times as large, and with ``v_proj`` the projected values
    [U][T][H*enc_dim] are held as well (~22 GB for 2620 utterances of ~828 frames at H = 4), counted twice because the
    plain multi-head step holds a head-major copy beside them while it makes it.  ``time_reduction`` is the encoder's
    input-to-output frame ratio (``Encoder.sample_rate``: 4 for the VGG front end alone, 2 for config/librispeech_asr.yaml's
    encoder without it), ``front_reduction`` the part of it before the first recurrent layer (4 with the VGG front end, 1
    without).  Where a recurrent layer sub-samples (the two differ) the terms at the output frame rate under-count the
    encoder: its first recurrent layer runs over all U * l_max / front_reduction frames of the batch at once
    (Encoder.forward_ragged_packed) and holds the packed input, the gates [F, 4*enc_dim], the recurrence output and the
    sub-sampled output together; that term is added."""
    u, t = int(n_utts), (int(l_max) // int(time_reduction) + 3) // 4 * 4
    vp = (int(vocab) + 3) // 4 * 4
    n = u * beam
    feats = u * int(l_max) * feat_dim * 4
    enc = u * t * enc_dim * 4 * 2                                   # padded output + the packed frames it is scattered from
    h = int(num_head)
    keys = u * t * att_dim * h * 4 * 2                              # proj_k output and its channel-major copy
    # tanh(proj_v(enc)) (no projection: the encoder output), twice: the plain multi-head step re-lays it out head-major
    values = u * t * enc_dim * h * 4 * 2 if v_proj else 0
    post = 2 * u * t * vp * 4 + u * t * 8                           # logits + posteriors (+ blank running sum)
    states = 2 * u * t * beam * max(1, n_cand) * 8
    attn = 3 * n * h * t * 4
    lstm = n * (lm_layers * (3 * 2 * lm_dim * 2 + 4 * lm_dim * 4) + 4 * lm_dim * 4) + 3 * n * vp * 4
    hist = 3 * (int(l_max) // 5 + 2) * n * 4
    chunk = min(u, encoder_chunk) * int(l_max) * 40 * 128 * 4 * 3 + (3 << 30) * 2      # VGG activations + unfolded operand + GEMM result
    first = 0
    if int(time_reduction) != int(front_reduction):
        f1 = u * (int(l_max) // int(front_reduction))
        in_w = feat_dim if int(front_reduction) == 1 else 4 * enc_dim    # the VGG output: 256 channels x F/4 bins (2560 at full size)
        first = f1 * (in_w + 4 * enc_dim + 2 * enc_dim) * 4
    return int(1.1 * (feats + enc + keys + values + post + states + attn + lstm + hist + chunk + first))


def make_batches(indices, lengths, max_utts=512, max_padded_frames=None, max_bytes=None, bytes_fn=None):
    """Split ``indices`` (any order) into length-sorted batches: utterances of similar length
    share a batch so that padding and idle decode steps stay small.  ``max_bytes`` with
    ``bytes_fn(n_utts, l_max) -> bytes`` (e.g. a partial of :func:`estimate_decode_bytes`) also closes a batch
    before its estimated footprint exceeds the budget; a single utterance is never refused."""
    lengths = np.asarray(lengths)
    idx = sorted((int(i) for i in indices), key=lambda i: (-int(lengths[i]), i))
    batches, cur = [], []
    for i in idx:
        longest = int(lengths[cur[0]]) if cur else int(lengths[i])
        if cur and (len(cur) >= max_utts or (max_padded_frames and (len(cur) + 1) * longest > max_padded_frames)
                    or (max_bytes and bytes_fn is not None and bytes_fn(len(cur) + 1, longest) > max_bytes)):
            batches.append(cur)
            cur = []
        cur.append(i)
    if cur:
        batches.append(cur)
    return batches


def row_width(beam, cap):
    """int32 words per utterance of a RECTANGULAR buffer padded to the set's longest utterance (round 1's format; kept as
    the yardstick the ragged layout is compared with)."""
    return 2 + 2 * beam + 2 * beam * cap


# ---- ragged N-best buffer ------------------------------------------------------------------------
# Every rank knows every utterance's length, hence how many tokens each hypothesis can have (S_u = ceil(L_u * ratio),
# + 1 for a closing <eos>) and where every utterance of every shard sits in its rank's buffer: no ids travel, nothing
# is padded to the longest utterance of the set, and all ranks agree on the (equal) buffer size without talking.
# buffer (int32) = [ per utterance: n, len_0..len_{B-1}, avgbits_0..avgbits_{B-1} ]      headers, U x (1 + 2B)
#                  [ per utterance, per hypothesis: cap_u tokens ]                        sum_u B * cap_u
#                  [ the same for the per-token score bits ]                              sum_u B * cap_u
# Packing and unpacking are a handful of vectorised gathers (no per-utterance Python loop).
def ragged_layout(shard_ids, lengths, beam, max_len_ratio):
    """(cap [n], total) of one rank's buffer for the utterances ``shard_ids`` (in this order)."""
    caps = np.ceil(np.asarray(lengths)[np.asarray(shard_ids, dtype=np.int64)] * max_len_ratio).astype(np.int64) + 1
    return caps, int(len(caps) * (1 + 2 * beam) + 2 * beam * caps.sum())


def _segment_index(starts, seg_len):
    """Concatenation of arange(starts[i], starts[i] + seg_len[i]) for all i, as one int64 array."""
    total = int(seg_len.sum())
    if total == 0:
        return np.zeros(0, dtype=np.int64)
    first = np.cumsum(seg_len) - seg_len
    return np.repeat(starts - first, seg_len) + np.arange(total, dtype=np.int64)


def pack_nbest_ragged(utt_ids, tok, sc, ln, avg, n, shard_ids, lengths, beam, max_len_ratio, size):
    """CPU int32 [size]: the N-best of the decoded utterances ``utt_ids`` (any order; rows of tok/sc/ln/avg/n) at their
    slots of the shard's layout; utterances of the shard that were not decoded keep n = -1."""
    caps, total = ragged_layout(shard_ids, lengths, beam, max_len_ratio)
    if total > size:
        raise ValueError("ragged N-best buffer too small")
    n_shard, hdr_w = len(caps), 1 + 2 * beam
    buf = torch.zeros(size, dtype=torch.int32)
    hdr = buf[:n_shard * hdr_w].view(n_shard, hdr_w)
    hdr[:, 0] = -1
    if len(utt_ids) == 0:
        return buf
    slot_of = {int(u): k for k, u in enumerate(shard_ids)}
    slots = np.array([slot_of[int(u)] for u in utt_ids], dtype=np.int64)          # decoded row -> slot in the layout
    if int((ln.long() > torch.as_tensor(caps[slots])[:, None]).sum()) > 0:
        raise ValueError("a hypothesis is longer than ceil(L * max_len_ratio) + 1 tokens")
    have = tok.shape[2]
    if have < int(caps[slots].max()):
        tok = torch.nn.functional.pad(tok, (0, int(caps[slots].max()) - have))
        sc = torch.nn.functional.pad(sc, (0, int(caps[slots].max()) - have))
        have = tok.shape[2]
    st = torch.as_tensor(slots)
    hdr[st, 0] = n.to(torch.int32)
    hdr[st, 1:1 + beam] = ln.to(torch.int32)
    hdr[st, 1 + beam:] = avg.to(torch.float32).contiguous().view(torch.int32)
    # token / score sections: segment (slot k, hypothesis b) holds cap_k values
    seg_len_all = np.repeat(caps, beam)                                           # layout order
    seg_first_all = np.cumsum(seg_len_all) - seg_len_all
    rows = np.repeat(np.arange(len(slots), dtype=np.int64), beam)                 # decoded (row, b) pairs
    hyp = np.tile(np.arange(beam, dtype=np.int64), len(slots))
    seg = np.repeat(slots, beam) * beam + hyp                                     # their segment in the layout
    seg_len = seg_len_all[seg]
    src = torch.as_tensor(_segment_index((rows * beam + hyp) * have, seg_len))
    dst = torch.as_tensor(_segment_index(seg_first_all[seg], seg_len))
    t0 = n_shard * hdr_w
    t1 = t0 + int(seg_len_all.sum())
    buf[t0:t1][dst] = tok.to(torch.int32).contiguous().view(-1)[src]
    buf[t1:t1 + int(seg_len_all.sum())][dst] = sc.to(torch.float32).contiguous().view(torch.int32).view(-1)[src]
    return buf


def unpack_nbest_ragged(buf, shards, lengths, beam, max_len_ratio, size):
    """Inverse over the concatenation of all ranks' buffers ([world * size] int32): dense arrays indexed by utterance."""
    buf = buf.cpu()
    n_total = len(lengths)
    cap_max = int(np.ceil(np.asarray(lengths).max() * max_len_ratio)) + 1 if n_total else 1
    tok = torch.zeros((n_total, beam, cap_max), dtype=torch.int32)
    sc_bits = torch.zeros((n_total, beam, cap_max), dtype=torch.int32)
    ln = torch.zeros((n_total, beam), dtype=torch.int32)
    avg = torch.zeros((n_total, beam), dtype=torch.float32)
    n = torch.full((n_total,), -1, dtype=torch.int32)
    hdr_w = 1 + 2 * beam
    for r, ids in enumerate(shards):
        if len(ids) == 0:
            continue
        caps, total = ragged_layout(ids, lengths, beam, max_len_ratio)
        part = buf[r * size:r * size + total]
        ut = torch.as_tensor(np.asarray(ids, dtype=np.int64))
        hdr = part[:len(ids) * hdr_w].view(len(ids), hdr_w)
        n[ut] = hdr[:, 0]
        ln[ut] = hdr[:, 1:1 + beam]
        avg[ut] = hdr[:, 1 + beam:].contiguous().view(torch.float32)
        seg_len = np.repeat(caps, beam)
        hyp = np.tile(np.arange(beam, dtype=np.int64), len(ids))
        dst = torch.as_tensor(_segment_index((np.repeat(np.asarray(ids, dtype=np.int64), beam) * beam + hyp) * cap_max, seg_len))
        t0 = len(ids) * hdr_w
        t1 = t0 + int(seg_len.sum())
        tok.view(-1)[dst] = part[t0:t1]
        sc_bits.view(-1)[dst] = part[t1:t1 + int(seg_len.sum())]
    assert int((n < 0).sum()) == 0, "N-best gather lost utterances"
    return tok, sc_bits.view(torch.float32), ln, avg, n


class RaggedPacker:
    """Device-side packing of one rank's ragged buffer: the layout tables (slot, token offset, capacity per utterance)
    live on the device, and the N-best of every decoded batch goes from ``beam_finalize``'s outputs straight into the
    buffer with one small kernel (``e2e_nbest_pack_ragged``) — no host copy, no CPU temporaries."""

    def __init__(self, shard_ids, lengths, beam, max_len_ratio, size, device):
        caps, total = ragged_layout(shard_ids, lengths, beam, max_len_ratio)
        if total > size:
            raise ValueError("ragged N-best buffer too small")
        self.beam, self.size, self.device = beam, int(size), device
        self.n_shard = len(caps)
        self.hdr_len = self.n_shard * (1 + 2 * beam)
        self.tok_len = int(beam * caps.sum())
        off = beam * (np.cumsum(caps) - caps)                                  # first token element of every layout slot
        self._slot_of = {int(u): k for k, u in enumerate(shard_ids)}
        self._caps, self._off = caps, off
        self.buf = torch.zeros(self.size, dtype=torch.int32, device=device)
        self._tables = {}

    def reset(self):
        """Headers back to 'not decoded' (n = -1); the token / score sections are overwritten by the packs."""
        self.buf[:self.hdr_len].view(self.n_shard, -1)[:, 0] = -1

    def pack(self, utt_ids, tok, sc, ln, avg, n):
        """N-best of the decoded utterances ``utt_ids`` (device tensors, rows in this order) -> their slots."""
        from . import ops
        key = tuple(int(u) for u in utt_ids)
        tab = self._tables.get(key)
        if tab is None:
            slots = np.array([self._slot_of[u] for u in key], dtype=np.int64)
            tab = (torch.as_tensor(slots.astype(np.int32), device=self.device),
                   torch.as_tensor(self._off[slots].astype(np.int64), device=self.device),
                   torch.as_tensor(self._caps[slots].astype(np.int32), device=self.device))
            self._tables[key] = tab
        hdr = self.buf[:self.hdr_len]
        t0 = self.hdr_len
        ops.nbest_pack_ragged(tok.contiguous(), sc.contiguous(), ln.contiguous(), avg.contiguous(), n.contiguous(), tab[0], tab[1], tab[2],
                              hdr, self.buf[t0:t0 + self.tok_len], self.buf[t0 + self.tok_len:t0 + 2 * self.tok_len])
        return self.buf


def ragged_size(shards, lengths, beam, max_len_ratio):
    """The common buffer size: the largest shard's (every rank computes the same number from the same plan)."""
    return max([ragged_layout(ids, lengths, beam, max_len_ratio)[1] for ids in shards] + [1])


_PINNED = {}


def _pinned(shape, dtype):
    """One persistent pinned read-back buffer per (shape, dtype): allocating page-locked memory costs milliseconds, so the
    buffer is kept; a gather overwrites what the previous one returned."""
    key = (tuple(shape), dtype)
    buf = _PINNED.get(key)
    if buf is None:
        buf = torch.empty(shape, dtype=dtype, pin_memory=True)
        _PINNED.clear()
        _PINNED[key] = buf
    return buf


def gather_nbest(local_buf, device=None, marks=None):
    """The one collective of the sharded decode: all-gather of the packed buffers (same shape on every rank).
    Returns the concatenation of all ranks' buffers on the host.  A CUDA ``local_buf`` (RaggedPacker) is gathered where
    it lies and read back ONCE into a persistent pinned host buffer (overwritten by the next gather); a CPU buffer (gloo tests, legacy CPU packing) is sent as it is."""
    multi = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    if local_buf.is_cuda:
        recv = local_buf
        if multi:
            recv = torch.empty((dist.get_world_size() * local_buf.shape[0],) + tuple(local_buf.shape[1:]),
                               dtype=local_buf.dtype, device=local_buf.device)
            dist.all_gather_into_tensor(recv, local_buf.contiguous())
        if marks is not None:
            marks[0].record()                                                  # (CUDA events: after the gather, after the read-back)
        host = _pinned(recv.shape, recv.dtype)
        host.copy_(recv, non_blocking=True)
        if marks is not None:
            marks[1].record()
        torch.cuda.current_stream(local_buf.device).synchronize()
        return host
    if not multi:
        return local_buf
    world = dist.get_world_size()
    send = local_buf.to(device) if device is not None else local_buf
    recv = torch.empty((world * send.shape[0],) + tuple(send.shape[1:]), dtype=send.dtype, device=send.device)
    dist.all_gather_into_tensor(recv, send.contiguous())
    return recv.cpu()


def decode_sharded(decode_fn, lengths, beam, max_len_ratio, rank=0, world_size=1, device=None,
                   max_utts=512, max_padded_frames=None):
    """Decode utterances 0..len(lengths)-1 across ``world_size`` ranks.

    ``decode_fn(batch_ids) -> (tok, sc, ln, avg, n)`` for the utterances in ``batch_ids``: what
    ``BeamDecoder.decode_batch(..., return_arrays="device")`` returns (CUDA tensors: packed on the device, gathered over
    NCCL, one read-back) or ``return_arrays=True`` (CPU tensors: packed on the host — the gloo tests).
    Every rank returns the full (tok, sc, ln, avg, n) arrays in utterance order."""
    lengths = np.asarray(lengths)
    shards = plan_shards(lengths, world_size, max_len_ratio)
    size = ragged_size(shards, lengths, beam, max_len_ratio)
    mine = shards[rank]
    parts, ids, packer = [], [], None
    for batch in make_batches(mine, lengths, max_utts, max_padded_frames):
        part = decode_fn(batch)
        if part[0].is_cuda:
            if packer is None:
                packer = RaggedPacker(mine, lengths, beam, max_len_ratio, size, part[0].device)
                packer.reset()
            packer.pack(batch, *part)
        else:
            parts.append(part)
        ids.extend(batch)
    if packer is not None:
        local = packer.buf
    else:
        if parts:
            width = max(p[0].shape[2] for p in parts)
            pad = lambda a: torch.nn.functional.pad(a, (0, width - a.shape[2]))
            tok = torch.cat([pad(p[0]) for p in parts]); sc = torch.cat([pad(p[1]) for p in parts])
            ln = torch.cat([p[2] for p in parts]); avg = torch.cat([p[3] for p in parts]); n = torch.cat([p[4] for p in parts])
        else:
            tok = torch.zeros((0, beam, 1), dtype=torch.int32); sc = torch.zeros((0, beam, 1))
            ln = torch.zeros((0, beam), dtype=torch.int32); avg = torch.zeros((0, beam)); n = torch.zeros((0,), dtype=torch.int32)
        local = pack_nbest_ragged(ids, tok, sc, ln, avg, n, mine, lengths, beam, max_len_ratio, size)
        if device is not None and len(mine) == 0:
            local = local.to(device)
    return unpack_nbest_ragged(gather_nbest(local, device), shards, lengths, beam, max_len_ratio, size)
