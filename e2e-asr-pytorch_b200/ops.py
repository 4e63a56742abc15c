"""Typed torch-tensor wrappers over the C ABI (include/e2e_asr_b200.h).

PyTorch is only the plumbing here: it owns the device buffers and the stream;
every function below validates its tensors and enqueues ONE hand-written kernel
through ctypes.  Nothing in this module computes on the CPU.
"""
import torch

from . import _lib as L

I32, F32 = torch.int32, torch.float32


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _chk(t, dtype, name, numel=None):
    if t is None:
        return
    if not t.is_cuda:
        raise L.E2EError("%s must be a CUDA tensor (no CPU path)" % name)
    if t.dtype != dtype:
        raise TypeError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    if numel is not None and t.numel() < numel:
        raise ValueError("%s has %d elements, needs %d" % (name, t.numel(), numel))


def padded_vocab(v):
    return L.load().e2e_padded_vocab(int(v))


def ctc_log_softmax(logits, enc_len=None, apply_relu=True, out=None):
    """logits [U,Tmax,V] (CTC Linear output) -> x [Tmax,U,Vp] frame-major log-posteriors."""
    _chk(logits, F32, "logits")
    _chk(enc_len, I32, "enc_len")
    u, t, v = logits.shape
    vp = padded_vocab(v)
    x = out if out is not None else torch.empty((t, u, vp), dtype=F32, device=logits.device)
    _chk(x, F32, "x", t * u * vp)
    L.check(L.load().e2e_ctc_log_softmax(L.ptr(logits), u, t, v, L.ptr(enc_len), int(bool(apply_relu)),
                                        L.ptr(x), vp, _stream()))
    return x


def ctc_init_state(x, enc_len=None, out=None):
    """x [Tmax,U,Vp] -> r0 [U,Tmax,1,2] (state of the empty prefix)."""
    _chk(x, F32, "x")
    _chk(enc_len, I32, "enc_len")
    t, u, vp = x.shape
    r0 = out if out is not None else torch.empty((u, t, 1, 2), dtype=F32, device=x.device)
    _chk(r0, F32, "r0", u * t * 2)
    L.check(L.load().e2e_ctc_init_state(L.ptr(x), t, u, vp, L.ptr(enc_len), L.ptr(r0), _stream()))
    return r0


def ctc_prefix_score(x, vocab, enc_len, r_prev, prev_lane, last_tok, prefix_len, n_live, cand,
                     beam, n_cand, flags=0, psi=None, r_out=None, status=None, n_run=0):
    """One launch of the prefix-score kernel; see e2e_ctc_prefix_score in the header."""
    t, u, vp = x.shape
    _chk(x, F32, "x")
    _chk(enc_len, I32, "enc_len", u)
    _chk(r_prev, F32, "r_prev")
    lanes_prev = r_prev.shape[2]
    if r_prev.shape[0] != u or r_prev.shape[1] != t or r_prev.shape[3] != 2:
        raise ValueError("r_prev must be [U,Tmax,lanes,2]")
    n = u * beam
    _chk(prev_lane, I32, "prev_lane", n)
    _chk(last_tok, I32, "last_tok", n)
    _chk(prefix_len, I32, "prefix_len", n)
    _chk(n_live, I32, "n_live", u)
    _chk(cand, I32, "cand", n * n_cand)
    if psi is None:
        psi = torch.empty((n, n_cand), dtype=F32, device=x.device)
    if r_out is None:
        r_out = torch.empty((u, t, beam * n_cand, 2), dtype=F32, device=x.device)
    _chk(psi, F32, "psi", n * n_cand)
    _chk(r_out, F32, "r_out", u * t * beam * n_cand * 2)
    _chk(status, I32, "status", u)
    L.check(L.load().e2e_ctc_prefix_score(
        L.ptr(x), t, u, vp, int(vocab), L.ptr(enc_len), L.ptr(r_prev), lanes_prev,
        L.ptr(prev_lane), L.ptr(last_tok), L.ptr(prefix_len), L.ptr(n_live), L.ptr(cand),
        int(beam), int(n_cand), int(flags), L.ptr(psi), L.ptr(r_out), L.ptr(status), int(n_run), _stream()))
    return psi, r_out


def prefix_step_supported(vocab, beam, n_cand):
    return bool(L.load().e2e_ctc_prefix_step_supported(padded_vocab(vocab), int(beam), int(n_cand)))


def ctc_prefix_step(x, vocab, enc_len, r_prev, parent_slot, last_tok, parent_tok, prefix_len, n_live, cand,
                    beam, n_cand, flags=0, psi=None, r_out=None, status=None, n_run=0):
    """One fused launch of the per-step kernel (lazy state evaluation); see e2e_ctc_prefix_step in the header.
    r_prev [U,Tmax,lanes_prev,2] -> (psi [U*B,C], r_out [U,Tmax,B,2])."""
    t, u, vp = x.shape
    _chk(x, F32, "x")
    _chk(enc_len, I32, "enc_len", u)
    _chk(r_prev, F32, "r_prev")
    if r_prev.dim() != 4 or r_prev.shape[0] != u or r_prev.shape[1] != t or r_prev.shape[3] != 2:
        raise ValueError("r_prev must be [U,Tmax,lanes,2]")
    lanes_prev = r_prev.shape[2]
    n = u * beam
    _chk(parent_slot, I32, "parent_slot", n)
    _chk(last_tok, I32, "last_tok", n)
    _chk(parent_tok, I32, "parent_tok", n)
    _chk(prefix_len, I32, "prefix_len", n)
    _chk(n_live, I32, "n_live", u)
    _chk(cand, I32, "cand", n * n_cand)
    if psi is None:
        psi = torch.empty((n, n_cand), dtype=F32, device=x.device)
    if r_out is None:
        r_out = torch.empty((u, t, beam, 2), dtype=F32, device=x.device)
    _chk(psi, F32, "psi", n * n_cand)
    _chk(r_out, F32, "r_out", u * t * beam * 2)
    _chk(status, I32, "status", u)
    L.check(L.load().e2e_ctc_prefix_step(
        L.ptr(x), t, u, vp, int(vocab), L.ptr(enc_len), L.ptr(r_prev), lanes_prev,
        L.ptr(parent_slot), L.ptr(last_tok), L.ptr(parent_tok), L.ptr(prefix_len), L.ptr(n_live), L.ptr(cand),
        int(beam), int(n_cand), int(flags), L.ptr(psi), L.ptr(r_out), L.ptr(status), int(n_run), _stream()))
    return psi, r_out


def beam_candidates(att_logits, n_utts, beam, vocab, n_cand, n_live, att_stats, cand):
    _chk(att_logits, F32, "att_logits")
    ld = att_logits.stride(0) if att_logits.dim() == 2 else vocab
    _chk(n_live, I32, "n_live", n_utts)
    _chk(att_stats, F32, "att_stats", n_utts * beam * 2)
    _chk(cand, I32, "cand", n_utts * beam * n_cand)
    L.check(L.load().e2e_beam_candidates(L.ptr(att_logits), int(ld), int(n_utts), int(beam), int(vocab), int(n_cand),
                                        L.ptr(n_live), L.ptr(att_stats), L.ptr(cand), _stream()))


def emb_fuse_candidates(dec_logits, emb_logits, n_utts, beam, vocab, n_cand, scale, lam, eps, n_live, logp, att_stats, cand):
    """beam_candidates for a model decoded with embedding fusion (see e2e_emb_fuse_candidates): the first n_utts*beam
    rows of dec_logits / emb_logits [>=n_utts*beam, V] -> logp (the fused log-probs, rows of the same shape), zero
    att_stats and the top-n_cand ids of logp.  scale = relu(temp) and lam (after the sigmoid of a learnable weight)
    hold 1 or V entries."""
    for t, nm in ((dec_logits, "dec_logits"), (emb_logits, "emb_logits"), (logp, "logp")):
        _chk(t, F32, nm)
        if t.dim() != 2 or t.shape[0] < n_utts * beam or t.shape[1] < vocab:
            raise ValueError("%s must be [>=%d, >=%d]" % (nm, n_utts * beam, vocab))
    _chk(scale, F32, "scale")
    _chk(lam, F32, "lam")
    _chk(n_live, I32, "n_live", n_utts)
    _chk(att_stats, F32, "att_stats", n_utts * beam * 2)
    _chk(cand, I32, "cand", n_utts * beam * n_cand)
    L.check(L.load().e2e_emb_fuse_candidates(L.ptr(dec_logits), int(dec_logits.stride(0)), L.ptr(emb_logits), int(emb_logits.stride(0)),
                                            int(n_utts), int(beam), int(vocab), int(n_cand), L.ptr(scale), int(scale.numel()),
                                            L.ptr(lam), int(lam.numel()), float(eps), L.ptr(n_live), L.ptr(logp), int(logp.stride(0)),
                                            L.ptr(att_stats), L.ptr(cand), _stream()))
    return logp


class BeamBuffers:
    """Device-resident beam-search bookkeeping for a batch of U utterances
    (the arrays e2e_beam_combine_prune updates in place)."""

    def __init__(self, n_utts, beam, n_cand, max_steps, min_len, max_len, device, fin_cap=None):
        u, b = n_utts, beam
        self.U, self.B, self.C, self.S = u, b, n_cand, max(1, int(max_steps))
        z = lambda *s, dt=I32: torch.zeros(s, dtype=dt, device=device)
        self.min_len = min_len.to(device=device, dtype=I32).contiguous()
        self.max_len = max_len.to(device=device, dtype=I32).contiguous()
        self.n_live = (self.max_len > 0).to(I32)                 # one empty hypothesis per utterance
        self.n_active = self.n_live.clone()
        self.last_tok, self.prefix_len, self.prev_lane = z(u, b), z(u, b), z(u, b)
        self.score_sum, self.ctc_prob = z(u, b, dt=F32), z(u, b, dt=F32)
        self.parent_slot = z(u, b)
        self.parent_row = torch.arange(u * b, dtype=torch.int64, device=device).view(u, b)     # u*B + parent slot
        self.last_tok64 = z(u, b, dt=torch.int64)
        self.parent_tok = torch.full((u, b), -1, dtype=I32, device=device)       # last token of each hypothesis' parent
        self.hist_tok, self.hist_parent = z(self.S, u, b), z(self.S, u, b)
        self.hist_score = z(self.S, u, b, dt=F32)
        self.fin_cap = int(fin_cap if fin_cap is not None else b)      # best-B closed hypotheses suffice
        self.fin_count = z(u)
        self.fin_step, self.fin_parent = z(u, self.fin_cap), z(u, self.fin_cap)
        self.fin_sum, self.fin_score = z(u, self.fin_cap, dt=F32), z(u, self.fin_cap, dt=F32)
        self.status = z(u)
        self.att_stats = z(u * b, 2, dt=F32)
        self.cand = z(u * b, max(1, n_cand))
        self.psi = z(u * b, max(1, n_cand), dt=F32)


# Beam sizes: e2e_beam_combine_prune gives every parent its own warp up to BEAM_NARROW_MAX; e2e_beam_combine_prune_wide
# takes any beam up to BEAM_MAX (the same bits at the narrow sizes).
BEAM_NARROW_MAX = 32
BEAM_MAX = 64


def beam_combine_prune(buf, att_logits, lm_logits, vocab, step, ctc_weight, lm_weight, eos_threshold=1.5, n_run=0):
    """One decode step of score combine + eos threshold + top-k + prune for all utterances (see e2e_beam_combine_prune;
    e2e_beam_combine_prune_wide above BEAM_NARROW_MAX hypotheses)."""
    _chk(att_logits, F32, "att_logits")
    _chk(lm_logits, F32, "lm_logits")
    flags = (L.BEAM_USE_CTC if ctc_weight > 0 else 0) | (L.BEAM_USE_LM if lm_logits is not None else 0)
    lib = L.load()
    fn = lib.e2e_beam_combine_prune if buf.B <= BEAM_NARROW_MAX else lib.e2e_beam_combine_prune_wide
    L.check(fn(
        L.ptr(att_logits), int(att_logits.stride(0)), L.ptr(buf.att_stats),
        L.ptr(lm_logits), int(lm_logits.stride(0)) if lm_logits is not None else 0,
        L.ptr(buf.cand), L.ptr(buf.psi),
        buf.U, buf.B, int(vocab), buf.C, int(step),
        L.ptr(buf.min_len), L.ptr(buf.max_len),
        float(ctc_weight), float(lm_weight), float(eos_threshold), flags,
        L.ptr(buf.n_live), L.ptr(buf.n_active), L.ptr(buf.last_tok), L.ptr(buf.prefix_len),
        L.ptr(buf.score_sum), L.ptr(buf.ctc_prob), L.ptr(buf.prev_lane),
        L.ptr(buf.parent_slot),
        L.ptr(buf.hist_tok), L.ptr(buf.hist_parent), L.ptr(buf.hist_score),
        L.ptr(buf.fin_count), L.ptr(buf.fin_step), L.ptr(buf.fin_parent), L.ptr(buf.fin_sum), L.ptr(buf.fin_score),
        buf.fin_cap, L.ptr(buf.status), int(n_run), L.ptr(buf.parent_row), L.ptr(buf.last_tok64), L.ptr(buf.parent_tok), _stream()))


def beam_finalize(buf, out_cap=None):
    """Final N-best: returns (tokens [U,B,cap] i32, scores [U,B,cap] f32, lens [U,B], avg [U,B], n [U])."""
    dev = buf.n_live.device
    cap = int(out_cap if out_cap is not None else buf.S + 1)
    tok = torch.zeros((buf.U, buf.B, cap), dtype=I32, device=dev)
    sc = torch.zeros((buf.U, buf.B, cap), dtype=F32, device=dev)
    ln = torch.zeros((buf.U, buf.B), dtype=I32, device=dev)
    avg = torch.zeros((buf.U, buf.B), dtype=F32, device=dev)
    n = torch.zeros((buf.U,), dtype=I32, device=dev)
    L.check(L.load().e2e_beam_finalize(
        buf.U, buf.B, L.ptr(buf.max_len), L.ptr(buf.n_live), L.ptr(buf.score_sum),
        L.ptr(buf.hist_tok), L.ptr(buf.hist_parent), L.ptr(buf.hist_score),
        L.ptr(buf.fin_count), L.ptr(buf.fin_step), L.ptr(buf.fin_parent), L.ptr(buf.fin_sum), L.ptr(buf.fin_score),
        buf.fin_cap, L.ptr(tok), L.ptr(sc), L.ptr(ln), L.ptr(avg), L.ptr(n), cap, _stream()))
    return tok, sc, ln, avg, n


def nbest_pack_ragged(tok, sc, ln, avg, n, slot, tok_off, cap, hdr, tok_out, sc_out):
    """Device N-best (beam_finalize's outputs, any row pitch) -> the rank's ragged gather buffer; see
    e2e_nbest_pack_ragged.  slot / cap int32 [U], tok_off int64 [U]; hdr / tok_out / sc_out int32 views of the buffer."""
    u, beam, cap_in = tok.shape
    _chk(tok, I32, "tok"); _chk(sc, F32, "sc"); _chk(ln, I32, "ln", u * beam); _chk(avg, F32, "avg", u * beam); _chk(n, I32, "n", u)
    _chk(slot, I32, "slot", u); _chk(tok_off, torch.int64, "tok_off", u); _chk(cap, I32, "cap", u)
    _chk(hdr, I32, "hdr"); _chk(tok_out, I32, "tok_out"); _chk(sc_out, I32, "sc_out")
    if u == 0:
        return
    L.check(L.load().e2e_nbest_pack_ragged(u, beam, cap_in, L.ptr(tok), L.ptr(sc), L.ptr(ln), L.ptr(avg), L.ptr(n), L.ptr(slot),
                                          L.ptr(tok_off), L.ptr(cap), L.ptr(hdr), L.ptr(tok_out), L.ptr(sc_out), _stream()))


def attention_loc_full(key_t, value, query, prev_att, enc_len, w_conv, w_proj, w_energy, b_energy, temperature, beam,
                       n_run=None, hyps_per_unit=0, attn=None, ctx=None):
    """The whole location-aware attention step (conv + energies + masked softmax + context) for the first
    ``n_run`` utterances: key_t [U,A,T] (channel-major keys), value [U,T,E], query [>=n_run*B,A],
    prev_att [>=n_run*B,T], w_conv [K,W] -> (attn [n_run*B,T], ctx [n_run*B,E])."""
    for t, nm in ((key_t, "key_t"), (value, "value"), (query, "query"), (prev_att, "prev_att"), (w_conv, "w_conv"),
                  (w_proj, "w_proj"), (w_energy, "w_energy")):
        _chk(t, F32, nm)
    _chk(enc_len, I32, "enc_len")
    u, a, t_len = key_t.shape
    e = value.shape[2]
    k, w = w_conv.shape
    n_run = u if n_run is None else int(n_run)
    n = n_run * beam
    if value.shape[0] != u or value.shape[1] != t_len or prev_att.shape[1] != t_len or n_run > u:
        raise ValueError("attention_loc_full: inconsistent shapes")
    _chk(query, F32, "query", n * a)
    _chk(prev_att, F32, "prev_att", n * t_len)
    if attn is None:
        attn = torch.empty((n, t_len), dtype=F32, device=key_t.device)
    if ctx is None:
        ctx = torch.empty((n, e), dtype=F32, device=key_t.device)
    _chk(attn, F32, "attn", n * t_len)
    _chk(ctx, F32, "ctx", n * e)
    L.check(L.load().e2e_attention_loc_full(L.ptr(key_t), L.ptr(value), L.ptr(query), L.ptr(prev_att), L.ptr(enc_len),
                                           L.ptr(w_conv), L.ptr(w_proj), L.ptr(w_energy), float(b_energy), float(temperature),
                                           n_run, int(beam), int(t_len), int(a), int(k), int(w), int(e), int(hyps_per_unit),
                                           L.ptr(attn), L.ptr(ctx), _stream()))
    return attn, ctx


def attention_loc_heads_supported(beam, heads, dim, n_filt, width):
    """Whether e2e_attention_loc_heads launches for this shape (the launcher's own size computation)."""
    return bool(L.load().e2e_attention_loc_heads_supported(int(beam), int(heads), int(dim), int(n_filt), int(width)))


def attention_loc_heads(key_t, value, query, prev_att, enc_len, w_conv, w_proj, w_energy, b_energy, temperature, beam,
                        per_head_values, n_run=None, hyps_per_unit=0, attn=None, ctx=None):
    """The multi-head location-aware attention step for the first ``n_run`` utterances: key_t [U,H,A,T] (channel-major
    keys per head), value [U,T,E] shared by the heads or [U,T,H*E] (``per_head_values``), query [>=n_run*B,H*A],
    prev_att [>=n_run*B,H,T], w_conv [K,H,W] -> (attn [n_run*B,H,T], ctx [n_run*B,H*E], merge_head's input)."""
    for t, nm in ((key_t, "key_t"), (value, "value"), (query, "query"), (prev_att, "prev_att"), (w_conv, "w_conv"),
                  (w_proj, "w_proj"), (w_energy, "w_energy")):
        _chk(t, F32, nm)
    _chk(enc_len, I32, "enc_len")
    u, h, a, t_len = key_t.shape
    k, h_w, w = w_conv.shape
    e = value.shape[2] // h if per_head_values else value.shape[2]
    n_run = u if n_run is None else int(n_run)
    n = n_run * beam
    if (h_w != h or value.shape[0] != u or value.shape[1] != t_len or (per_head_values and value.shape[2] != h * e)
            or prev_att.shape[-1] != t_len or n_run > u):
        raise ValueError("attention_loc_heads: inconsistent shapes")
    _chk(query, F32, "query", n * h * a)
    _chk(prev_att, F32, "prev_att", n * h * t_len)
    if attn is None:
        attn = torch.empty((n, h, t_len), dtype=F32, device=key_t.device)
    if ctx is None:
        ctx = torch.empty((n, h * e), dtype=F32, device=key_t.device)
    _chk(attn, F32, "attn", n * h * t_len)
    _chk(ctx, F32, "ctx", n * h * e)
    L.check(L.load().e2e_attention_loc_heads(L.ptr(key_t), L.ptr(value), L.ptr(query), L.ptr(prev_att), L.ptr(enc_len),
                                            L.ptr(w_conv), L.ptr(w_proj), L.ptr(w_energy), float(b_energy), float(temperature),
                                            n_run, int(beam), int(h), int(t_len), int(a), int(k), int(w), int(e),
                                            int(bool(per_head_values)), int(hyps_per_unit), L.ptr(attn), L.ptr(ctx), _stream()))
    return attn, ctx


def lstm_split_rows(src, row_idx, n, dst, k, off, scale=None):
    """dst[r, p*k + off : p*k + off + w] = p-th piece of src[row_idx[r]] (src [*,w] fp32).  dst bf16 [>=n, 3k]: the exact
    3-piece split; dst fp16 [>=n, 2k] (``scale`` = a power of two): the 2-piece split of scale*src."""
    pieces = _pieces(dst, scale)
    _chk(src, F32, "src")
    _chk(row_idx, torch.int64, "row_idx", n)
    w = src.shape[1]
    if dst.shape[0] < n or dst.shape[1] < pieces * k:
        raise ValueError("lstm_split_rows: dst too small")
    if row_idx is None and src.shape[0] < n:
        raise ValueError("lstm_split_rows: src has fewer than n rows")
    if pieces == 3:
        L.check(L.load().e2e_lstm_split_rows(L.ptr(src), int(src.stride(0)), L.ptr(row_idx), int(n), int(w),
                                            L.ptr(dst), int(dst.stride(0)), int(k), int(off), _stream()))
    else:
        L.check(L.load().e2e_lstm_split_rows_f16x2(L.ptr(src), int(src.stride(0)), L.ptr(row_idx), int(n), int(w),
                                                  L.ptr(dst), int(dst.stride(0)), int(k), int(off), float(scale), _stream()))


def _pieces(dst, scale):
    """Operand format of a split destination: 3 bf16 pieces, or 2 fp16 pieces of the scaled value."""
    if dst is None:
        return 3 if scale is None else 2
    if not dst.is_cuda:
        raise L.E2EError("split operand must be a CUDA tensor (no CPU path)")
    if not dst.is_contiguous():
        raise ValueError("split operand must be contiguous")
    if dst.dtype == torch.bfloat16 and scale is None:
        return 3
    if dst.dtype == torch.float16 and scale is not None:
        return 2
    raise TypeError("split operand must be bf16 (3 pieces, no scale) or fp16 (2 pieces, with a scale), got %s" % dst.dtype)


class SplitPlan:
    """Pre-marshalled argument arrays of e2e_lstm_split_rows_multi for a fixed set of (src, dst, K, off) pairs:
    the per-step call then costs one ctypes dispatch.  ``scale`` selects the 2-piece fp16 format."""

    def __init__(self, pairs, scale=None):
        import ctypes
        n = len(pairs)
        for src, dst, k, off in pairs:
            _chk(src, F32, "src")
            if _pieces(dst, scale) != (3 if scale is None else 2):
                raise TypeError("SplitPlan: mixed operand formats")
        self.scale = scale
        self.keep = pairs
        self.n = n
        self.srcs = (ctypes.c_void_p * n)(*[p[0].data_ptr() for p in pairs])
        self.src_pitch = (ctypes.c_longlong * n)(*[int(p[0].stride(0)) for p in pairs])
        self.widths = (ctypes.c_int * n)(*[int(p[0].shape[1]) for p in pairs])
        self.dsts = (ctypes.c_void_p * n)(*[p[1].data_ptr() for p in pairs])
        self.dst_pitch = (ctypes.c_longlong * n)(*[int(p[1].stride(0)) for p in pairs])
        self.ks = (ctypes.c_int * n)(*[int(p[2]) for p in pairs])
        self.offs = (ctypes.c_int * n)(*[int(p[3]) for p in pairs])
        self.rows = min(min(p[0].shape[0], p[1].shape[0]) for p in pairs)

    def run(self, row_idx, n_rows):
        if n_rows > self.rows or (row_idx is not None and (row_idx.dtype != torch.int64 or not row_idx.is_cuda or row_idx.numel() < n_rows)):
            raise ValueError("SplitPlan.run: bad row index / row count")
        if self.scale is None:
            L.check(L.load().e2e_lstm_split_rows_multi(self.n, self.srcs, self.src_pitch, self.widths, self.dsts, self.dst_pitch,
                                                      self.ks, self.offs, L.ptr(row_idx), int(n_rows), _stream()))
        else:
            L.check(L.load().e2e_lstm_split_rows_multi_f16x2(self.n, self.srcs, self.src_pitch, self.widths, self.dsts, self.dst_pitch,
                                                            self.ks, self.offs, L.ptr(row_idx), int(n_rows), float(self.scale), _stream()))


def lstm_cell(gates, bias, c_prev, row_idx, n, c_new, h_new, table=None, tok=None, a_next=None, k_next=0, off_next=0,
              gate_scale=None, next_scale=None):
    """Fused LSTM cell (see e2e_lstm_cell): gates [>=n,4D] fp32 -> c_new, h_new [>=n,D] (+ split of h into a_next).
    ``gate_scale`` (a power of two) selects the fp16x2 format: gates *= gate_scale first, a_next fp16 [>=n, 2*k_next]
    receives the 2-piece split of next_scale*h."""
    _chk(gates, F32, "gates")
    _chk(bias, F32, "bias")
    _chk(c_prev, F32, "c_prev")
    _chk(row_idx, torch.int64, "row_idx", n)
    _chk(c_new, F32, "c_new")
    _chk(h_new, F32, "h_new")
    _chk(table, F32, "table")
    _chk(tok, torch.int64, "tok", n)
    f16 = gate_scale is not None
    if a_next is not None and _pieces(a_next, next_scale if f16 else None) != (2 if f16 else 3):
        raise TypeError("lstm_cell: a_next does not match the operand format")
    d = c_prev.shape[1]
    if gates.shape[0] < n or gates.shape[1] < 4 * d or c_new.shape[0] < n or h_new.shape[0] < n or bias.numel() < 4 * d:
        raise ValueError("lstm_cell: inconsistent shapes")
    a_pitch = int(a_next.stride(0)) if a_next is not None else 0
    if not f16:
        L.check(L.load().e2e_lstm_cell(L.ptr(gates), int(gates.stride(0)), L.ptr(bias), L.ptr(table), L.ptr(tok), L.ptr(c_prev),
                                      L.ptr(row_idx), int(n), int(d), L.ptr(c_new), L.ptr(h_new), L.ptr(a_next),
                                      a_pitch, int(k_next), int(off_next), _stream()))
    else:
        L.check(L.load().e2e_lstm_cell_f16x2(L.ptr(gates), int(gates.stride(0)), float(gate_scale), L.ptr(bias), L.ptr(table), L.ptr(tok),
                                            L.ptr(c_prev), L.ptr(row_idx), int(n), int(d), L.ptr(c_new), L.ptr(h_new), L.ptr(a_next),
                                            a_pitch, int(k_next), int(off_next), float(next_scale if next_scale is not None else 1.0),
                                            _stream()))


def gru_cell(gates, bias, h_prev, row_idx, n, h_new, table=None, tok=None, a_next=None, k_next=0, off_next=0,
             gate_scale=None, next_scale=None):
    """Fused GRU cell (see e2e_gru_cell): gates [>=n,4D] fp32 in the blocks [r | z | n_x | n_h] -> h_new [>=n,D] (+ split
    of h into a_next).  h_prev is read through ``row_idx``.  ``gate_scale`` / ``next_scale`` as in lstm_cell."""
    _chk(gates, F32, "gates")
    _chk(bias, F32, "bias")
    _chk(h_prev, F32, "h_prev")
    _chk(row_idx, torch.int64, "row_idx", n)
    _chk(h_new, F32, "h_new")
    _chk(table, F32, "table")
    _chk(tok, torch.int64, "tok", n)
    f16 = gate_scale is not None
    if a_next is not None and _pieces(a_next, next_scale if f16 else None) != (2 if f16 else 3):
        raise TypeError("gru_cell: a_next does not match the operand format")
    d = h_prev.shape[1]
    if gates.shape[0] < n or gates.shape[1] < 4 * d or h_new.shape[0] < n or bias.numel() < 4 * d:
        raise ValueError("gru_cell: inconsistent shapes")
    if h_new.data_ptr() == h_prev.data_ptr():
        raise ValueError("gru_cell: h_new must not alias h_prev")
    a_pitch = int(a_next.stride(0)) if a_next is not None else 0
    if not f16:
        L.check(L.load().e2e_gru_cell(L.ptr(gates), int(gates.stride(0)), L.ptr(bias), L.ptr(table), L.ptr(tok), L.ptr(h_prev),
                                     L.ptr(row_idx), int(n), int(d), L.ptr(h_new), L.ptr(a_next),
                                     a_pitch, int(k_next), int(off_next), _stream()))
    else:
        L.check(L.load().e2e_gru_cell_f16x2(L.ptr(gates), int(gates.stride(0)), float(gate_scale), L.ptr(bias), L.ptr(table), L.ptr(tok),
                                           L.ptr(h_prev), L.ptr(row_idx), int(n), int(d), L.ptr(h_new), L.ptr(a_next),
                                           a_pitch, int(k_next), int(off_next), float(next_scale if next_scale is not None else 1.0),
                                           _stream()))


def conv3x3_unfold_split(x_nhwc, valid_rows, first_pixel, n_pixels, out, amax=None):
    """Unfold + split of a block of NHWC pixels (see e2e_conv3x3_unfold_split): out bf16 [>=n_pixels, 27*C] (exact 3-piece
    split), or fp16 [>=n_pixels, 18*C] with ``amax`` (int32 [1]: float bits of the input's maximum) for the 2-piece format."""
    _chk(x_nhwc, F32, "x_nhwc")
    _chk(valid_rows, I32, "valid_rows", x_nhwc.shape[0])
    n, h, w, c = x_nhwc.shape
    if amax is None:
        _chk(out, torch.bfloat16, "out", n_pixels * 27 * c)
        L.check(L.load().e2e_conv3x3_unfold_split(L.ptr(x_nhwc), L.ptr(valid_rows), n, h, w, c, int(first_pixel), int(n_pixels),
                                                 L.ptr(out), _stream()))
    else:
        _chk(out, torch.float16, "out", n_pixels * 18 * c)
        _chk(amax, I32, "amax", 1)
        L.check(L.load().e2e_conv3x3_unfold_split_f16x2(L.ptr(x_nhwc), L.ptr(valid_rows), n, h, w, c, int(first_pixel), int(n_pixels),
                                                       L.ptr(amax), L.ptr(out), _stream()))


def conv3x3_igemm_supported(c_in, c_out):
    """Whether e2e_conv3x3_igemm takes this layer shape."""
    return bool(L.load().e2e_conv3x3_igemm_supported(int(c_in), int(c_out)))


IGEMM_EPILOGUE = {"raw": 0, "relu": 1, "pool": 2}


def conv3x3_igemm(x_nhwc, valid_rows, w_split, bias, epilogue="relu"):
    """3x3 "same" convolution as one tcgen05 implicit split GEMM (see e2e_conv3x3_igemm): x [N,H,W,C] fp32 NHWC,
    w_split bf16 [3, Cout, 9C] (the pieces of weight.permute(0,2,3,1).reshape(Cout, 9C)).  ``epilogue``: "raw" -> the
    GEMM result [N*H*W, Cout]; "relu" -> relu(y + bias) masked to rows h < valid_rows[n], [N,H,W,Cout]; "pool" -> its
    2x2 ceil-mode max pool [N,ceil(H/2),ceil(W/2),Cout]."""
    _chk(x_nhwc, F32, "x_nhwc")
    _chk(valid_rows, I32, "valid_rows", x_nhwc.shape[0])
    _chk(w_split, torch.bfloat16, "w_split")
    n, h, w, c = x_nhwc.shape
    if w_split.dim() != 3 or w_split.shape[0] != 3 or w_split.shape[2] != 9 * c:
        raise ValueError("w_split must be [3, Cout, 9*%d], got %s" % (c, tuple(w_split.shape)))
    cout = w_split.shape[1]
    if epilogue not in IGEMM_EPILOGUE:
        raise ValueError("unknown epilogue " + str(epilogue))
    if epilogue != "raw":
        _chk(bias, F32, "bias", cout)
    if epilogue == "raw":
        out = torch.empty((n * h * w, cout), dtype=F32, device=x_nhwc.device)
    elif epilogue == "relu":
        out = torch.empty((n, h, w, cout), dtype=F32, device=x_nhwc.device)
    else:
        out = torch.empty((n, (h + 1) // 2, (w + 1) // 2, cout), dtype=F32, device=x_nhwc.device)
    L.check(L.load().e2e_conv3x3_igemm(L.ptr(x_nhwc), L.ptr(valid_rows), n, h, w, c, L.ptr(w_split),
                                      L.ptr(bias) if epilogue != "raw" else None, int(cout), IGEMM_EPILOGUE[epilogue],
                                      L.ptr(out), _stream()))
    return out


def conv_bias_relu_mask(y_nhwc, bias, valid_rows, amax_in=None, inv_w_scale=None, amax_out=None):
    """In place: y = relu(y + bias) on rows h < valid_rows[n], 0 elsewhere; y [N,H,W,C] NHWC.  With ``amax_in`` (the scale
    word of the layer's INPUT) y is an fp16x2 GEMM result: it is first multiplied by inv_w_scale / act_scale(amax_in);
    the maximum of the result goes to ``amax_out`` (the next layer's scale word)."""
    _chk(y_nhwc, F32, "y_nhwc")
    _chk(bias, F32, "bias", y_nhwc.shape[3])
    _chk(valid_rows, I32, "valid_rows", y_nhwc.shape[0])
    n, h, w, c = y_nhwc.shape
    if amax_in is None:
        L.check(L.load().e2e_conv_bias_relu_mask(L.ptr(y_nhwc), L.ptr(bias), L.ptr(valid_rows), n, h, w, c, 0, n * h * w, _stream()))
    else:
        _chk(amax_in, I32, "amax_in", 1)
        _chk(amax_out, I32, "amax_out", 1)
        L.check(L.load().e2e_conv_bias_relu_mask_scaled(L.ptr(y_nhwc), L.ptr(bias), L.ptr(valid_rows), n, h, w, c, 0, n * h * w,
                                                       L.ptr(amax_in), float(inv_w_scale), L.ptr(amax_out), _stream()))


# Hidden sizes of the packed recurrence: e2e_lstm_sequence / e2e_gru_sequence run one CTA per utterance group with one
# thread per unit up to SEQ_MAX_H; the *_wide entry points split the units of a group over a thread-block cluster and
# take multiples of SEQ_WIDE_UNIT up to SEQ_WIDE_MAX_H.
SEQ_MAX_H = 384
SEQ_WIDE_UNIT = 128
SEQ_WIDE_MAX_H = 1024


def sequence_supported(hidden):
    """True for the hidden sizes lstm_sequence / gru_sequence accept."""
    h = int(hidden)
    return 0 < h <= SEQ_MAX_H or (h % SEQ_WIDE_UNIT == 0 and h <= SEQ_WIDE_MAX_H)


def lstm_sequence(gates, out, frame_off, lens, group_first, group_rows, hidden, fw, bw=None):
    """Packed (B)LSTM recurrence (see e2e_lstm_sequence; e2e_lstm_sequence_wide above SEQ_MAX_H units).  gates
    [F, >=4H*dirs] fp32, out [F, >=H*dirs]; fw / bw = (bias [4H] | None, w_t [H,H,4], gate_off, out_off)."""
    _chk(gates, F32, "gates")
    _chk(out, F32, "out")
    for t, nm in ((frame_off, "frame_off"), (lens, "lens"), (group_first, "group_first"), (group_rows, "group_rows")):
        _chk(t, I32, nm)
    dirs = [fw] + ([bw] if bw is not None else [])
    for b, w, _, _ in dirs:
        _chk(b, F32, "bias", 4 * hidden)
        _chk(w, F32, "w_t", 4 * hidden * hidden)
    if bw is None:
        bw = (None, None, 0, 0)
    lib = L.load()
    fn = lib.e2e_lstm_sequence if hidden <= SEQ_MAX_H else lib.e2e_lstm_sequence_wide
    L.check(fn(L.ptr(gates), int(gates.stride(0)), L.ptr(out), int(out.stride(0)),
               L.ptr(frame_off), L.ptr(lens), L.ptr(group_first), L.ptr(group_rows),
               int(lens.numel()), int(hidden), int(group_first.numel()), len(dirs),
               L.ptr(fw[0]), L.ptr(fw[1]), int(fw[2]), int(fw[3]),
               L.ptr(bw[0]), L.ptr(bw[1]), int(bw[2]), int(bw[3]), _stream()))


def gru_sequence(gates, out, frame_off, lens, group_first, group_rows, hidden, fw, bw=None):
    """Packed (B)GRU recurrence (see e2e_gru_sequence; e2e_gru_sequence_wide above SEQ_MAX_H units).  gates
    [F, >=3H*dirs] fp32, out [F, >=H*dirs]; fw / bw = (bias [4H] = [b_ir+b_hr | b_iz+b_hz | b_in | b_hn] | None,
    w_t [H,H,4] (lane 3 zero), gate_off, out_off)."""
    _chk(gates, F32, "gates")
    _chk(out, F32, "out")
    for t, nm in ((frame_off, "frame_off"), (lens, "lens"), (group_first, "group_first"), (group_rows, "group_rows")):
        _chk(t, I32, nm)
    dirs = [fw] + ([bw] if bw is not None else [])
    for b, w, _, _ in dirs:
        _chk(b, F32, "bias", 4 * hidden)
        _chk(w, F32, "w_t", 4 * hidden * hidden)
    if bw is None:
        bw = (None, None, 0, 0)
    lib = L.load()
    fn = lib.e2e_gru_sequence if hidden <= SEQ_MAX_H else lib.e2e_gru_sequence_wide
    L.check(fn(L.ptr(gates), int(gates.stride(0)), L.ptr(out), int(out.stride(0)),
               L.ptr(frame_off), L.ptr(lens), L.ptr(group_first), L.ptr(group_rows),
               int(lens.numel()), int(hidden), int(group_first.numel()), len(dirs),
               L.ptr(fw[0]), L.ptr(fw[1]), int(fw[2]), int(fw[3]),
               L.ptr(bw[0]), L.ptr(bw[1]), int(bw[2]), int(bw[3]), _stream()))


def packed_subsample_ln(x, in_off, out_off, out_len, n_out, stride=1, g=1, weight=None, bias=None, eps=1e-5):
    """LayerNorm and / or frame sub-sampling of packed utterances (see e2e_packed_subsample_ln): x [F, W] fp32 ->
    out [n_out, g*W] with out[out_off[n] + j, s*W:(s+1)*W] = LN(x[in_off[n] + j*stride + s]) for j < out_len[n], s < g.
    ``weight`` None: a plain gather.  n_out (a host int) is the number of output rows."""
    _chk(x, F32, "x")
    for t, nm in ((in_off, "in_off"), (out_off, "out_off"), (out_len, "out_len")):
        _chk(t, I32, nm)
    n = in_off.numel()
    if x.dim() != 2 or out_off.numel() != n or out_len.numel() != n:
        raise ValueError("packed_subsample_ln: x must be [F, W] and in_off / out_off / out_len of one length")
    if weight is None and bias is not None:
        raise ValueError("packed_subsample_ln: a LayerNorm bias needs its weight")
    w = x.shape[1]
    _chk(weight, F32, "weight", w)
    _chk(bias, F32, "bias", w)
    out = torch.empty((int(n_out), g * w), dtype=F32, device=x.device)
    if n == 0 or n_out == 0:
        return out
    L.check(L.load().e2e_packed_subsample_ln(L.ptr(x), int(x.stride(0)), L.ptr(out), int(out.stride(0)), L.ptr(in_off),
                                            L.ptr(out_off), L.ptr(out_len), int(n), int(w), int(stride), int(g),
                                            L.ptr(weight), L.ptr(bias), float(eps), _stream()))
    return out


def conv1_direct(feat, weight, bias, valid_rows, n_freq, amax_out=None):
    """First VGG layer from the feature frames: feat [N,L,Cin*F] (last dim contiguous, rows of an utterance contiguous)
    -> relu(conv + bias) [N,L,F,Cout] NHWC.  ``amax_out`` (int32 [1], zeroed by the caller) receives the float bits of the
    maximum over the valid rows (the scale word of the next layer's fp16x2 operand)."""
    _chk(weight, F32, "weight")
    _chk(bias, F32, "bias")
    _chk(valid_rows, I32, "valid_rows", feat.shape[0])
    _chk(amax_out, I32, "amax_out", 1)
    if not feat.is_cuda or feat.dtype != F32 or feat.stride(2) != 1 or feat.stride(1) != feat.shape[2]:
        raise ValueError("conv1_direct: feat must be a CUDA fp32 [N,L,D] tensor with contiguous utterances")
    n, l, d = feat.shape
    cout, cin = weight.shape[0], weight.shape[1]
    if d != cin * n_freq:
        raise ValueError("conv1_direct: feature width %d != Cin*F" % d)
    out = torch.empty((n, l, n_freq, cout), dtype=F32, device=feat.device)
    if amax_out is None:
        L.check(L.load().e2e_conv1_direct(L.ptr(feat), int(feat.stride(0)), L.ptr(weight), L.ptr(bias), L.ptr(valid_rows),
                                         n, l, int(n_freq), int(cin), int(cout), L.ptr(out), _stream()))
    else:
        L.check(L.load().e2e_conv1_direct_amax(L.ptr(feat), int(feat.stride(0)), L.ptr(weight), L.ptr(bias), L.ptr(valid_rows),
                                              n, l, int(n_freq), int(cin), int(cout), L.ptr(out), L.ptr(amax_out), _stream()))
    return out


def conv_bias_relu_mask_pool(y_nhwc, bias, valid_rows, amax_in=None, inv_w_scale=None, amax_out=None):
    """max_pool2d(2, 2, ceil_mode=True) of mask(relu(y + bias)); y [N,H,W,C] NHWC -> [N,ceil(H/2),ceil(W/2),C].
    ``amax_in`` / ``inv_w_scale`` / ``amax_out`` as in conv_bias_relu_mask."""
    _chk(y_nhwc, F32, "y_nhwc")
    _chk(bias, F32, "bias", y_nhwc.shape[3])
    _chk(valid_rows, I32, "valid_rows", y_nhwc.shape[0])
    n, h, w, c = y_nhwc.shape
    out = torch.empty((n, (h + 1) // 2, (w + 1) // 2, c), dtype=F32, device=y_nhwc.device)
    if amax_in is None:
        L.check(L.load().e2e_conv_bias_relu_mask_pool(L.ptr(y_nhwc), L.ptr(bias), L.ptr(valid_rows), n, h, w, c, L.ptr(out), _stream()))
    else:
        _chk(amax_in, I32, "amax_in", 1)
        _chk(amax_out, I32, "amax_out", 1)
        L.check(L.load().e2e_conv_bias_relu_mask_pool_scaled(L.ptr(y_nhwc), L.ptr(bias), L.ptr(valid_rows), n, h, w, c, L.ptr(out),
                                                            L.ptr(amax_in), float(inv_w_scale), L.ptr(amax_out), _stream()))
    return out


def launch_count():
    return int(L.load().e2e_launch_count())


def add_launch_count(n):
    L.load().e2e_add_launch_count(int(n))
