"""Drop-in ``BeamDecoder`` / ``Hypothesis`` running the joint CTC/attention(+RNNLM)
beam search batched over utterances on one B200.

Mirrors the interface of ``/root/reference/src/decode.py``:

* ``BeamDecoder(asr, emb_decoder, beam_size, min_len_ratio, max_len_ratio,
  lm_path='', lm_config='', lm_weight=0.0, ctc_weight=0.0)``      (decode.py:17-48)
* ``.forward(audio_feature[1,L,D], feature_len[1]) -> list[Hypothesis]`` best first
  (decode.py:65-183), ``.create_msg()`` (decode.py:50-63) and the public attributes
  ``beam_size, min_len_ratio, max_len_ratio, asr, apply_ctc, ctc_w, ctc_beam_size,
  apply_lm, lm_w, lm_path, lm, apply_emb, emb_decoder``
* ``Hypothesis.outIndex`` / ``.avgScore()`` / ``.output_seq`` / ``.output_scores``
  (decode.py:186-217,279-281)

so ``bin/test_asr.py:80-82,159-173`` can use it unchanged.  In addition
``decode_batch(features[U,Lmax,D], lengths[U])`` decodes many utterances at once —
the reference fans single utterances out to joblib processes
(``bin/test_asr.py:138-139``); here they share every kernel launch.

Per decode step the device runs: the batched PyTorch model step (``stepper.py``),
then (3a) ``e2e_beam_candidates`` (``e2e_emb_fuse_candidates`` for a model decoded with the word-embedding
fusion plug-in, ``emb_decoder``), (2) ``e2e_ctc_prefix_step`` (the fused lazy prefix
kernel; ``e2e_ctc_prefix_score``, the eager one, with ``lazy_prefix = False``), (3b)
``e2e_beam_combine_prune``; the posteriors come from (1) ``e2e_ctc_log_softmax``
once per batch.  Nothing is copied to the host until the final N-best.
There is no CPU fallback: inputs must live on a CUDA device.
"""
import os

import numpy as np
import torch
import torch.nn.functional as F
import yaml
from torch import nn

from . import _lib as L
from . import ops
from .model import RNNLM
from .stepper import BatchedStepper

CTC_BEAM_RATIO = 1.5      # decode.py:10
LOG_ZERO = -10000000.0    # decode.py:11
EOS_THRESHOLD = 1.5       # decode.py:220


class Hypothesis:
    """Result record with the reference's read interface (decode.py:186-217,279-281)."""

    def __init__(self, tokens, scores, avg):
        self._tokens = np.asarray(tokens, dtype=np.int64)
        self._scores = np.asarray(scores, dtype=np.float32)
        self._avg = np.float32(avg)

    @property
    def outIndex(self):
        return [int(t) for t in self._tokens]

    @property
    def output_seq(self):
        return [torch.tensor(int(t)) for t in self._tokens]

    @property
    def output_scores(self):
        return [torch.tensor(float(s), dtype=torch.float32) for s in self._scores]

    def avgScore(self):
        assert len(self._scores) != 0
        return torch.tensor(float(self._avg), dtype=torch.float32)

    def __repr__(self):
        return "Hypothesis(len=%d, avg=%.6f)" % (len(self._tokens), float(self._avg))


class _Fp32Math:
    """The reference computes in fp32 on the CPU: keep cuBLAS/cuDNN out of TF32 and keep the
    bf16 split GEMMs (stepper.SplitLinear) on full fp32 accumulation."""

    def __enter__(self):
        mm = torch.backends.cuda.matmul
        self.prev = (mm.allow_tf32, torch.backends.cudnn.allow_tf32, mm.allow_bf16_reduced_precision_reduction,
                     mm.allow_fp16_reduced_precision_reduction)
        mm.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        mm.allow_bf16_reduced_precision_reduction = False
        mm.allow_fp16_reduced_precision_reduction = False

    def __exit__(self, *exc):
        mm = torch.backends.cuda.matmul
        (mm.allow_tf32, torch.backends.cudnn.allow_tf32, mm.allow_bf16_reduced_precision_reduction,
         mm.allow_fp16_reduced_precision_reduction) = self.prev


class BeamDecoder(nn.Module):
    ''' Beam decoder for ASR (batched, device resident) '''

    def __init__(self, asr, emb_decoder, beam_size, min_len_ratio, max_len_ratio,
                 lm_path='', lm_config='', lm_weight=0.0, ctc_weight=0.0):
        super().__init__()
        self.beam_size = beam_size
        self.min_len_ratio = min_len_ratio
        self.max_len_ratio = max_len_ratio
        self.asr = asr
        assert self.asr.enable_att                                     # decode.py:27
        if not 1 <= beam_size <= ops.BEAM_MAX:
            raise ValueError("beam_size must be in 1..%d" % ops.BEAM_MAX)

        self.apply_ctc = ctc_weight > 0
        if self.apply_ctc:
            assert self.asr.ctc_weight > 0, 'ASR was not trained with CTC decoder'   # decode.py:32
            self.ctc_w = ctc_weight
            self.ctc_beam_size = int(CTC_BEAM_RATIO * self.beam_size)

        self.apply_lm = lm_weight > 0
        if self.apply_lm:
            self.lm_w = lm_weight
            self.lm_path = lm_path
            cfg = yaml.load(open(lm_config, 'r'), Loader=yaml.FullLoader)
            self.lm = RNNLM(self.asr.vocab_size, **cfg['model'])
            self.lm.load_state_dict(torch.load(self.lm_path, map_location='cpu')['model'])
            self.lm.eval()

        self.apply_emb = emb_decoder is not None
        if self.apply_emb:
            # the word-embedding fusion plug-in (src/plugin.py EmbeddingRegularizer, model.EmbeddingRegularizer)
            if getattr(emb_decoder, "use_bert", False):
                raise NotImplementedError("embedding fusion with a BERT table (use_bert) is not supported")
            if not getattr(emb_decoder, "apply_fuse", False):
                # the reference would take the plug-in's None log-prob as the attention scores and fail on it
                raise ValueError("emb_decoder has no probability fusion (apply_fuse is False, fuse == 0): nothing to decode with")
            self.emb_decoder = emb_decoder

        # knobs of the device path (not part of the reference interface)
        self.fast_math = False          # MUFU log-add-exp in the prefix-score kernel
        # log-add-exp evaluator of the prefix-score kernel: "poly" (default: MUFU.EX2 + degree-8 polynomial, no table and no
        # shared-memory look-up on the dependent chain; within 2 ulp of the oracle on every chain test, measured 20 % faster
        # than the table in the decode), "lut" (table, 1 ulp), "poly_estrin" (eager kernel only)
        self.prefix_math = os.environ.get("E2E_PREFIX_MATH", "poly")
        self.skip_dead_rows = True      # do not write state rows t < len(prefix) nobody reads back
        # fused per-step prefix kernel with lazy state evaluation (csrc/prefix_lazy.cu): states only for the <= B
        # hypotheses the beam kept, psi alone for the B*C candidates.  False: the eager kernel (csrc/prefix_score.cu)
        self.lazy_prefix = os.environ.get("E2E_PREFIX_LAZY", "1") != "0"
        self.split_gemm = True          # fp32-accurate 3-way bf16 split of the recurrent GEMMs (stepper.py)
        # operand format of the RNNLM's recurrent GEMMs: "bf16x3" (six partial products) or "fp16x2" (three; every
        # input is a hidden state, |h| <= 1).  The environment variable is for A/B runs of the bench.
        self.lm_split = os.environ.get("E2E_LM_SPLIT", "bf16x3")
        # the same choice for the VGG convolutions (their activations have no fixed range: the scale is chosen on
        # the device from the running maximum of every layer's input, csrc/conv_split.cu)
        self.vgg_split = os.environ.get("E2E_VGG_SPLIT", "bf16x3")
        # bf16x3 VGG convolutions: "igemm" runs the 128-channel layer as one tcgen05 implicit GEMM (csrc/conv_igemm.cu),
        # "unfold" every layer as unfold + three library GEMMs + epilogue kernel (model.VGGFrontEnd.conv_path); same bits
        self.vgg_conv = "igemm"
        self.fused_attention = True     # hand-written location-aware attention kernel (csrc/attention_full.cu)
        # replay the LSTM stacks of a decode step from CUDA graphs when few utterances are live (stepper._FusedLstm): the tail of a
        # decode is bound by the host's launch rate
        self.step_graphs = os.environ.get("E2E_STEP_GRAPHS", "1") != "0"
        self._stepper = None            # (device, split_gemm, stepper): weights are split once per device
        self.profile_prefix = False     # bench.py: CUDA-event pair around every prefix-score launch
        self.prefix_events = []         # (start, end, cand_frames [SURVEY §8d formula], cand_frames actually computed)
        self.profile_phases = False     # tools/profile_phases.py: CUDA-event time per phase of decode_batch
        self.phase_ms = {}
        self.last_stats = {}
        self.last_h2d_bytes = 0         # decode_batch_from_host: bytes of the last host->device feature copy

    def __getstate__(self):
        # bin/test_asr.py:108,138 deep-copies and pickles the decoder: drop the per-device caches
        d = self.__dict__.copy()
        d["_stepper"], d["prefix_events"] = None, []
        d.pop("_copier", None)
        return d

    def create_msg(self):
        msg = ['Decode spec| Beam size = {}\t| Min/Max len ratio = {}/{}'.format(
            self.beam_size, self.min_len_ratio, self.max_len_ratio)]
        if self.apply_ctc:
            msg.append('           |Joint CTC decoding enabled \t| weight = {:.2f}\t'.format(self.ctc_w))
        if self.apply_lm:
            msg.append('           |Joint LM decoding enabled \t| weight = {:.2f}\t| src = {}'.format(self.lm_w, self.lm_path))
        if self.apply_emb:
            msg.append('           |Joint Emb. decoding enabled \t| weight = {:.2f}'.format(
                float(self.emb_decoder.fuse_lambda.mean().cpu().item())))
        return msg

    # ------------------------------------------------------------------------------------------
    def forward(self, audio_feature, feature_len):
        assert audio_feature.shape[0] == 1, "Batchsize == 1 is required for beam search"   # decode.py:67
        return self.decode_batch(audio_feature, feature_len)[0]

    ENCODER_CHUNK = 128       # utterances per encoder chunk (stepper.encode); the host->device copy is pipelined in the same units

    @torch.no_grad()
    def decode_batch_from_host(self, audio_feature, feature_len, device, return_arrays=False):
        """``decode_batch`` for PINNED HOST features [U,Lmax,D] (zero padded) and host lengths [U].  Only the valid frames
        of every utterance cross the bus (a dev-clean-like set is 4.6x smaller than its padded tensor; the padding is a
        device-side memset), one asynchronous copy per utterance, issued longest first on a COPY STREAM in chunks of
        ``ENCODER_CHUNK`` utterances — the order and the units in which the encoder consumes them, so the encoder starts
        on the first chunk while the rest is still in flight (one event per chunk).  ``last_h2d_bytes`` holds the bytes copied."""
        if audio_feature.is_cuda:
            return self.decode_batch(audio_feature, feature_len, return_arrays)
        if audio_feature.shape[0] == 0 and len(feature_len) == 0:      # an empty shard
            self.last_h2d_bytes = 0
            return self._no_utterances(torch.device(device) if return_arrays == "device" else "cpu", return_arrays)
        if not audio_feature.is_pinned():
            raise ValueError("decode_batch_from_host needs pinned host features (torch.Tensor.pin_memory): pageable memory "
                             "would turn every copy into a synchronous one")
        dev = torch.device(device)
        lens = [int(n) for n in feature_len]
        n_utts = len(lens)
        if audio_feature.dim() != 3 or n_utts != audio_feature.shape[0] or (lens and max(lens) > audio_feature.shape[1]):
            raise ValueError("decode_batch_from_host: features [U,Lmax,D] and lengths [U] disagree")
        # decode order (decode_batch's own: longest output first, ties by index): rows arrive already sorted
        max_np = np.array([int(np.ceil(n * self.max_len_ratio)) for n in lens], dtype=np.int64)
        order = np.lexsort((np.arange(n_utts), -max_np)) if n_utts else np.zeros(0, dtype=np.int64)
        inverse = np.argsort(order)
        with torch.cuda.device(dev):
            main = torch.cuda.current_stream(dev)
            feat_dev = torch.zeros(audio_feature.shape, dtype=torch.float32, device=dev)
            len_dev = torch.as_tensor(np.asarray(lens, dtype=np.int64)[order]).to(dev, non_blocking=True)
            copier = self._copy_stream(dev)
            copier.wait_stream(main)                                   # the memset above
            feat_dev.record_stream(copier)
            n_chunks = (n_utts + self.ENCODER_CHUNK - 1) // self.ENCODER_CHUNK
            events = [torch.cuda.Event() for _ in range(n_chunks)]
            for ev in events:
                ev.record(copier)                      # creates the underlying cudaEvent_t (re-recorded by the copy loop)
            import ctypes
            lens32 = np.asarray(lens, dtype=np.int32)
            order64 = np.ascontiguousarray(order, dtype=np.int64)
            ev_arr = (ctypes.c_void_p * max(1, n_chunks))(*[ev.cuda_event for ev in events])
            if audio_feature.dtype != torch.float32 or not audio_feature.is_contiguous():
                raise ValueError("decode_batch_from_host: features must be a contiguous fp32 tensor")
            L.check(L.load().e2e_copy_rows_h2d(audio_feature.data_ptr(), feat_dev.data_ptr(), int(audio_feature.shape[1] * audio_feature.shape[2]),
                                              int(audio_feature.shape[2]), lens32.ctypes.data, order64.ctypes.data, n_utts,
                                              self.ENCODER_CHUNK, ev_arr, copier.cuda_stream))
            self.last_h2d_bytes = sum(lens) * audio_feature.shape[2] * 4 + feature_len.numel() * feature_len.element_size()
            enc_mod = self.asr.encoder

            def rows_ready(lo, hi):          # the current stream waits for the copies of rows [lo, hi)
                for c in range(lo // self.ENCODER_CHUNK, (max(hi, lo + 1) - 1) // self.ENCODER_CHUNK + 1):
                    torch.cuda.current_stream(dev).wait_event(events[c])

            enc_mod.chunk_ready = rows_ready          # stepper.encode / Encoder.forward_ragged_packed call it before touching rows
            try:
                out = self._decode_batch(feat_dev, len_dev, return_arrays)
            finally:
                enc_mod.chunk_ready = None
                main.wait_stream(copier)
            if return_arrays:
                sel = torch.as_tensor(inverse, device=out[0].device)
                return tuple(a.index_select(0, sel) for a in out)
            return [out[int(k)] for k in inverse]

    def _copy_stream(self, dev):
        st = getattr(self, "_copier", None)
        if st is None or st[0] != dev:
            st = (dev, torch.cuda.Stream(device=dev))
            self._copier = st
        return st[1]

    @torch.no_grad()
    def decode_batch(self, audio_feature, feature_len, return_arrays=False):
        """audio_feature [U,Lmax,D] (zero padded), feature_len [U] -> list (per utterance) of
        N-best ``Hypothesis`` lists, best first.  ``return_arrays=True`` returns the raw
        (tokens, scores, lens, avg, n) CPU tensors instead, ``return_arrays="device"`` the same as CUDA tensors
        (no read-back: the sharded driver packs and gathers them on the device)."""
        if not audio_feature.is_cuda:
            raise L.E2EError("BeamDecoder has no CPU path: move the features and the decoder to a CUDA device")
        if audio_feature.shape[0] == 0:                                # an empty shard: nothing to launch
            return self._no_utterances(audio_feature.device if return_arrays == "device" else "cpu", return_arrays)
        # the hand-written kernels are enqueued on the CURRENT device's current stream: make the features' device current
        with torch.cuda.device(audio_feature.device):
            return self._decode_batch(audio_feature, feature_len, return_arrays)

    def _no_utterances(self, where, return_arrays):
        self.last_stats = {"utterances": 0, "steps": 0, "enc_frames": [], "cand_frames": 0}
        if not return_arrays:
            return []
        b = self.beam_size
        return (torch.zeros((0, b, 1), dtype=torch.int32, device=where), torch.zeros((0, b, 1), dtype=torch.float32, device=where),
                torch.zeros((0, b), dtype=torch.int32, device=where), torch.zeros((0, b), dtype=torch.float32, device=where),
                torch.zeros((0,), dtype=torch.int32, device=where))

    def _decode_batch(self, audio_feature, feature_len, return_arrays):
        dev = audio_feature.device
        n_utts = audio_feature.shape[0]
        beam = self.beam_size
        vocab = self.asr.vocab_size
        n_cand = self.ctc_beam_size if self.apply_ctc else 0
        ctc_w = self.ctc_w if self.apply_ctc else 0.0
        lm_w = self.lm_w if self.apply_lm else 0.0
        lens_cpu = feature_len.detach().cpu().long()
        # decode.py:74-78: output length limits come from the INPUT length
        max_np = np.array([int(np.ceil(int(l) * self.max_len_ratio)) for l in lens_cpu], dtype=np.int64)
        min_np = np.array([int(np.ceil(int(l) * self.min_len_ratio)) for l in lens_cpu], dtype=np.int64)
        # Longest first: the utterances still decoding at any step are then a prefix of the batch,
        # and every kernel / model step only visits that prefix.
        order = np.lexsort((np.arange(n_utts), -max_np)) if n_utts else np.zeros(0, dtype=np.int64)
        inverse = np.argsort(order)
        if n_utts and not np.array_equal(order, np.arange(n_utts)):
            sel = torch.as_tensor(order, device=dev)
            audio_feature, feature_len = audio_feature.index_select(0, sel), feature_len.to(dev).index_select(0, sel)
        max_len = torch.as_tensor(max_np[order], dtype=torch.int32)
        min_len = torch.as_tensor(min_np[order], dtype=torch.int32)
        n_steps = int(max_len.max()) if n_utts else 0
        n_run = [int((max_np > s).sum()) for s in range(n_steps)]      # live utterances per step

        marks = []

        coarse = self.profile_phases == "coarse"        # phase boundaries only: nothing is recorded inside the step loop

        def mark(name, boundary=False):
            if self.profile_phases and (boundary or not coarse):
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                marks.append((name, e))

        with _Fp32Math():
            mark("start", True)
            emb = self.emb_decoder if self.apply_emb else None
            knobs = (self.split_gemm, self.fused_attention, self.lm_split, self.vgg_split, self.step_graphs, self.vgg_conv, emb)
            if self._stepper is None or self._stepper[0] != dev or self._stepper[1] != knobs:
                self._stepper = (dev, knobs, BatchedStepper(self.asr, self.lm if self.apply_lm else None,
                                                            self.split_gemm, self.fused_attention, self.lm_split, self.vgg_split,
                                                            self.step_graphs, self.vgg_conv, emb))
            stepper = self._stepper[2]
            stepper.mark = mark
            enc, enc_len = stepper.encode(audio_feature, feature_len.to(dev))
            mark("encode", True)
            enc_len32 = enc_len.to(torch.int32).contiguous()
            stepper.start(enc, enc_len, beam)
            t_max = enc.shape[1]
            buf = ops.BeamBuffers(n_utts, beam, n_cand, n_steps, min_len, max_len, dev)
            fusion = stepper.emb
            if fusion is not None:
                fused = torch.empty((n_utts * beam, vocab), dtype=torch.float32, device=dev)     # the fused log-probs of a step
            r_prev = r_a = r_b = x = None
            if self.apply_ctc:
                lin = self.asr.ctc_layer[0]
                logits = F.linear(enc, lin.weight, lin.bias).contiguous()          # cuBLAS; ReLU + log-softmax fused in (1)
                x = ops.ctc_log_softmax(logits, enc_len32, apply_relu=True)        # decode.py:94-95
                del logits                                                         # [U,Tmax,V]: as large as x with a subword vocabulary
                r_prev = r_init = ops.ctc_init_state(x, enc_len32)                 # decode.py:97
                lazy = self.lazy_prefix and not self.fast_math and ops.prefix_step_supported(vocab, beam, n_cand)
                r_a = torch.empty((n_utts, t_max, beam if lazy else beam * n_cand, 2), dtype=torch.float32, device=dev)
                r_b = torch.empty_like(r_a)
            pflags = (L.PREFIX_FAST_MATH if self.fast_math else 0) | (L.PREFIX_SKIP_DEAD_ROWS if self.skip_dead_rows else 0)
            if not self.fast_math:
                pflags |= {"lut": 0, "poly": L.PREFIX_POLY_MATH, "poly_estrin": L.PREFIX_POLY_MATH | L.PREFIX_POLY_ESTRIN}[self.prefix_math]
            if self.profile_prefix and self.apply_ctc:
                t_np, s_np = enc_len.cpu().numpy().astype(np.int64), max_len.numpy().astype(np.int64)

            mark("ctc_posterior", True)
            for step in range(n_steps):                                            # decode.py:104
                k = n_run[step]
                if fusion is None:
                    att_logits, lm_logits = stepper.step(buf.last_tok64[:k].view(-1), k)
                    mark("step_rest")
                    ops.beam_candidates(att_logits, k, beam, vocab, n_cand, buf.n_active, buf.att_stats, buf.cand)
                else:
                    # embedding fusion: the fused log-probs take the attention log-softmax's place, with zero statistics
                    dec_logits, lm_logits, emb_logits = stepper.step(buf.last_tok64[:k].view(-1), k)
                    mark("step_rest")
                    att_logits = ops.emb_fuse_candidates(dec_logits, emb_logits, k, beam, vocab, n_cand, fusion.scale, fusion.lam,
                                                         fusion.eps, buf.n_active, fused[:k * beam], buf.att_stats, buf.cand)
                if self.apply_ctc:
                    r_cur = r_a if (step % 2 == 0) else r_b
                    if self.profile_prefix:
                        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        ev0.record()
                    if lazy:
                        # states of the live hypotheses from their parents' (the init buffer at steps 0 and 1) + psi of all candidates
                        ops.ctc_prefix_step(x, vocab, enc_len32, r_init if step <= 1 else r_prev, buf.parent_slot.view(-1),
                                            buf.last_tok.view(-1), buf.parent_tok.view(-1), buf.prefix_len.view(-1), buf.n_active,
                                            buf.cand, beam, n_cand, pflags & ~L.PREFIX_SKIP_DEAD_ROWS,
                                            psi=buf.psi, r_out=r_cur, status=buf.status, n_run=k)
                    else:
                        ops.ctc_prefix_score(x, vocab, enc_len32, r_prev, buf.prev_lane.view(-1), buf.last_tok.view(-1),
                                             buf.prefix_len.view(-1), buf.n_active, buf.cand, beam, n_cand, pflags,
                                             psi=buf.psi, r_out=r_cur, status=buf.status, n_run=k)
                    if self.profile_prefix:
                        ev1.record()
                        act = s_np > step                     # utterances that still decode at this step
                        hyps = (1 if step == 0 else beam) * n_cand      # H_s * C (n_live < B after an <eos> closure is ignored)
                        self.prefix_events.append((ev0, ev1, float(hyps * t_np[act].sum()),
                                                   float(hyps * np.maximum(t_np[act] - max(1, step), 0).sum())))
                    r_prev = r_cur
                ops.beam_combine_prune(buf, att_logits, lm_logits, vocab, step, ctc_w, lm_w, EOS_THRESHOLD, n_run=k)
                mark("beam_kernels")
                stepper.reorder(buf.parent_row)
                mark("reorder")

            mark("steps", True)
            tok, sc, ln, avg, n = ops.beam_finalize(buf)
            mark("finalize", True)
            status = buf.status.cpu()
            inv = torch.as_tensor(inverse, device=dev)
            # N-best back to the host through pinned buffers (the caching host allocator reuses them)
            dev_out = [a.index_select(0, inv) for a in (tok, sc, ln, avg, n)]
            if return_arrays == "device":
                tok, sc, ln, avg, n = dev_out              # stays on the device (shard.RaggedPacker packs it there)
            else:
                host_out = [torch.empty(a.shape, dtype=a.dtype, pin_memory=True) for a in dev_out]
                for h, a in zip(host_out, dev_out):
                    h.copy_(a, non_blocking=True)
                torch.cuda.current_stream(dev).synchronize()
                tok, sc, ln, avg, n = host_out
            status = status[torch.as_tensor(inverse)]

        if self.profile_phases:
            torch.cuda.synchronize()
            for (_, a), (name, b) in zip(marks[:-1], marks[1:]):
                self.phase_ms[name] = self.phase_ms.get(name, 0.0) + a.elapsed_time(b)
        self._raise_like_reference(status, None, max_len)
        enc_len_cpu = enc_len.cpu()[torch.as_tensor(inverse)]
        max_len = max_len[torch.as_tensor(inverse)]
        self.last_stats = {
            "utterances": n_utts, "steps": n_steps, "enc_frames": [int(t) for t in enc_len_cpu],
            # unit count of SURVEY.md §8d: sum_s H_s * C * T per utterance
            "cand_frames": int(sum((1 + (int(s) - 1) * beam) * n_cand * int(t)
                                   for s, t in zip(max_len, enc_len_cpu) if int(s) > 0)) if self.apply_ctc else 0,
        }
        if return_arrays:
            return tok, sc, ln, avg, n
        return nbest_from_arrays(tok, sc, ln, avg, n)

    @staticmethod
    def _raise_like_reference(status, n_out, max_len):
        bad = status.nonzero().reshape(-1).tolist()
        for u in bad:
            s = int(status[u])
            if s & L.STATUS_PREFIX_TOO_LONG:
                raise IndexError("utterance %d: hypothesis longer than the encoder output "
                                 "(src/ctc.py:85; needs ceil(L*max_len_ratio) <= T_enc)" % u)
            if s & L.STATUS_TOKEN_NOT_CAND:
                raise ValueError("utterance %d: beam winner is not in the CTC candidate list "
                                 "(src/decode.py:252: x is not in list)" % u)


def nbest_from_arrays(tok, sc, ln, avg, n):
    out = []
    tok, sc, ln, avg, n = (a.numpy() for a in (tok, sc, ln, avg, n))
    for u in range(tok.shape[0]):
        hyps = []
        for k in range(int(n[u])):
            m = int(ln[u, k])
            hyps.append(Hypothesis(tok[u, k, :m], sc[u, k, :m], avg[u, k]))
        out.append(hyps)
    return out
