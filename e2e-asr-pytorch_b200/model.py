"""Acoustic model + RNNLM with the reference's module tree.

The ``forward`` methods are plain PyTorch restatements of the reference modules (north_star keeps
the encoder, the attention decoder step and the RNNLM step library backed); the ``*_split`` /
``*_packed`` methods are the device path of the encoder (SURVEY §8f row f-4: library GEMMs on an
exact bf16 split + hand-written kernels for everything around them).  The modules exist here so that

* ``bench.py`` / ``smoke()`` can build the BASELINE configs on the GPU box,
  where ``/root/reference`` is absent, with random-init weights, and
* checkpoints of the reference load unchanged: parameter names and shapes
  follow ``/root/reference/src/asr.py`` (ASR :13-52, Decoder :183-270,
  Attention :273-364, Encoder :390-476), ``src/module.py`` (VGGExtractor
  :659-716, RNNLayer :1003-1081, LocationAwareAttention :1135-1173,
  ScaleDotAttention :1120-1132) and ``src/lm.py`` (RNNLM :5-38), so
  ``ref_model.load_state_dict(our_model.state_dict())`` works both ways.

The modules also expose the small stateful protocol the reference's
``BeamDecoder`` drives (``decoder.init_state/get_state/set_state/get_query``,
``attention.reset_mem/set_mem``, ``asr.set_state``): the CPU oracle
(``oracle/beam_oracle.py``) uses it one hypothesis at a time, exactly like the
reference.  The batched device beam search (``decode.py``/``stepper.py``) does
not call these forward methods per hypothesis; it reads the weights and runs
its own batched step.

Supported subset (what the shipped configs under ``config/`` need for decode):
encoder ``vgg`` 0/1 + (B)LSTM/GRU layers with drop/concat sub-sampling, optional
LayerNorm and projection; attention ``loc`` or ``dot``; LSTM/GRU decoder; RNNLM
LSTM/GRU with or without embedding tying.
"""
import math

import numpy as np
import torch
from torch import nn
import torch.nn.functional as F

FBANK_SIZE = 40   # src/option.py / module.py check_dim: fbank features come in blocks of 40


def reference_init_(module):
    """Weight init of ``src/util.py:60-83`` (Embedding ~ N(0,1); matrices and
    conv kernels ~ N(0, 1/fan_in); biases zero), applied through
    ``nn.Module.apply``."""
    if isinstance(module, nn.Embedding):
        module.weight.data.normal_(0, 1)
        return
    for p in module.parameters():
        d = p.data
        if d.dim() == 1:
            d.zero_()
        elif d.dim() == 2:
            d.normal_(0, 1.0 / math.sqrt(d.size(1)))
        elif d.dim() in (3, 4):
            fan = d.size(1)
            for k in d.size()[2:]:
                fan *= k
            d.normal_(0, 1.0 / math.sqrt(fan))
        else:
            raise NotImplementedError


def split_gemm_rows(x, lin, a_bytes=3 << 30):
    """y = x @ W^T (no bias) as fp32-accurate bf16 tensor-core GEMMs: x [F, K] fp32 (contiguous, CUDA),
    ``lin`` a stepper.SplitLinear holding the weight's three operand stacks.  The exact 3-piece split of a
    block of rows is written by one hand-written kernel (csrc/lstm_step.cu), the three GEMMs accumulate in
    place; row blocks bound the size of the bf16 operand."""
    from . import ops
    f, k = x.shape
    m_out = lin.b0.shape[1]
    y = torch.empty((f, m_out), dtype=torch.float32, device=x.device)
    blk = max(1, min(f, a_bytes // (3 * k * 2)))
    a = torch.empty((blk, 3 * k), dtype=torch.bfloat16, device=x.device)
    for r0 in range(0, f, blk):
        m = min(blk, f - r0)
        ops.lstm_split_rows(x[r0:r0 + m], None, m, a, k, 0)
        am, ym = a[:m], y[r0:r0 + m]
        torch.mm(am, lin.b2, out_dtype=torch.float32, out=ym)
        torch.addmm(ym, am[:, :2 * k], lin.b1, out_dtype=torch.float32, out=ym)
        torch.addmm(ym, am[:, :k], lin.b0, out_dtype=torch.float32, out=ym)
    return y


class VGGFrontEnd(nn.Module):
    """2x(conv3x3,conv3x3,maxpool2) front end, 4x time reduction (module.py:659-716)."""

    def __init__(self, input_dim):
        super().__init__()
        if input_dim % 13 == 0:
            self.in_channel, self.freq_dim = input_dim // 13, 13
        elif input_dim % FBANK_SIZE == 0:
            self.in_channel, self.freq_dim = input_dim // FBANK_SIZE, FBANK_SIZE
        else:
            raise ValueError("VGG front end needs 13k (MFCC) or 40k (fbank) features, got %d" % input_dim)
        c1, c2 = 128, 256
        self.out_dim = (self.freq_dim // 4) * c2
        self.extractor = nn.Sequential(
            nn.Conv2d(self.in_channel, c1, 3, stride=1, padding=1), nn.ReLU(),
            nn.Conv2d(c1, c1, 3, stride=1, padding=1), nn.ReLU(),
            nn.MaxPool2d(2, stride=2, ceil_mode=True),
            nn.Conv2d(c1, c2, 3, stride=1, padding=1), nn.ReLU(),
            nn.Conv2d(c2, c2, 3, stride=1, padding=1), nn.ReLU(),
            nn.MaxPool2d(2, stride=2, ceil_mode=True))

    def _as_image(self, feat):
        drop = feat.shape[1] % 4
        if drop:
            feat = feat[:, :-drop, :].contiguous()
        n, t, _ = feat.shape
        return feat.view(n, t, self.in_channel, self.freq_dim).transpose(1, 2)

    def forward(self, feat, feat_len):
        img = self.extractor(self._as_image(feat))              # [N, 256, T/4, F/4]
        out = img.transpose(1, 2).contiguous()
        return out.view(out.shape[0], out.shape[1], self.out_dim), feat_len // 4

    def forward_masked(self, feat, feat_len):
        """Batched variant for ragged utterances: activations beyond each
        utterance's own length are zeroed after every convolution, so a padded
        batch row sees the same zero padding a batch-1 call would."""
        img = self._as_image(feat)
        n, _, t, _ = img.shape
        own = (feat_len // 4 * 4).to(img.device)          # a batch-1 call crops to a multiple of 4

        def keep(a):
            valid = own // (t // a.shape[2])
            m = torch.arange(a.shape[2], device=a.device)[None, :] < valid[:, None]
            return a * m[:, None, :, None].to(a.dtype)

        img = keep(img)
        for layer in self.extractor:
            img = layer(img)
            if isinstance(layer, nn.ReLU):
                img = keep(img)
        out = img.transpose(1, 2).contiguous()
        return out.view(out.shape[0], out.shape[1], self.out_dim), feat_len // 4


    # -- fp32-accurate tensor-core path (CUDA only; SURVEY §8f row f-4) ---------------------------------
    A_BYTES = 3 << 30      # budget of the unfolded bf16 operand per GEMM block

    conv_split_format = "bf16x3"     # "fp16x2": 2-piece fp16 operands, scale per layer input chosen on the device (csrc/conv_split.cu)
    # bf16x3 layers: "igemm" runs the layers with at most IGEMM_MAX_COUT output channels as one tcgen05 implicit split GEMM
    # with the epilogue fused (csrc/conv_igemm.cu, bit-equal to the unfold path); "unfold": every layer as unfold+split ->
    # three library GEMMs -> epilogue kernel.  The 256-channel layers stay on the library either way: at N = 256 its GEMMs
    # run the split products at 1.1-1.2 PFLOP/s, the implicit GEMM at 0.6 (at N = 128 the library reaches 0.65), DESIGN §4.
    conv_path = "igemm"
    IGEMM_MAX_COUT = 128

    def _split_weights(self, conv):
        """[9*Cin, Cout] GEMM weights of a 3x3 convolution as the operand stacks of stepper.SplitLinear /
        SplitLinearF16 (k = (dy*3+dx)*Cin + c), cached per layer, device and format."""
        from .stepper import SplitLinear, SplitLinearF16
        cache = self.__dict__.setdefault("_split_cache", {})
        key = (id(conv), conv.weight.device, self.conv_split_format)
        if key not in cache:
            w2d = conv.weight.detach().permute(2, 3, 1, 0).reshape(-1, conv.out_channels).t().contiguous()   # [Cout, 9*Cin]
            cache[key] = SplitLinearF16(w2d, act_scale=1.0) if self.conv_split_format == "fp16x2" else SplitLinear(w2d)
        return cache[key]

    def _igemm_weights(self, conv):
        """[3, Cout, 9*Cin] bf16: the pieces w1, w2, w3 of _split_weights' SplitLinear, K-major, for e2e_conv3x3_igemm."""
        cache = self.__dict__.setdefault("_split_cache", {})
        key = (id(conv), conv.weight.device, "igemm")
        if key not in cache:
            lin, k = self._split_weights(conv), 9 * conv.in_channels
            cache[key] = torch.stack([lin.b0.t(), lin.b1[:k].t(), lin.b2[:k].t()]).contiguous()
        return cache[key]

    def _conv_split(self, x, valid, conv, pool=False, amax_in=None, amax_out=None):
        """x [N,H,W,C] fp32 NHWC, valid [N] int32 -> relu(conv(x) + b) [N,H,W,Cout] NHWC, rows >= valid zeroed;
        with ``pool`` the 2x2 ceil-mode max pooling that follows is fused into the epilogue kernel.
        ``amax_in`` / ``amax_out`` (int32 [1] device words) select the fp16x2 format: the scale of this layer's
        operand comes from amax_in, the maximum of its output goes to amax_out."""
        from . import ops
        n, h, w, c = x.shape
        bias = conv.bias.detach().float().contiguous()
        if (amax_in is None and self.conv_path == "igemm" and conv.out_channels <= self.IGEMM_MAX_COUT
                and ops.conv3x3_igemm_supported(c, conv.out_channels)):
            return ops.conv3x3_igemm(x, valid, self._igemm_weights(conv), bias, "pool" if pool else "relu")
        k = 9 * c
        lin = self._split_weights(conv)
        total = n * h * w
        f16 = amax_in is not None
        pieces, a_dtype = (2, torch.float16) if f16 else (3, torch.bfloat16)
        blk = max(1, min(total, self.A_BYTES // (pieces * k * 2)))
        a = torch.empty((blk, pieces * k), dtype=a_dtype, device=x.device)
        y = torch.empty((total, conv.out_channels), dtype=torch.float32, device=x.device)
        for p0 in range(0, total, blk):
            m = min(blk, total - p0)
            ops.conv3x3_unfold_split(x, valid, p0, m, a, amax=amax_in)
            am, ym = a[:m], y[p0:p0 + m]
            if f16:
                torch.mm(am, lin.b1, out_dtype=torch.float32, out=ym)                      # a1w2 + a2w1
            else:
                torch.mm(am, lin.b2, out_dtype=torch.float32, out=ym)                      # a1w3 + a2w2 + a3w1
                torch.addmm(ym, am[:, :2 * k], lin.b1, out_dtype=torch.float32, out=ym)    # + a1w2 + a2w1
            torch.addmm(ym, am[:, :k], lin.b0, out_dtype=torch.float32, out=ym)            # + a1w1
        y = y.view(n, h, w, conv.out_channels)
        scale_args = (amax_in, lin.out_scale, amax_out) if f16 else ()
        if pool:
            return ops.conv_bias_relu_mask_pool(y, bias, valid, *scale_args)
        ops.conv_bias_relu_mask(y, bias, valid, *scale_args)
        return y

    def forward_masked_split(self, feat, feat_len):
        """forward_masked on the device path: the 4->128 layer is a direct kernel from the feature frames
        into NHWC, the three wide convolutions (128->128, 128->256, 256->256: 98 % of the front end's FLOPs)
        run on the tensor cores — unfold+split (csrc/conv_split.cu) -> three bf16 GEMMs with fp32
        accumulation -> bias/ReLU/mask(/2x2 max-pool) kernel — and the activations stay NHWC throughout."""
        from . import ops
        drop = feat.shape[1] % 4
        if drop:
            feat = feat[:, :-drop, :]
        if feat.stride(2) != 1 or feat.stride(1) != feat.shape[2]:
            feat = feat.contiguous()
        own = (feat_len // 4 * 4).to(feat.device)
        v1 = own.to(torch.int32).contiguous()
        v2 = (own // 2).to(torch.int32).contiguous()
        convs = [m for m in self.extractor if isinstance(m, nn.Conv2d)]
        w1 = convs[0].weight.detach().float().contiguous()
        f16 = self.conv_split_format == "fp16x2"
        # scale words (float bits of max|x|) of the inputs of conv2, conv3, conv4 and of the output, written on the device
        amax = torch.zeros(4, dtype=torch.int32, device=feat.device) if f16 else None
        word = lambda i: amax[i:i + 1] if f16 else None
        y = ops.conv1_direct(feat, w1, convs[0].bias.detach().float().contiguous(), v1, self.freq_dim, amax_out=word(0))   # [N,L,F,C1]
        y = self._conv_split(y, v1, convs[1], pool=True, amax_in=word(0), amax_out=word(1))   # rows >= own read as zero inside
        y = self._conv_split(y, v2, convs[2], amax_in=word(1), amax_out=word(2))
        y = self._conv_split(y, v2, convs[3], pool=True, amax_in=word(2), amax_out=word(3))   # [N, T/4, F/4, C2]
        out = y.permute(0, 1, 3, 2).contiguous()                                       # [N, T/4, C2, F/4]
        return out.view(out.shape[0], out.shape[1], self.out_dim), feat_len // 4


class RecurrentLayer(nn.Module):
    """(B)LSTM/GRU + optional LayerNorm/dropout/sub-sampling/projection (module.py:1003-1081)."""

    def __init__(self, input_dim, module, dim, bidirection, dropout, layer_norm, sample_rate, sample_style, proj):
        super().__init__()
        if sample_style not in ("drop", "concat"):
            raise ValueError("Unsupported Sample Style: " + sample_style)
        width = 2 * dim if bidirection else dim
        self.out_dim = sample_rate * width if (sample_rate > 1 and sample_style == "concat") else width
        self.sample_rate, self.sample_style = sample_rate, sample_style
        self.dropout, self.layer_norm, self.proj = dropout, layer_norm, proj
        self.layer = getattr(nn, module.upper())(input_dim, dim, bidirectional=bidirection, num_layers=1, batch_first=True)
        if layer_norm:
            self.ln = nn.LayerNorm(width)
        if dropout > 0:
            self.dp = nn.Dropout(p=dropout)
        if proj:
            self.pj = nn.Linear(width, width)

    def _post(self, out, x_len):
        if self.layer_norm:
            out = self.ln(out)
        if self.dropout > 0:
            out = self.dp(out)
        if self.sample_rate > 1:
            n, t, d = out.shape
            x_len = x_len // self.sample_rate
            if self.sample_style == "drop":
                out = out[:, ::self.sample_rate, :].contiguous()
            else:
                if t % self.sample_rate:
                    out = out[:, :-(t % self.sample_rate), :]
                out = out.contiguous().view(n, t // self.sample_rate, d * self.sample_rate)
        if self.proj:
            out = torch.tanh(self.pj(out))
        return out, x_len

    def forward(self, x, x_len):
        out, _ = self.layer(x)                      # reference runs the padded batch unpacked
        return self._post(out, x_len)

    def forward_ragged(self, x, x_len):
        """Zero-padded batch of utterances of different lengths, per-utterance results equal to
        batch-1 calls for every frame t < x_len — without packed sequences (cuDNN runs packed
        input one time step per kernel).  The forward direction of a padded row is already exact
        on its valid frames; the backward direction is run as a forward pass over each row
        reversed in place within its own length."""
        rnn = self.layer
        if not rnn.bidirectional:
            out, _ = rnn(x)
            return self._post(out, x_len)
        n, t, _ = x.shape
        fn = torch._VF.lstm if isinstance(rnn, nn.LSTM) else torch._VF.gru
        zeros = x.new_zeros(1, n, rnn.hidden_size)
        hx = (zeros, zeros) if isinstance(rnn, nn.LSTM) else zeros
        names = ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0")
        w_fw = [getattr(rnn, k) for k in names]
        w_bw = [getattr(rnn, k + "_reverse") for k in names]
        ar = torch.arange(t, device=x.device)[None, :]
        ln = x_len.to(x.device).clamp(min=1)[:, None]
        rev = torch.where(ar < ln, ln - 1 - ar, ar)                      # [n, t] own-length reversal, padding stays put
        gather = rev[:, :, None]
        fw = fn(x, hx, w_fw, True, 1, 0.0, False, False, True)[0]
        x_rev = x.gather(1, gather.expand(n, t, x.shape[2]))
        bw = fn(x_rev, hx, w_bw, True, 1, 0.0, False, False, True)[0]
        bw = bw.gather(1, gather.expand(n, t, bw.shape[2]))
        return self._post(torch.cat([fw, bw], dim=-1), x_len)


    # -- packed device path (CUDA only; SURVEY §8f row f-4) ----------------------------------------------
    def packed_supported(self):
        rnn = self.layer
        return (isinstance(rnn, (nn.LSTM, nn.GRU)) and rnn.num_layers == 1 and self.sample_rate == 1 and not self.layer_norm
                and rnn.hidden_size <= 384)

    def _packed_weights(self):
        from .stepper import SplitLinear
        rnn = self.layer
        cache = self.__dict__.setdefault("_packed_cache", {})
        key = rnn.weight_hh_l0.device
        if key not in cache:
            sfx = ["", "_reverse"] if rnn.bidirectional else [""]
            g = lambda n: getattr(rnn, n).detach().float()
            h = rnn.hidden_size
            w_in = torch.cat([g("weight_ih_l0" + x) for x in sfx], dim=0)                       # [dirs*4H (GRU: 3H), in]
            if isinstance(rnn, nn.LSTM):
                dirs = [((g("bias_ih_l0" + x) + g("bias_hh_l0" + x)).contiguous(),
                         g("weight_hh_l0" + x).view(4, h, h).permute(2, 1, 0).contiguous())
                        for x in sfx]                                                              # w_t [k][u][gate]
            else:
                # bias [b_ir+b_hr | b_iz+b_hz | b_in | b_hn]; w_t [k][u][r, z, n, 0] (csrc/lstm_seq.cu, GRU form)
                dirs = []
                for x in sfx:
                    b_ih, b_hh, w_hh = g("bias_ih_l0" + x), g("bias_hh_l0" + x), g("weight_hh_l0" + x).view(3, h, h)
                    bias = torch.cat([b_ih[:2 * h] + b_hh[:2 * h], b_ih[2 * h:], b_hh[2 * h:]]).contiguous()
                    w_t = torch.cat([w_hh, w_hh.new_zeros(1, h, h)]).permute(2, 1, 0).contiguous()
                    dirs.append((bias, w_t))
            pj = (SplitLinear(self.pj.weight.detach().float()), self.pj.bias.detach().float()) if self.proj else None
            cache[key] = (SplitLinear(w_in), dirs, pj)
        return cache[key]

    def forward_packed(self, x, frame_off, lens32, group_first, group_rows):
        """x [F, in]: the valid frames of all utterances back to back (utterance n at rows frame_off[n] ..
        + lens32[n]).  Input projections of both directions are one split-bf16 GEMM over all frames, the
        recurrence is one persistent kernel launch (csrc/lstm_seq.cu, LSTM or GRU form), the projection another GEMM."""
        from . import ops
        lin_in, dirs, pj = self._packed_weights()
        h = self.layer.hidden_size
        gru = isinstance(self.layer, nn.GRU)
        n_gates = 3 if gru else 4
        gates = split_gemm_rows(x.contiguous(), lin_in)                                          # [F, dirs*n_gates*H]
        out = torch.empty((x.shape[0], h * len(dirs)), dtype=torch.float32, device=x.device)
        fw = (dirs[0][0], dirs[0][1], 0, 0)
        bw = (dirs[1][0], dirs[1][1], n_gates * h, h) if len(dirs) == 2 else None
        (ops.gru_sequence if gru else ops.lstm_sequence)(gates, out, frame_off, lens32, group_first, group_rows, h, fw, bw)
        if pj is not None:
            out = torch.tanh(split_gemm_rows(out, pj[0]).add_(pj[1]))
        return out


class Encoder(nn.Module):
    """Listener (asr.py:390-476): optional VGG front end + recurrent stack."""

    def __init__(self, input_size, batch_size, vgg, vgg_freq, vgg_low_filt, module, bidirection, dim, dropout,
                 layer_norm, proj, sample_rate, sample_style):
        super().__init__()
        assert len(sample_rate) == len(dropout) == len(dim), "Number of layer mismatch"
        self.vgg, self.vgg_freq, self.vgg_low_filt = vgg, vgg_freq, vgg_low_filt
        self.sample_rate = 1
        stack, width = [], input_size
        if vgg == 1:
            stack.append(VGGFrontEnd(input_size))
            width = stack[-1].out_dim
            self.sample_rate *= 4
        elif vgg != 0:
            raise NotImplementedError("vgg = {} front end is outside the decode hot path scope".format(vgg))
        if module not in ("LSTM", "GRU"):
            raise NotImplementedError("encoder module " + str(module))
        for l in range(len(dim)):
            stack.append(RecurrentLayer(width, module, dim[l], bidirection, dropout[l], layer_norm[l],
                                        sample_rate[l], sample_style, proj[l]))
            width = stack[-1].out_dim
            self.sample_rate *= sample_rate[l]
        self.in_dim, self.out_dim = input_size, width
        self.layers = nn.ModuleList(stack)

    def forward(self, x, x_len):
        for layer in self.layers:
            x, x_len = layer(x, x_len)
        return x, x_len

    def packed_supported(self):
        return all(isinstance(l, VGGFrontEnd) or (isinstance(l, RecurrentLayer) and l.packed_supported()) for l in self.layers)

    @staticmethod
    def _groups(t_host):
        """CTA -> utterance grouping of the recurrent kernel: utterances arrive sorted by decreasing length;
        long ones get small groups so that the longest sequence does not set the run time."""
        first, rows, i, n = [], [], 0, len(t_host)
        while i < n:
            t = int(t_host[i])
            r = 4 if t >= 600 else (8 if t >= 300 else 16)
            r = min(r, n - i)
            first.append(i)
            rows.append(r)
            i += r
        return first, rows

    def forward_ragged_packed(self, x, x_len, chunk=128):
        """forward_ragged for a CUDA batch sorted by decreasing length: the front end runs in ``chunk``-utterance
        pieces cropped to their own longest utterance, the valid frames are PACKED back to back and the
        recurrent layers run over the packed frames (no padding is computed)."""
        lens_host = x_len.cpu()
        n_utts = x.shape[0]
        front = self.layers[0] if isinstance(self.layers[0], VGGFrontEnd) else None
        packs, tls = [], []
        ready = getattr(self, "chunk_ready", None)      # decode_batch_from_host: rows [lo, hi) have arrived from the host
        for lo in range(0, n_utts, chunk):
            hi = min(n_utts, lo + chunk)
            if ready is not None:
                ready(lo, hi)
            l_max = int(lens_host[lo:hi].max())
            xc, lc = x[lo:hi, :l_max], x_len[lo:hi]
            if front is not None:
                if getattr(self, "split_conv", False):
                    xc, lc = front.forward_masked_split(xc, lc)
                else:
                    xc, lc = front.forward_masked(xc, lc)
            lc = lc.to(x.device).reshape(-1)
            mask = torch.arange(xc.shape[1], device=x.device)[None, :] < lc[:, None]
            packs.append(xc[mask])                                      # utterance-major, time ascending
            tls.append(lc)
        feat = torch.cat(packs, dim=0)
        t_len = torch.cat(tls).long()
        t_host = t_len.cpu()
        frame_off = (torch.cumsum(t_len, 0) - t_len).to(torch.int32).contiguous()
        lens32 = t_len.to(torch.int32).contiguous()
        first, rows = self._groups(t_host)
        g_first = torch.tensor(first, dtype=torch.int32, device=x.device)
        g_rows = torch.tensor(rows, dtype=torch.int32, device=x.device)
        for layer in self.layers:
            if isinstance(layer, RecurrentLayer):
                feat = layer.forward_packed(feat, frame_off, lens32, g_first, g_rows)
        t_max = int(t_host.max())
        enc = feat.new_zeros((n_utts, t_max, feat.shape[1]))
        enc[torch.arange(t_max, device=x.device)[None, :] < t_len[:, None]] = feat
        return enc, t_len

    def forward_ragged(self, x, x_len):
        """Batched encode of zero-padded utterances of different lengths with
        per-utterance results equal (up to library kernel selection) to
        batch-1 calls: masked VGG + per-row reversed recurrent layers."""
        for layer in self.layers:
            if isinstance(layer, VGGFrontEnd):
                if getattr(self, "split_conv", False) and x.is_cuda:
                    x, x_len = layer.forward_masked_split(x, x_len)
                else:
                    x, x_len = layer.forward_masked(x, x_len)
            else:
                x, x_len = layer.forward_ragged(x, x_len)
        return x, x_len


class _AttentionCore(nn.Module):
    """Mask + temperature softmax + context (module.py:1084-1117)."""

    def __init__(self, temperature, num_head):
        super().__init__()
        self.temperature, self.num_head = temperature, num_head
        self.mask, self.k_len = None, None

    def reset_mem(self):
        self.mask, self.k_len = None, None

    def set_mem(self, prev_att):
        pass

    def compute_mask(self, k, k_len):
        self.k_len = k_len
        n, t, _ = k.shape
        pad = torch.arange(t, device=k_len.device)[None, :] >= k_len[:, None]
        self.mask = pad[:, None, :].expand(n, self.num_head, t).reshape(-1, t)

    def _attend(self, energy, value):
        score = (energy / self.temperature).masked_fill(self.mask, -np.inf)
        attn = torch.softmax(score, dim=-1)
        return torch.bmm(attn.unsqueeze(1), value).squeeze(1), attn


class ScaleDotAttention(_AttentionCore):
    def forward(self, q, k, v):
        energy = torch.bmm(q.unsqueeze(1), k.transpose(1, 2)).squeeze(1)
        out, attn = self._attend(energy, v)
        return out, attn.view(-1, self.num_head, k.shape[1])


class LocationAwareAttention(_AttentionCore):
    """energy = w^T tanh(key + query + U(F * prev_att))   (module.py:1135-1173)."""

    def __init__(self, kernel_size, kernel_num, dim, num_head, temperature):
        super().__init__(temperature, num_head)
        self.prev_att = None
        self.loc_conv = nn.Conv1d(num_head, kernel_num, kernel_size=2 * kernel_size + 1, padding=kernel_size, bias=False)
        self.loc_proj = nn.Linear(kernel_num, dim, bias=False)
        self.gen_energy = nn.Linear(dim, 1)
        self.dim = dim

    def reset_mem(self):
        super().reset_mem()
        self.prev_att = None

    def set_mem(self, prev_att):
        self.prev_att = prev_att

    def forward(self, q, k, v):
        nh, t, _ = k.shape
        n = nh // self.num_head
        if self.prev_att is None:                                   # uniform over the valid frames
            self.prev_att = torch.zeros((n, self.num_head, t), device=k.device)
            for i, sl in enumerate(self.k_len):
                self.prev_att[i, :, :sl] = 1.0 / sl
        loc = torch.tanh(self.loc_proj(self.loc_conv(self.prev_att).transpose(1, 2)))      # [n, t, dim]
        loc = loc.unsqueeze(1).repeat(1, self.num_head, 1, 1).view(-1, t, self.dim)
        energy = self.gen_energy(torch.tanh(k + q.unsqueeze(1) + loc)).squeeze(2)
        out, attn = self._attend(energy, v)
        attn = attn.view(n, self.num_head, t)
        self.prev_att = attn
        return out, attn


class Attention(nn.Module):
    """Query/key projections + attention core with cached keys (asr.py:273-364)."""

    def __init__(self, v_dim, q_dim, mode, dim, num_head, temperature, v_proj, loc_kernel_size, loc_kernel_num):
        super().__init__()
        self.v_dim, self.dim, self.mode, self.num_head, self.v_proj = v_dim, dim, mode.lower(), num_head, v_proj
        self.proj_q = nn.Linear(q_dim, dim * num_head)
        self.proj_k = nn.Linear(v_dim, dim * num_head)
        if v_proj:
            self.proj_v = nn.Linear(v_dim, v_dim * num_head)
        if self.mode == "dot":
            self.att_layer = ScaleDotAttention(temperature, num_head)
        elif self.mode == "loc":
            self.att_layer = LocationAwareAttention(loc_kernel_size, loc_kernel_num, dim, num_head, temperature)
        else:
            raise NotImplementedError
        if num_head > 1:
            self.merge_head = nn.Linear(v_dim * num_head, v_dim)
        self.key = self.value = self.mask = None

    def reset_mem(self):
        self.key = self.value = self.mask = None
        self.att_layer.reset_mem()

    def set_mem(self, prev_attn):
        self.att_layer.set_mem(prev_attn)

    def forward(self, dec_state, enc_feat, enc_len):
        n, t, _ = enc_feat.shape
        query = torch.tanh(self.proj_q(dec_state)).view(n * self.num_head, self.dim)
        if self.key is None:
            self.att_layer.compute_mask(enc_feat, enc_len.to(enc_feat.device))
            self.key = torch.tanh(self.proj_k(enc_feat))
            self.value = torch.tanh(self.proj_v(enc_feat)) if self.v_proj else enc_feat
            if self.num_head > 1:
                self.key = self.key.view(n, t, self.num_head, self.dim).permute(0, 2, 1, 3).contiguous().view(-1, t, self.dim)
                if self.v_proj:
                    self.value = self.value.view(n, t, self.num_head, self.v_dim).permute(0, 2, 1, 3).contiguous().view(-1, t, self.v_dim)
                else:
                    self.value = self.value.repeat(self.num_head, 1, 1)
        context, attn = self.att_layer(query, self.key, self.value)
        if self.num_head > 1:
            context = self.merge_head(context.view(n, self.num_head * self.v_dim))
        return attn, context


class Decoder(nn.Module):
    """Speller: RNN over [embedding ; context] + vocabulary projection (asr.py:183-270)."""

    def __init__(self, batch_size, input_dim, vocab_size, module, dim, layer, dropout):
        super().__init__()
        if module not in ("LSTM", "GRU"):
            raise NotImplementedError("decoder module " + str(module))
        self.in_dim, self.layer, self.dim, self.dropout = input_dim, layer, dim, dropout
        self.hidden_state = None
        self.enable_cell = module == "LSTM"
        self.layers = getattr(nn, module)(input_dim, dim, num_layers=layer, dropout=dropout, batch_first=True)
        self.char_trans = nn.Linear(dim, vocab_size)
        self.final_dropout = nn.Dropout(dropout)

    def init_state(self, bs):
        dev = next(self.parameters()).device
        z = lambda: torch.zeros((self.layer, bs, self.dim), device=dev)
        self.hidden_state = (z(), z()) if self.enable_cell else z()
        return self.get_state()

    def set_state(self, hidden_state):
        dev = next(self.parameters()).device
        if self.enable_cell:
            self.hidden_state = (hidden_state[0].to(dev), hidden_state[1].to(dev))
        else:
            self.hidden_state = hidden_state.to(dev)

    def get_state(self):
        if self.enable_cell:
            return (self.hidden_state[0].cpu(), self.hidden_state[1].cpu())
        return self.hidden_state.cpu()

    def get_query(self):
        h = self.hidden_state[0] if self.enable_cell else self.hidden_state
        return h.transpose(0, 1).reshape(-1, self.dim * self.layer)

    def forward(self, x):
        x, self.hidden_state = self.layers(x.unsqueeze(1), self.hidden_state)
        x = x.squeeze(1)
        return self.char_trans(self.final_dropout(x)), x


class ASR(nn.Module):
    """Joint CTC/attention model container (asr.py:13-64).  Only what decoding
    needs: the training ``forward`` of the reference is out of scope."""

    def __init__(self, input_size, vocab_size, batch_size, ctc_weight, encoder, attention, decoder,
                 emb_drop=0.0, init_adadelta=True):
        super().__init__()
        assert 0 <= ctc_weight <= 1
        self.vocab_size, self.ctc_weight = vocab_size, ctc_weight
        self.enable_ctc, self.enable_att = ctc_weight > 0, ctc_weight != 1
        self.lm = None
        self.encoder = Encoder(input_size, batch_size, **encoder)
        if self.enable_ctc:
            self.ctc_layer = nn.Sequential(nn.Linear(self.encoder.out_dim, vocab_size), nn.ReLU())   # asr.py:29-32
        if self.enable_att:
            self.dec_dim = decoder["dim"]
            self.pre_embed = nn.Embedding(vocab_size, self.dec_dim)
            self.embed_drop = nn.Dropout(emb_drop)
            self.decoder = Decoder(batch_size, self.encoder.out_dim + self.dec_dim, vocab_size, **decoder)
            self.attention = Attention(self.encoder.out_dim, self.dec_dim * self.decoder.layer, **attention)
        # asr.py:44-50: the reference always applies its own init + forget-gate bias 1
        self.apply(reference_init_)
        if self.enable_att and self.decoder.enable_cell:
            for l in range(self.decoder.layer):
                b = getattr(self.decoder.layers, "bias_ih_l{}".format(l))
                n = b.size(0)
                b.data[n // 4:n // 2].fill_(1.0)

    def set_state(self, prev_state, prev_attn):
        self.decoder.set_state(prev_state)
        self.attention.set_mem(prev_attn)

    def forward(self, *a, **k):
        raise NotImplementedError("training forward (asr.py:89-177) is outside the decode hot-path scope")


class RNNLM(nn.Module):
    """Embedding -> n-layer LSTM/GRU -> tied or separate output layer (lm.py:5-38)."""

    def __init__(self, vocab_size, emb_tying, emb_dim, module, dim, n_layers, dropout):
        super().__init__()
        self.dim, self.n_layers, self.emb_tying, self.vocab_size = dim, n_layers, emb_tying, vocab_size
        if emb_tying:
            assert emb_dim == dim, "Output dim of RNN should be identical to embedding if using weight tying."
        self.emb = nn.Embedding(vocab_size, emb_dim)
        self.dp1, self.dp2 = nn.Dropout(dropout), nn.Dropout(dropout)
        self.rnn = getattr(nn, module.upper())(emb_dim, dim, num_layers=n_layers, dropout=dropout, batch_first=True)
        if not emb_tying:
            self.trans = nn.Linear(emb_dim, vocab_size)

    def forward(self, x, lens, hidden=None):
        emb = self.dp1(self.emb(x))
        packed = nn.utils.rnn.pack_padded_sequence(emb, lens, batch_first=True, enforce_sorted=False)
        out, hidden = self.rnn(packed, hidden)
        out, _ = nn.utils.rnn.pad_packed_sequence(out, batch_first=True)
        out = F.linear(self.dp2(out), self.emb.weight) if self.emb_tying else self.trans(self.dp2(out))
        return out, hidden
