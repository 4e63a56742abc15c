"""Batched (utterance x beam) model step.

north_star keeps the dense contractions of the encoder, the attention decoder
step and the RNNLM step as library (cuBLAS) GEMMs.  The reference runs these
modules one hypothesis at a time on batch-1 tensors and bounces every state
through the CPU (src/decode.py:105-123,144-151,265-277); here the same arithmetic
runs once per decode step over all N = U*B hypotheses with device-resident states:

* attention  (src/asr.py:333-364, src/module.py:1152-1173 / :1120-1132)
* speller    (src/asr.py:259-266)
* RNNLM      (src/lm.py:27-38)

The stepper reads the weights straight out of the ``asr`` / ``lm`` modules it is
given (parameter names of the reference), so it works with the reference's own
objects as well as with ``model.py``.

On a GPU everything around the GEMMs is hand-written (SURVEY §8f rows f-1, f-2, f-4: csrc/attention_full.cu,
csrc/lstm_step.cu, csrc/conv_split.cu, csrc/lstm_seq.cu); on the CPU (host-logic tests only) the plain
PyTorch restatement below runs.  What keeps the step fast without leaving fp32:

* utterances arrive sorted by decreasing length, so the ones still decoding are
  always a PREFIX of the batch; every step only touches the first ``k`` of them;
* ``split_gemm``: the recurrent GEMMs ([N,2048]x[2048,4096] per LM layer) run on
  the tensor cores as a 3-way bf16 split of both operands (6 partial products
  a1w1+a1w2+a2w1+a1w3+a2w2+a3w1, fp32 accumulation, see SplitLinear).  x = a1+a2+a3
  is exact for fp32 inputs, the dropped products are below 2^-23 of |a||w|, so
  the result is as accurate as cuBLAS' fp32 SIMT GEMM (tests/test_gpu_decode.py
  checks it against fp64) at less than half its time;
* ``fused_attention``: the location-aware energies + masked softmax run in one
  hand-written kernel (csrc/attention_full.cu: location convolution, energies, masked
  softmax and the context product) instead of a cuDNN convolution, ~8 passes over
  [U*B, T, 300] temporaries and a batched GEMM, and never touches padded frames; multi-head models
  (attention.num_head = H <= 4) run the same kernel's multi-head form followed by merge_head, and fall back to
  a plain PyTorch multi-head step for what that kernel's shape query refuses (and for scaled-dot attention);
* the LSTM / GRU states are never permuted: a step reads them through the parents' row index
  (``_FusedLstm``), and the encoder runs over packed frames (``model.Encoder.forward_ragged_packed``).
"""
import numpy as np
import torch
import torch.nn.functional as F


def _split3(x):
    """fp32 -> three bf16 tensors with x == a1 + a2 + a3 (exactly, barring underflow)."""
    a1 = x.to(torch.bfloat16)
    r = x - a1.float()
    a2 = r.to(torch.bfloat16)
    a3 = (r - a2.float()).to(torch.bfloat16)
    return a1, a2, a3


class SplitLinear:
    """y = x @ W^T + b with fp32 accuracy on bf16 tensor cores.

    x = a1+a2+a3 and W = w1+w2+w3 (bf16 pieces).  The six partial products that matter are grouped
    by magnitude — {a1w1}, {a1w2, a2w1}, {a1w3, a2w2, a3w1} — one GEMM per group (pieces
    concatenated along K) accumulated smallest group first through the fp32 C operand, because a
    tensor-core accumulator that mixes magnitudes loses the small terms (measured: 2.8e-4 vs 4.4e-5
    max error on a 2048-long dot product; cuBLAS fp32 SIMT: 3.7e-5).  Small batches stay on the
    plain fp32 GEMM, where the split's extra passes do not pay."""

    MIN_ROWS = 1024

    def __init__(self, weight, bias=None):
        self.weight = weight.detach().float()
        self.bias = None if bias is None else bias.detach().float()
        w1, w2, w3 = _split3(self.weight)
        self.b0 = w1.t().contiguous()                                   # [K, M]
        self.b1 = torch.cat([w2, w1], dim=1).t().contiguous()           # [2K, M]
        self.b2 = torch.cat([w3, w2, w1], dim=1).t().contiguous()       # [3K, M]

    def __call__(self, x):
        if x.shape[0] < self.MIN_ROWS:
            return F.linear(x, self.weight, self.bias)
        a1, a2, a3 = _split3(x)
        y = torch.mm(torch.cat([a1, a2, a3], dim=1), self.b2, out_dtype=torch.float32)
        y = torch.addmm(y, torch.cat([a1, a2], dim=1), self.b1, out_dtype=torch.float32)
        y = torch.addmm(y, a1, self.b0, out_dtype=torch.float32)
        return y if self.bias is None else y + self.bias


F16_ACT_SCALE = 2.0 ** 14     # |h| <= 1 for an LSTM hidden state: scale*h stays far inside fp16's range (65504)


def _split2_f16(x, scale):
    """fp32 -> two fp16 tensors with scale*x == a1 + a2 up to 2^-22 |scale*x| (scale a power of two)."""
    xs = x * scale
    a1 = xs.to(torch.float16)
    a2 = (xs - a1.float()).to(torch.float16)
    return a1, a2


class SplitLinearF16:
    """y = x @ W^T on fp16 tensor cores from 2-piece splits: s_a*x = a1+a2, s_w*W = w1+w2 (22 mantissa bits each),
    three partial products grouped by magnitude — {a1w1}, {a1w2, a2w1} — smallest group first through the fp32 C
    operand, HALF the tensor-core work of SplitLinear's six.  Only for operands of known range (LSTM hidden states):
    fp16 has 5 exponent bits, so the scales must keep every piece that matters out of the subnormals and the largest
    below 65504.  s_w puts the largest |W| in [2^13, 2^14).  The product carries the factor s_a*s_w (``1/out_scale``),
    a power of two the cell kernel removes exactly.  Representation error of the operands: 2^-22 relative (bf16x3:
    2^-24), below the fp32 accumulation error of a K >= 1024 dot product (tests/test_host_logic.py checks the budget
    against float64)."""

    def __init__(self, weight, act_scale=F16_ACT_SCALE):
        w = weight.detach().float()
        w_max = float(w.abs().max())
        self.w_scale = 2.0 ** (13 - int(np.floor(np.log2(w_max)))) if w_max > 0 else 1.0
        w1, w2 = _split2_f16(w, self.w_scale)
        self.b0 = w1.t().contiguous()                                   # [K, M]
        self.b1 = torch.cat([w2, w1], dim=1).t().contiguous()           # [2K, M]:  [a1 | a2] @ [w2; w1]
        self.act_scale = float(act_scale)
        self.out_scale = 1.0 / (self.act_scale * self.w_scale)

    def __call__(self, x):
        a1, a2 = _split2_f16(x, self.act_scale)
        y = torch.mm(torch.cat([a1, a2], dim=1), self.b1, out_dtype=torch.float32)
        y = torch.addmm(y, a1, self.b0, out_dtype=torch.float32)
        return y * self.out_scale


class _Rnn:
    """n-layer LSTM/GRU advanced one token at a time for a batch of rows.  States are lists of
    per-layer [N, D] tensors so that row prefixes are contiguous views."""

    def __init__(self, rnn, split_gemm=False, first_input_table=None):
        self.is_lstm = isinstance(rnn, torch.nn.LSTM)
        if not self.is_lstm and not isinstance(rnn, torch.nn.GRU):
            raise NotImplementedError("only LSTM / GRU recurrent layers are supported")
        self.layers, self.dim = rnn.num_layers, rnn.hidden_size
        self.split = split_gemm and self.is_lstm
        self.w, self.fused, self.table0 = [], [], None
        for l in range(self.layers):
            w = tuple(getattr(rnn, "{}_l{}".format(k, l)) for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"))
            self.w.append(w)
            if not self.split:
                continue
            if l == 0 and first_input_table is not None:
                # layer 0 sees one of V embeddings: its input projection is a [V, 4D] table
                self.table0 = (first_input_table.double() @ w[0].double().t() + w[2].double()).float()
                self.fused.append(SplitLinear(w[1], w[3]))
            else:
                self.fused.append(SplitLinear(torch.cat([w[0], w[1]], dim=1), w[2] + w[3]))

    def zeros(self, n, device):
        z = lambda: [torch.zeros(n, self.dim, device=device) for _ in range(self.layers)]
        return (z(), z() if self.is_lstm else None)

    def step(self, x, state, n, tok=None):
        """x [n, in] (or token ids for a tabled layer 0), state rows [:n] are used."""
        h, c = state
        hs, cs = [], []
        for l in range(self.layers):
            hl = h[l][:n]
            if self.is_lstm:
                if self.split:
                    if l == 0 and self.table0 is not None:
                        gates = self.table0.index_select(0, tok) + self.fused[0](hl)
                    else:
                        gates = self.fused[l](torch.cat([x, hl], dim=1))
                else:
                    w_ih, w_hh, b_ih, b_hh = self.w[l]
                    gates = F.linear(x, w_ih, b_ih) + F.linear(hl, w_hh, b_hh)
                i, f, g, o = gates.chunk(4, dim=-1)
                c2 = torch.sigmoid(f) * c[l][:n] + torch.sigmoid(i) * torch.tanh(g)
                x = torch.sigmoid(o) * torch.tanh(c2)
                cs.append(c2)
            else:
                w_ih, w_hh, b_ih, b_hh = self.w[l]
                gi, gh = F.linear(x, w_ih, b_ih), F.linear(hl, w_hh, b_hh)
                ir, iz, inn = gi.chunk(3, dim=-1)
                hr, hz, hn = gh.chunk(3, dim=-1)
                r, z = torch.sigmoid(ir + hr), torch.sigmoid(iz + hz)
                x = (1 - z) * torch.tanh(inn + r * hn) + z * hl
            hs.append(x)
        return x, (hs, cs if self.is_lstm else None)

    @staticmethod
    def gather(state, idx):
        h, c = state
        return ([t.index_select(0, idx) for t in h], [t.index_select(0, idx) for t in c] if c is not None else None)


def _gru_blocks(w_ih, w_hh, b_ih, b_hh, emb=None):
    """One nn.GRU layer in the 4-block gate form [r | z | n_x | n_h] of e2e_gru_cell -> (weight, bias, table).
    Without ``emb``: weight [[W_ir, W_hr], [W_iz, W_hz], [W_in, 0], [0, W_hn]] against [x | h], bias
    [b_ir+b_hr | b_iz+b_hz | b_in | b_hn], table None.  With the V embeddings ``emb`` of a tabled layer 0: table
    [E W_ir^T + b_ir | E W_iz^T + b_iz | E W_in^T + b_in | 0] (computed in float64), weight [[W_hr], [W_hz], [0], [W_hn]]
    against h, bias [b_hr | b_hz | 0 | b_hn].  The zero blocks keep the n-gate products apart (n = tanh(n_x + r * n_h))
    in one GEMM chain per layer, at the tensor-core cost of an LSTM layer of the same width."""
    (w_ir, w_iz, w_in), (w_hr, w_hz, w_hn) = w_ih.chunk(3), w_hh.chunk(3)
    (b_ir, b_iz, b_in), (b_hr, b_hz, b_hn) = b_ih.chunk(3), b_hh.chunk(3)
    if emb is None:
        zi, zh = torch.zeros_like(w_in), torch.zeros_like(w_hn)
        weight = torch.cat([torch.cat([w_ir, w_hr], 1), torch.cat([w_iz, w_hz], 1), torch.cat([w_in, zh], 1), torch.cat([zi, w_hn], 1)])
        return weight, torch.cat([b_ir + b_hr, b_iz + b_hz, b_in, b_hn]), None
    proj = emb.double() @ w_ih.double().t() + b_ih.double()                               # [V, 3D]
    table = torch.cat([proj, proj.new_zeros(proj.shape[0], w_hh.shape[1])], 1).to(w_ih.dtype)
    return torch.cat([w_hr, w_hz, torch.zeros_like(w_hn), w_hn]), torch.cat([b_hr, b_hz, torch.zeros_like(b_hn), b_hn]), table


class _FusedLstm:
    """n-layer LSTM or GRU advanced one token at a time for a batch of rows, entirely on the device path
    (SURVEY §8f row f-2): per layer one hand-written split kernel, the three split GEMMs (library,
    tensor cores, fp32 accumulation) and one hand-written cell kernel (csrc/lstm_step.cu).  States
    are never permuted: a step reads the previous states through the parents' row index ``idx``
    and writes the new ones to the other half of a ping-pong buffer.  A GRU layer uses the same
    [n, 4D] accumulator through the 4-block gate form of ``_gru_blocks`` and has no c state.

    ``split`` selects the GEMM operand format: "bf16x3" (exact 3-piece bf16 split, six partial products, any operand
    range) or "fp16x2" (2-piece fp16 split, three partial products; needs a tabled layer 0 so that every GEMM input
    is a hidden state, |h| <= 1 — the RNNLM, src/lm.py:27-38)."""

    def __init__(self, rnn, first_input_table=None, split="bf16x3"):
        if not isinstance(rnn, (torch.nn.LSTM, torch.nn.GRU)):
            raise NotImplementedError("only LSTM / GRU recurrent layers are supported")
        self.gru = isinstance(rnn, torch.nn.GRU)
        if split not in ("bf16x3", "fp16x2"):
            raise ValueError("unknown split format " + str(split))
        if split == "fp16x2" and first_input_table is None:
            raise NotImplementedError("the fp16x2 operand format needs a tabled layer 0 (inputs of unknown range)")
        self.f16 = split == "fp16x2"
        make_lin = SplitLinearF16 if self.f16 else SplitLinear
        self.layers, self.dim = rnn.num_layers, rnn.hidden_size
        self.lin, self.bias, self.k_in, self.table0 = [], [], [], None
        for l in range(self.layers):
            w_ih, w_hh, b_ih, b_hh = (getattr(rnn, "{}_l{}".format(k, l)).detach().float()
                                      for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"))
            tabled = l == 0 and first_input_table is not None
            if self.gru:
                weight, bias, table = _gru_blocks(w_ih, w_hh, b_ih, b_hh, first_input_table if tabled else None)
                if tabled:
                    self.table0 = table.contiguous()
                self.lin.append(make_lin(weight))
                self.bias.append(bias.contiguous())
                self.k_in.append(0 if tabled else w_ih.shape[1])
            elif tabled:
                # layer 0 sees one of V embeddings: its input projection is a [V, 4D] table
                self.table0 = (first_input_table.double() @ w_ih.double().t() + b_ih.double()).float().contiguous()
                self.lin.append(make_lin(w_hh))
                self.bias.append(b_hh.contiguous())
                self.k_in.append(0)
            else:
                self.lin.append(make_lin(torch.cat([w_ih, w_hh], dim=1)))
                self.bias.append((b_ih + b_hh).contiguous())
                self.k_in.append(w_ih.shape[1])
        self.cur = 0

    # Rows (live utterances x beam) up to which a step is REPLAYED FROM A CUDA GRAPH: below ~500 live utterances a decode step
    # is bound by the host's launch rate (tools/profile_tail.py: the last 360 steps of the bench take 215 ms of host time for
    # 215 ms of device time), and the LSTM stacks are 23 of a step's ~48 launches.  Row counts are rounded up to a ladder so
    # that a graph is reused while the live count shrinks; the padding rows belong to finished utterances and are never read.
    GRAPH_MAX_ROWS = 4096
    GRAPH_LADDER = (64, 128, 256, 384, 512, 768, 1024, 1536, 2048, 2560, 3072, 3584, 4096)
    use_graphs = False

    def start(self, n, device):
        d = self.dim
        if getattr(self, "cap", 0) >= n and getattr(self, "device", None) == device:
            # same buffers as the last decode (and the graphs captured over them): only the initial states are reset
            for l in range(self.layers):
                self.h[0][l][:n].zero_()
                if self.c is not None:
                    self.c[0][l][:n].zero_()
            self.idx = self.idx_buf[:n]
            self.idx_buf.copy_(self._arange)
            self.cur = 0
            return
        self.cap, self.device, self.graphs = n, device, {}
        self.h = [[torch.zeros(n, d, device=device) for _ in range(self.layers)] for _ in range(2)]
        self.c = None if self.gru else [[torch.zeros(n, d, device=device) for _ in range(self.layers)] for _ in range(2)]
        pieces, a_dtype = (2, torch.float16) if self.f16 else (3, torch.bfloat16)
        self.a = [torch.empty(n, pieces * (self.k_in[l] + d), dtype=a_dtype, device=device) for l in range(self.layers)]
        self.gates = torch.empty(n, 4 * d, device=device)          # GEMM accumulator, reused by every layer
        # static homes of a step's varying inputs (what a captured graph reads): parent rows, tokens, layer-0 input
        self._arange = torch.arange(n, device=device)
        self.idx_buf = self._arange.clone()
        self.tok_buf = torch.zeros(n, dtype=torch.int64, device=device)
        self.x0_buf = torch.zeros(n, self.k_in[0], device=device) if self.k_in[0] > 0 else None
        self.idx = self.idx_buf[:n]
        self.cur = 0
        from . import ops
        vec = d % 4 == 0 and all(k % 4 == 0 for k in self.k_in)
        self.scale = F16_ACT_SCALE if self.f16 else None
        self.plans = [ops.SplitPlan([(self.h[c][l], self.a[l], self.k_in[l] + d, self.k_in[l]) for l in range(self.layers)], self.scale)
                      if (vec and self.layers <= 8) else None for c in range(2)]

    def hidden(self, n):
        """[n, layers*D] hidden states of the rows' parents (what Decoder.get_query reads, asr.py:251-254)."""
        hs = [h.index_select(0, self.idx[:n]) for h in self.h[self.cur]]
        return hs[0] if len(hs) == 1 else torch.cat(hs, dim=1)

    def x0_home(self, n):
        """Where the caller may build the layer-0 input of the next step directly (the static buffer a graph reads)."""
        return self.x0_buf[:n] if (self.x0_buf is not None and self._graph_rows(n)) else None

    def _graph_rows(self, n):
        if not self.use_graphs or n > self.GRAPH_MAX_ROWS or torch.cuda.is_current_stream_capturing():
            return 0
        for r in self.GRAPH_LADDER:
            if n <= r:
                return min(r, self.cap)
        return 0

    def step(self, n, x0=None, tok=None):
        """Advance rows [:n]; x0 [n, in] fp32 (or tok [n] for a tabled layer 0) -> top hidden [n, D]."""
        nr = self._graph_rows(n)
        if nr == 0:
            return self._step_eager(n, x0, tok, self.idx)
        # stage the step's varying inputs in their static buffers, then replay the graph of (padded rows, ping-pong parity)
        from . import ops
        if self.idx.data_ptr() != self.idx_buf.data_ptr():
            self.idx_buf[:n].copy_(self.idx[:n])
        if tok is not None and self.table0 is not None:
            self.tok_buf[:n].copy_(tok[:n])
        if x0 is not None and x0.data_ptr() != self.x0_buf.data_ptr():
            self.x0_buf[:n].copy_(x0)
        key = (nr, self.cur)
        g = self.graphs.get(key)
        if g is None:
            cur = self.cur
            body = lambda: self._step_eager(nr, self.x0_buf[:nr] if self.x0_buf is not None else None, self.tok_buf[:nr], self.idx_buf)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):            # once for real on a side stream (library handles / workspaces), as torch asks
                body()
            torch.cuda.current_stream().wait_stream(side)
            self.cur = cur
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                body()
            self.cur = cur
            self.graphs[key] = g
        g.replay()
        ops.add_launch_count(1 + (1 if self.k_in[0] > 0 else 0) + self.layers)      # the library's own kernels inside the graph
        self.cur = 1 - self.cur
        return self.h[self.cur][self.layers - 1][:n]

    def _step_eager(self, n, x0, tok, idx):
        from . import ops
        cur, new, d = self.cur, 1 - self.cur, self.dim
        if self.plans[cur] is not None:                                # recurrent halves of all A operands, one launch
            self.plans[cur].run(idx, n)
        else:
            for l in range(self.layers):
                ops.lstm_split_rows(self.h[cur][l], idx, n, self.a[l], self.k_in[l] + d, self.k_in[l], self.scale)
        if self.k_in[0] > 0:
            ops.lstm_split_rows(x0.contiguous(), None, n, self.a[0], self.k_in[0] + d, 0)
        for l in range(self.layers):
            k = self.k_in[l] + d
            a, lin = self.a[l][:n], self.lin[l]
            y = self.gates[:n]                                         # accumulate in place: no C-operand copies
            if self.f16:
                torch.mm(a, lin.b1, out_dtype=torch.float32, out=y)
            else:
                torch.mm(a, lin.b2, out_dtype=torch.float32, out=y)
                torch.addmm(y, a[:, :2 * k], lin.b1, out_dtype=torch.float32, out=y)
            torch.addmm(y, a[:, :k], lin.b0, out_dtype=torch.float32, out=y)
            nxt = l + 1 < self.layers
            tail = dict(table=self.table0 if l == 0 else None, tok=tok if (l == 0 and self.table0 is not None) else None,
                        a_next=self.a[l + 1] if nxt else None, k_next=(self.k_in[l + 1] + d) if nxt else 0, off_next=0,
                        gate_scale=lin.out_scale if self.f16 else None, next_scale=self.scale)
            if self.gru:
                ops.gru_cell(y, self.bias[l], self.h[cur][l], idx, n, self.h[new][l], **tail)
            else:
                ops.lstm_cell(y, self.bias[l], self.c[cur][l], idx, n, self.c[new][l], self.h[new][l], **tail)
        self.cur = new
        return self.h[new][self.layers - 1][:n]

    def reorder(self, idx):
        self.idx = idx


class EmbFusion:
    """The per-step operands of the word-embedding fusion plug-in (src/plugin.py EmbeddingRegularizer), read from the
    module by the reference's parameter names, so the reference's own object works as well as model.py's.  What does
    not change during a decode is prepared once: the row-normalised table (``fuse_normalize``), ``scale`` = relu(temp)
    and ``lam``, the mixing weight (sigmoid of a learnable one).  :meth:`logits` is x_emb @ table^T of the speller's
    top-layer output: two library GEMMs and a ReLU for emb_net, then the table product (fp32: the decode loop runs under
    decode._Fp32Math)."""

    def __init__(self, emb):
        with torch.no_grad():
            lin0, lin2 = emb.emb_net[0], emb.emb_net[2]
            self.w0, self.b0 = lin0.weight.detach(), lin0.bias.detach()
            self.w2, self.b2 = lin2.weight.detach(), lin2.bias.detach()
            table = emb.emb_table.weight.detach()
            self.normalize = bool(emb.fuse_normalize)
            self.table = (F.normalize(table, dim=-1) if self.normalize else table).contiguous()
            self.scale = F.relu(emb.temp.detach()).float().contiguous()
            lam = emb.fuse_lambda.detach()
            self.lam = (torch.sigmoid(lam) if emb.fuse_learnable else lam).float().contiguous()
            self.eps = float(emb.eps)

    def logits(self, top):
        """top [n, D] -> emb_logits [n, V]."""
        x = F.linear(F.relu(F.linear(top, self.w0, self.b0)), self.w2, self.b2)
        if self.normalize:
            x = F.normalize(x, dim=-1)
        return F.linear(x, self.table)


ATT_MAX_SLOTS = 32      # beam slots per utterance the fused attention kernels take (kAfMaxB, csrc/attention_full.cu)


def attention_groups(beam):
    """The beam slots [lo, hi) of each fused attention call: one group up to ATT_MAX_SLOTS, else the fewest groups of
    near-equal size (beam 40: 20 + 20, beam 64: 32 + 32)."""
    n = -(-beam // ATT_MAX_SLOTS)
    size = -(-beam // n)
    return [(lo, min(beam, lo + size)) for lo in range(0, beam, size)]


class BatchedStepper:
    def __init__(self, asr, lm=None, split_gemm=False, fused_attention=False, lm_split="bf16x3", vgg_split="bf16x3", step_graphs=False,
                 vgg_conv="igemm", emb=None):
        att = asr.attention
        # the word-embedding fusion plug-in (None: off); step() then also returns its logits
        self.emb = EmbFusion(emb) if emb is not None else None
        if att.mode not in ("loc", "dot"):
            raise NotImplementedError("attention mode " + str(att.mode))
        self.asr, self.lm = asr, lm
        self.split_conv = bool(split_gemm)       # VGG convolutions as fp32-accurate tensor-core GEMMs (model.py)
        if vgg_split not in ("bf16x3", "fp16x2"):
            raise ValueError("unknown split format " + str(vgg_split))
        self.vgg_split = vgg_split               # their operand format
        if vgg_conv not in ("igemm", "unfold"):
            raise ValueError("unknown VGG convolution path " + str(vgg_conv))
        self.vgg_conv = vgg_conv                 # and kernel path (model.VGGFrontEnd.conv_path)
        self.mode, self.temperature = att.mode, att.att_layer.temperature
        self.H = att.num_head
        # fused device LSTM / GRU steps (csrc/lstm_step.cu) whenever the weights live on a GPU; the plain
        # PyTorch cells otherwise (CPU tests of the host logic, split_gemm = False)
        def make(rnn, table=None, split="bf16x3"):
            on_gpu = next(rnn.parameters()).is_cuda
            if split_gemm and on_gpu and isinstance(rnn, (torch.nn.LSTM, torch.nn.GRU)):
                return _FusedLstm(rnn, table, split)
            return _Rnn(rnn, split_gemm, table)
        self.dec = make(asr.decoder.layers)                  # speller inputs (embedding, context) have no fixed range: bf16x3
        self.lm_rnn = make(lm.rnn, lm.emb.weight.detach(), lm_split) if lm is not None else None
        for stack in (self.dec, self.lm_rnn):
            if isinstance(stack, _FusedLstm):
                stack.use_graphs = bool(step_graphs)
        self.mark = lambda name: None            # profiling hook (decode.py sets it)
        # fused_attention: the location-aware step may run csrc/attention_full.cu; with several heads whether it does is
        # decided per decode (start(): the kernel's own size query for the beam), and ``fused_step`` records it
        self.fused_attention = self.fused_step = False
        if fused_attention and self.mode == "loc":
            lay = att.att_layer
            if lay.loc_proj.weight.shape[1] <= 12 and lay.loc_proj.weight.shape[0] % 4 == 0:
                self.fused_attention = True
                w_conv = lay.loc_conv.weight.detach()                                     # [K, H, 2P+1]
                self._w_conv = w_conv[:, 0, :].contiguous() if self.H == 1 else w_conv.contiguous()
                self._w_proj = lay.loc_proj.weight.detach().contiguous()
                self._w_energy = lay.gen_energy.weight.detach().reshape(-1).contiguous()
                self._b_energy = float(lay.gen_energy.bias.detach().reshape(-1)[0])

    # -- once per batch ---------------------------------------------------------------------
    def encode(self, feats, lens, chunk=128):
        """feats [U,Lmax,D] zero padded, lens [U] -> enc [U,Tmax,E], enc_len [U] (long, same device).
        The batch is encoded ``chunk`` utterances at a time, each chunk cropped to its own longest
        utterance: with the batch sorted by length this removes most of the padding work."""
        enc_mod = self.asr.encoder
        n_utts = feats.shape[0]
        for layer in getattr(enc_mod, "layers", []):
            if hasattr(layer, "conv_split_format"):
                layer.conv_split_format = self.vgg_split
                layer.conv_path = self.vgg_conv
        packed = (n_utts > 1 and self.split_conv and feats.is_cuda and hasattr(enc_mod, "forward_ragged_packed")
                  and enc_mod.packed_supported())
        ready = getattr(enc_mod, "chunk_ready", None)
        if ready is not None and not packed:
            ready(0, n_utts)                      # features still arriving from the host (decode_batch_from_host): only the
                                                  # packed path below consumes them chunk by chunk
        if n_utts == 1:
            # one utterance: the plain module call, on the valid frames only — zero padding would otherwise reach the
            # backward LSTM direction (the reference's batch-1 call is never padded, bin/test_asr.py:159-167)
            enc, enc_len = enc_mod(feats[:, :int(lens[0])], lens)
        elif packed:
            # device path: split convolutions, packed frames, persistent recurrent kernel (model.py)
            enc_mod.split_conv = True
            enc, enc_len = enc_mod.forward_ragged_packed(feats, lens, chunk)
        elif hasattr(enc_mod, "forward_ragged"):
            enc_mod.split_conv = self.split_conv and feats.is_cuda
            lens_host = lens.cpu()
            outs, ls = [], []
            for lo in range(0, n_utts, chunk):
                hi = min(n_utts, lo + chunk)
                l_max = int(lens_host[lo:hi].max())
                e, l = enc_mod.forward_ragged(feats[lo:hi, :l_max], lens[lo:hi])
                outs.append(e)
                ls.append(l.reshape(-1))
            t_all = max(e.shape[1] for e in outs)
            enc = feats.new_zeros((n_utts, t_all, outs[0].shape[2]))
            lo = 0
            for e in outs:
                enc[lo:lo + e.shape[0], :e.shape[1]] = e
                lo += e.shape[0]
            enc_len = torch.cat(ls)
        else:   # opaque encoder (e.g. the reference's own module): one exact batch-1 call per utterance
            outs, ls = [], []
            for i in range(n_utts):
                n = int(lens[i])
                e, l = enc_mod(feats[i:i + 1, :n], lens[i:i + 1])
                outs.append(e[0])
                ls.append(l.reshape(-1)[0])
            enc = torch.nn.utils.rnn.pad_sequence(outs, batch_first=True)
            enc_len = torch.stack(ls)
        enc_len = enc_len.to(enc.device).long().clamp(max=enc.shape[1])
        t_max = int(enc_len.max())
        if n_utts > 1:
            t_max = (t_max + 3) // 4 * 4          # 16-byte aligned alignment rows for the attention kernel; the extra frames are masked
        if t_max > enc.shape[1]:
            enc = torch.nn.functional.pad(enc, (0, 0, 0, t_max - enc.shape[1]))
        return enc[:, :t_max].contiguous(), enc_len

    def start(self, enc, enc_len, beam):
        att = self.asr.attention
        u, t, _ = enc.shape
        self.U, self.B, self.T, self.N = u, beam, t, u * beam
        self._groups = attention_groups(beam)
        dev = enc.device
        if self.H == 1:
            self.fused_step = self.fused_attention
            self.key = torch.tanh(att.proj_k(enc))                               # [U,T,A]   asr.py:343
            if self.fused_attention:
                self.key_t = self.key.transpose(1, 2).contiguous()               # [U,A,T] channel-major for the fused kernel
                self.key = None
            self.value = torch.tanh(att.proj_v(enc)) if att.v_proj else enc      # [U,T,E]
        else:
            self._start_heads(enc, beam)
        self.pad = torch.arange(t, device=dev)[None, :] >= enc_len[:, None]      # [U,T]     module.py:1100-1107
        if self.mode == "loc":
            uni = (1.0 / enc_len.to(torch.float32))[:, None].expand(u, t).masked_fill(self.pad, 0.0)   # module.py:1157-1160
            if self.H == 1:
                self.prev_att = uni[:, None, :].expand(u, beam, t).reshape(self.N, t).contiguous()
            else:                                                                # [N,H,T]: every head starts uniform
                self.prev_att = uni[:, None, None, :].expand(u, beam, self.H, t).reshape(self.N, self.H, t).contiguous()
        else:
            self.prev_att = None
        self.dec_fused = isinstance(self.dec, _FusedLstm)
        self.lm_fused = isinstance(self.lm_rnn, _FusedLstm)
        if self.dec_fused:
            self.dec.start(self.N, dev)
        else:
            self.dec_state = self.dec.zeros(self.N, dev)
        if self.lm_fused:
            self.lm_rnn.start(self.N, dev)
        else:
            self.lm_state = self.lm_rnn.zeros(self.N, dev) if self.lm_rnn is not None else None
        self._enc_len32 = enc_len.to(torch.int32).contiguous()

    def _start_heads(self, enc, beam):
        """Keys and values of H > 1 heads.  Every head of a hypothesis attends ITS OWN utterance's encoder output: the
        batch-1 meaning of model.Attention (at batch > 1 its ``value.repeat(num_head, 1, 1)`` would pair heads with other
        utterances' values, which the per-hypothesis decode never does)."""
        att, h = self.asr.attention, self.H
        u, t, _ = enc.shape
        key = torch.tanh(att.proj_k(enc)).view(u, t, h, -1)                      # [U,T,H,A]  asr.py:343
        self.fused_step = False
        if self.fused_attention and enc.is_cuda:
            from . import ops
            k_filt, _, width = self._w_conv.shape
            widest = max(hi - lo for lo, hi in self._groups)
            self.fused_step = ops.attention_loc_heads_supported(widest, h, key.shape[3], k_filt, width)
        value = torch.tanh(att.proj_v(enc)) if att.v_proj else enc               # [U,T,H*E] or [U,T,E]
        if self.fused_step:
            self.key_t, self.key = key.permute(0, 2, 3, 1).contiguous(), None    # [U,H,A,T] channel-major per head
            self.value = value                                                   # the kernel reads head h's columns in place
        else:
            self.key = key.permute(0, 2, 1, 3).contiguous()                      # [U,H,T,A]
            self.value = value.view(u, t, h, -1).permute(0, 2, 1, 3).contiguous() if att.v_proj else value   # [U,H,T,E]

    def _attend(self, query, k):
        """The attention step of the first k utterances: query [k*B, H*A] -> (alignments, context [k*B, E])."""
        att = self.asr.attention
        b, t = self.B, self.T
        n = k * b
        if self.H > 1:
            attn, context = self._attend_heads(query, k)
        elif self.mode == "loc" and self.fused_attention:
            from . import ops
            # conv + energies + masked softmax + context in one kernel (csrc/attention_full.cu)
            attn, context = self._fused_attention(ops.attention_loc_full, query, k)
        else:
            if self.mode == "loc":
                lay = att.att_layer
                loc = lay.loc_conv(self.prev_att[:n, None, :]).transpose(1, 2)         # [n,T,K]
                loc = torch.tanh(lay.loc_proj(loc)).view(k, b, t, -1)
                mix = torch.tanh(self.key[:k, None] + query.view(k, b, 1, -1) + loc)
                energy = lay.gen_energy(mix).squeeze(-1)                               # [k,B,T]  module.py:1168
            else:
                energy = torch.bmm(query.view(k, b, -1), self.key[:k].transpose(1, 2))  # module.py:1126
            score = (energy / self.temperature).masked_fill(self.pad[:k, None, :], -np.inf)
            attn = torch.softmax(score, dim=-1)                                        # [k,B,T]
            context = torch.bmm(attn, self.value[:k]).view(n, -1)                      # module.py:1114
        return attn, context

    def _fused_attention(self, fn, query, k, *per_head_values):
        """ops.attention_loc_full / attention_loc_heads for the first k utterances, once per group of beam slots
        (self._groups).  The kernels take at most ATT_MAX_SLOTS slots per utterance and their results do not depend on how
        slots are grouped, so a wider beam runs group by group: each group's query and previous-alignment rows are made
        contiguous, and its alignments and contexts are scattered back into beam order."""
        b = self.B
        args = (self.key_t, self.value)
        tail = (self._enc_len32, self._w_conv, self._w_proj, self._w_energy, self._b_energy, self.temperature)
        if len(self._groups) == 1:
            return fn(*args, query.contiguous(), self.prev_att, *tail, b, *per_head_values, n_run=k)
        n = k * b
        q = query.view(k, b, -1)
        prev = self.prev_att[:n].view(k, b, *self.prev_att.shape[1:])
        attn = ctx = None
        for lo, hi in self._groups:
            g = hi - lo
            a, c = fn(*args, q[:, lo:hi].reshape(k * g, -1), prev[:, lo:hi].reshape(k * g, *prev.shape[2:]), *tail, g,
                      *per_head_values, n_run=k)
            if attn is None:
                attn = a.new_empty((k, b) + tuple(a.shape[1:]))
                ctx = c.new_empty((k, b) + tuple(c.shape[1:]))
            attn[:, lo:hi] = a.view(k, g, *a.shape[1:])
            ctx[:, lo:hi] = c.view(k, g, *c.shape[1:])
        return attn.view(n, *attn.shape[2:]), ctx.view(n, -1)

    def _attend_heads(self, query, k):
        """One attention step of H > 1 heads for the first k utterances: (alignments [k*B,H,T], merge_head(context))."""
        att, h = self.asr.attention, self.H
        b, t = self.B, self.T
        n = k * b
        if self.fused_step:
            from . import ops
            # conv over the H alignments + energies + masked softmax + per-head contexts in one kernel (csrc/attention_full.cu)
            attn, ctx = self._fused_attention(ops.attention_loc_heads, query, k, att.v_proj)
        else:
            q = query.view(k, b, h, -1)
            if self.mode == "loc":
                lay = att.att_layer
                loc = torch.tanh(lay.loc_proj(lay.loc_conv(self.prev_att[:n]).transpose(1, 2))).view(k, b, t, -1)   # shared by the heads
                # one head at a time: the temporaries stay the size of the single-head step's
                energy = torch.stack([lay.gen_energy(torch.tanh(self.key[:k, j, None] + q[:, :, j, None, :] + loc)).squeeze(-1)
                                      for j in range(h)], dim=2)                 # [k,B,H,T]
            else:
                energy = torch.matmul(q.transpose(1, 2), self.key[:k].transpose(2, 3)).transpose(1, 2)          # [k,B,H,T]
            score = (energy / self.temperature).masked_fill(self.pad[:k, None, None, :], -np.inf)
            attn = torch.softmax(score, dim=-1)                                  # [k,B,H,T]
            if att.v_proj:
                ctx = torch.matmul(attn.transpose(1, 2), self.value[:k]).transpose(1, 2)                          # [k,B,H,E]
            else:
                ctx = torch.bmm(attn.reshape(k, b * h, t), self.value[:k])       # [k,B*H,E]
            attn, ctx = attn.reshape(n, h, t), ctx.reshape(n, -1)
        return attn, F.linear(ctx, att.merge_head.weight, att.merge_head.bias)   # merge_head: [n,H*E] -> [n,E]

    # -- once per decode step ---------------------------------------------------------------
    def step(self, prev_tok, k=None):
        """Advance the first ``k`` utterances (all by default).  prev_tok [k*B] long ->
        (att_logits [k*B,V], lm_logits [k*B,V] | None), and emb_logits [k*B,V] third when the stepper has an
        embedding-fusion plug-in; the new states are held until :meth:`reorder` commits them in the surviving
        hypotheses' order."""
        asr, att = self.asr, self.asr.attention
        k = self.U if k is None else k
        b, t = self.B, self.T
        n = k * b
        self._k = k
        dec_h = self.dec.hidden(n) if self.dec_fused else torch.cat([h[:n] for h in self.dec_state[0]], dim=1)
        query = torch.tanh(att.proj_q(dec_h))                                              # asr.py:337 / :251-254
        attn, context = self._attend(query, k)
        self.mark("step_attention")
        if self.dec_fused:
            home = self.dec.x0_home(n)                                             # decode.py:114-115
            dec_in = torch.cat([asr.pre_embed(prev_tok), context], dim=-1, out=home) if home is not None else \
                torch.cat([asr.pre_embed(prev_tok), context], dim=-1)
            top = self.dec.step(n, x0=dec_in)
        else:
            dec_in = torch.cat([asr.pre_embed(prev_tok), context], dim=-1)
            top, self._new_dec = self.dec.step(dec_in, self.dec_state, n)
        att_logits = asr.decoder.char_trans(top)                                   # asr.py:265
        emb_logits = self.emb.logits(top) if self.emb is not None else None       # plugin.py fuse_prob, from d_state = top
        self._new_att = (attn.view(n, t) if self.H == 1 else attn) if self.mode == "loc" else None
        self.mark("step_speller")
        lm_logits = None
        if self.lm is not None:
            x0 = None if self.lm_rnn.table0 is not None else self.lm.emb(prev_tok)
            if self.lm_fused:
                top = self.lm_rnn.step(n, x0=x0, tok=prev_tok)
            else:
                top, self._new_lm = self.lm_rnn.step(x0, self.lm_state, n, tok=prev_tok)
            lm_logits = F.linear(top, self.lm.emb.weight) if self.lm.emb_tying else self.lm.trans(top)   # lm.py:33-37
            self.mark("step_lm")
        out = att_logits.contiguous(), (lm_logits.contiguous() if lm_logits is not None else None)
        return out if emb_logits is None else out + (emb_logits.contiguous(),)

    def reorder(self, parent_row):
        """parent_row [U,B] int64 (row u*B + slot of each survivor's parent, written by e2e_beam_combine_prune):
        children inherit the post-step states of their parent (decode.py:159-162,250-257).  Only the rows of
        the utterances advanced by the last :meth:`step` are touched."""
        k = self._k
        idx = parent_row[:k].view(-1)
        if self.dec_fused:
            self.dec.reorder(idx)
        else:
            self.dec_state = _Rnn.gather(self._new_dec, idx)
        if self._new_att is not None:
            self.prev_att = self._new_att.index_select(0, idx)
        if self.lm is not None:
            if self.lm_fused:
                self.lm_rnn.reorder(idx)
            else:
                self.lm_state = _Rnn.gather(self._new_lm, idx)
