"""GRU decode path, host side (no GPU): the 4-block gate form [r | z | n_x | n_h] that the fused stepper builds for an
nn.GRU layer reproduces nn.GRU, the cell's fp32 operation order is nn.GRU's on the CPU bit for bit, and the new C entry
points refuse bad arguments before touching a device."""
import ctypes

import pytest
import torch
import torch.nn.functional as F


def _cell64(weight, bias, table, x, h):
    """The 4-block GEMM + e2e_gru_cell in float64: z = [x | h] W^T + b (+ table row), the kernel's cell order."""
    a = h if x is None else torch.cat([x, h], dim=1)
    z = a @ weight.t() + bias
    if table is not None:
        z = z + table
    zr, zz, znx, znh = z.chunk(4, dim=1)
    r, u = torch.sigmoid(zr), torch.sigmoid(zz)
    n = torch.tanh(znx + r * znh)
    return (h - n) * u + n


@pytest.mark.parametrize("in_dim,d,layers", [(24, 16, 2), (40, 12, 3)])
def test_gate_blocks_reproduce_nn_gru_in_float64(in_dim, d, layers):
    from e2e_asr_pytorch_b200.stepper import _gru_blocks
    torch.manual_seed(in_dim)
    rnn = torch.nn.GRU(in_dim, d, num_layers=layers, batch_first=True).double()
    for p in rnn.parameters():
        p.data.normal_(0, 0.5)
    n = 9
    x = torch.randn(n, in_dim, dtype=torch.float64)
    h0 = torch.randn(layers, n, d, dtype=torch.float64).tanh()
    with torch.no_grad():
        out, hn = rnn(x[:, None], h0)
        inp = x
        for l in range(layers):
            w = [getattr(rnn, "%s_l%d" % (k, l)) for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
            weight, bias, table = _gru_blocks(*w)
            assert weight.shape == (4 * d, w[0].shape[1] + d) and table is None
            inp = _cell64(weight, bias, None, inp, h0[l])
            assert (inp - hn[l]).abs().max().item() < 1e-12
    assert (inp - out[:, 0]).abs().max().item() < 1e-12


def test_tabled_gate_blocks_reproduce_nn_gru_in_float64():
    from e2e_asr_pytorch_b200.stepper import _gru_blocks
    torch.manual_seed(1)
    d, vocab = 16, 11
    rnn = torch.nn.GRU(d, d, num_layers=1, batch_first=True).double()
    for p in rnn.parameters():
        p.data.normal_(0, 0.5)
    emb = torch.randn(vocab, d, dtype=torch.float64)
    tok = torch.randint(0, vocab, (13,))
    h0 = torch.randn(1, 13, d, dtype=torch.float64).tanh()
    with torch.no_grad():
        _, hn = rnn(emb[tok][:, None], h0)
        weight, bias, table = _gru_blocks(rnn.weight_ih_l0, rnn.weight_hh_l0, rnn.bias_ih_l0, rnn.bias_hh_l0, emb)
    assert weight.shape == (4 * d, d) and table.shape == (vocab, 4 * d)
    assert (table[:, 3 * d:] == 0).all() and (bias[2 * d:3 * d] == 0).all()
    got = _cell64(weight, bias, table[tok], None, h0[0])
    assert (got - hn[0]).abs().max().item() < 1e-12


def test_fused_stack_holds_the_gate_blocks():
    """What _FusedLstm keeps for a GRU stack (CPU construction: weights, biases, layer-0 table) is _gru_blocks' form."""
    from e2e_asr_pytorch_b200.stepper import _FusedLstm, _gru_blocks
    torch.manual_seed(2)
    d, vocab = 8, 5
    rnn = torch.nn.GRU(d, d, num_layers=2, batch_first=True)
    emb = torch.randn(vocab, d)
    for table in (None, emb):
        fused = _FusedLstm(rnn, table)
        assert fused.gru
        for l in range(2):
            w = [getattr(rnn, "%s_l%d" % (k, l)).detach() for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
            weight, bias, tab = _gru_blocks(*w, emb=table if l == 0 else None)
            assert torch.equal(fused.lin[l].weight, weight)
            assert torch.equal(fused.bias[l], bias)
            assert fused.k_in[l] == (0 if (l == 0 and table is not None) else d)
            if l == 0 and table is not None:
                assert torch.equal(fused.table0, tab)
        assert (fused.table0 is None) == (table is None)
    f16 = _FusedLstm(rnn, emb, split="fp16x2")
    assert f16.f16 and f16.gru


@pytest.mark.parametrize("n,in_dim,d", [(7, 20, 16), (64, 300, 1024), (33, 1324, 300)])
def test_cell_order_is_bit_equal_to_nn_gru_on_the_cpu(n, in_dim, d):
    """Given nn.GRU's own gate activations, h' = (h - n) * u + n with n = tanh(n_x + r * n_h), each op rounded in fp32,
    is nn.GRU's step bit for bit; the textbook (1 - u) * n + u * h is not.  (The activations are taken the way ATen takes
    them, in place on the chunks of the gate tensors: torch's CPU sigmoid of a strided view and of a contiguous copy can
    differ in the last bit, which is a property of that sigmoid, not of the order.)"""
    torch.manual_seed(d)
    rnn = torch.nn.GRU(in_dim, d, batch_first=True)
    x = torch.randn(n, in_dim)
    h = torch.randn(n, d).tanh()
    with torch.no_grad():
        _, want = rnn(x[:, None], h[None])
        gi = F.linear(x, rnn.weight_ih_l0, rnn.bias_ih_l0)
        gh = F.linear(h, rnn.weight_hh_l0, rnn.bias_hh_l0)
    (ir, iz, inn), (hr, hz, hn) = gi.chunk(3, 1), gh.chunk(3, 1)
    r, u = hr.add_(ir).sigmoid_(), hz.add_(iz).sigmoid_()
    nn_ = inn.add(hn.mul_(r)).tanh_()
    assert torch.equal((h - nn_) * u + nn_, want[0])
    if d == 1024:
        assert not torch.equal((1 - u) * nn_ + u * h, want[0])


def test_gru_entry_points_reject_bad_arguments_without_a_device():
    from e2e_asr_pytorch_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)                      # a non-null, aligned "device pointer" that is never dereferenced
    # e2e_gru_cell(gates, pitch, bias, table, tok, h_prev, idx, n, D, h_new, a_next, a_pitch, K_next, off_next, stream)
    assert lib.e2e_gru_cell(None, 16, fake, None, None, fake, None, 1, 4, fake, None, 0, 0, 0, None) == -1
    assert b"e2e_gru_cell" in lib.e2e_last_error()
    assert lib.e2e_gru_cell(fake, 16, fake, fake, None, fake, None, 1, 4, fake, None, 0, 0, 0, None) == -1   # table without tok
    assert lib.e2e_gru_cell(fake, 12, fake, None, None, fake, None, 1, 4, fake, None, 0, 0, 0, None) == -1   # pitch < 4D
    assert lib.e2e_gru_cell(fake, 16, fake, None, None, fake, None, 0, 4, fake, None, 0, 0, 0, None) == -1   # no rows
    assert lib.e2e_gru_cell(fake, 16, fake, None, None, fake, None, 1, 4, fake, fake, 8, 4, 0, None) == -1   # bf16 needs 3K
    assert b"next-layer" in lib.e2e_last_error()
    assert lib.e2e_gru_cell_f16x2(fake, 16, 0.75, fake, None, None, fake, None, 1, 4, fake, None, 0, 0, 0, 1.0, None) == -1
    assert b"powers of two" in lib.e2e_last_error()
    assert lib.e2e_gru_cell_f16x2(fake, 16, 1.0, fake, None, None, fake, None, 1, 4, fake, fake, 8, 4, 0, 3.0, None) == -1
    # e2e_gru_sequence(gates, pitch, out, out_pitch, frame_off, lens, g_first, g_rows, N, H, n_groups, n_dirs, fw..., bw..., stream)
    seq = lambda pitch, h, dirs, w_bw=fake: lib.e2e_gru_sequence(fake, pitch, fake, 2 * h, fake, fake, fake, fake, 1, h, 1, dirs,
                                                                 fake, fake, 0, 0, fake, w_bw, 3 * h, h, None)
    assert seq(16, 8, 2, w_bw=None) == -1                                  # backward weights missing
    assert b"e2e_gru_sequence" in lib.e2e_last_error()
    assert seq(23, 8, 1) == -1                                             # pitch < 3H
    assert seq(48, 8, 3) == -1                                             # 1 or 2 directions
    assert seq(3 * 400, 400, 1) == -3                                      # H > 384
    assert b"hidden size" in lib.e2e_last_error()
