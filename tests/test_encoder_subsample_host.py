"""Encoder sub-sampling and LayerNorm on the packed device path, host side (no GPU): the frame counts P (frames that
exist) and X (the reported x_len) that model.subsample_lengths carries through the stack are the ones batch-1 calls of
RecurrentLayer produce, which layers take the packed path, the argument checks of e2e_packed_subsample_ln, and the
decode memory estimate's time reduction."""
import ctypes
import itertools

import pytest
import torch


def _layer(in_dim, rate, style, h=2, module="LSTM", layer_norm=False, proj=False, bidirection=True):
    from e2e_asr_pytorch_b200.model import RecurrentLayer
    torch.manual_seed(0)
    return RecurrentLayer(in_dim, module, h, bidirection, 0.0, layer_norm, rate, style, proj).eval()


@pytest.mark.parametrize("style", ["drop", "concat"])
@pytest.mark.parametrize("rate", [2, 3])
def test_subsample_lengths_match_batch1_layer_calls(style, rate):
    """For every input length 1..40, P' is the number of rows a batch-1 call returns and X' its x_len; a length that the
    layer leaves without frames (concat, P < r) makes subsample_lengths raise, naming the utterance."""
    from e2e_asr_pytorch_b200.model import subsample_lengths
    layer = _layer(3, rate, style)
    with torch.no_grad():
        for t in range(1, 41):
            out, x_len = layer(torch.randn(1, t, 3), torch.tensor([t]))
            if out.shape[1] == 0:
                with pytest.raises(ValueError, match="utterance 0"):
                    subsample_lengths(torch.tensor([t]), torch.tensor([t]), rate, style)
                continue
            p2, x2 = subsample_lengths(torch.tensor([t]), torch.tensor([t]), rate, style)
            assert (int(p2[0]), int(x2[0])) == (out.shape[1], int(x_len[0])), (t, style, rate)


@pytest.mark.parametrize("style", ["drop", "concat"])
@pytest.mark.parametrize("rates", [(2, 2), (2, 3), (3, 2), (1, 2), (2, 1)])
def test_subsample_lengths_follow_a_chain_of_two_layers(style, rates):
    """Two stacked layers: the second walks the P' frames of the first (P' > X' after a 'drop' of an odd P), and the
    pair of counts after both is what the two batch-1 calls give."""
    from e2e_asr_pytorch_b200.model import subsample_lengths
    l1 = _layer(3, rates[0], style)
    l2 = _layer(l1.out_dim, rates[1], style)
    lens = torch.arange(1, 41)
    with torch.no_grad():
        for t in range(1, 41):
            h, xl = l1(torch.randn(1, t, 3), torch.tensor([t]))
            if h.shape[1] == 0:
                continue
            h, xl = l2(h, xl)
            p, x = subsample_lengths(torch.tensor([t]), torch.tensor([t]), rates[0], style)
            if h.shape[1] == 0:
                with pytest.raises(ValueError):
                    subsample_lengths(p, x, rates[1], style)
                continue
            p, x = subsample_lengths(p, x, rates[1], style)
            assert (int(p[0]), int(x[0])) == (h.shape[1], int(xl[0])), (t, style, rates)
    if style == "drop":
        p, x = subsample_lengths(lens, lens, rates[0], style)
        p, x = subsample_lengths(p, x, rates[1], style)
        assert (p >= x).all() and (p > x).any()


def test_subsample_lengths_names_the_empty_utterance():
    from e2e_asr_pytorch_b200.model import subsample_lengths
    with pytest.raises(ValueError, match="utterance 2"):
        subsample_lengths(torch.tensor([9, 4, 1, 1]), torch.tensor([9, 4, 1, 1]), 2, "concat")
    p, x = subsample_lengths(torch.tensor([9, 4, 1]), torch.tensor([9, 4, 1]), 2, "drop")
    assert p.tolist() == [5, 2, 1] and x.tolist() == [4, 2, 0]
    p, x = subsample_lengths(torch.tensor([7]), torch.tensor([7]), 1, "concat")
    assert p.tolist() == [7] and x.tolist() == [7]


def test_packed_supported_truth_table():
    """Sub-sampling (drop or concat, any rate) and LayerNorm take the packed path for LSTM and GRU layers with one or two
    directions; hidden sizes above 384 do not."""
    for module, bidir, rate, style, ln, proj in itertools.product(["LSTM", "GRU"], [True, False], [1, 2, 3], ["drop", "concat"],
                                                                  [False, True], [False, True]):
        assert _layer(4, rate, style, module=module, layer_norm=ln, proj=proj, bidirection=bidir).packed_supported()
    assert _layer(4, 1, "drop", h=384).packed_supported()
    assert not _layer(4, 2, "drop", h=385, layer_norm=True).packed_supported()
    from e2e_asr_pytorch_b200 import synth
    import copy
    for enc in ({"vgg": 0, "sample_rate": [1, 2], "sample_style": "drop"},
                {"sample_rate": [2, 1], "sample_style": "concat", "layer_norm": [True, True], "proj": [False, False]}):
        cfg = copy.deepcopy(synth.TINY_ASR_CFG)
        cfg["encoder"].update(enc)
        assert synth.build_asr(31, cfg).encoder.packed_supported()


def test_post_entry_point_rejects_bad_arguments_without_a_device():
    from e2e_asr_pytorch_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)                      # a non-null, aligned "device pointer" that is never dereferenced
    # e2e_packed_subsample_ln(in, in_pitch, out, out_pitch, in_off, out_off, out_len, N, W, stride, g, w, b, eps, stream)
    call = lambda **k: lib.e2e_packed_subsample_ln(*[k.get(n, d) for n, d in (
        ("src", fake), ("in_pitch", 640), ("out", fake), ("out_pitch", 1280), ("in_off", fake), ("out_off", fake),
        ("out_len", fake), ("n", 3), ("w", 640), ("stride", 2), ("g", 2), ("lw", fake), ("lb", fake), ("eps", 1e-5),
        ("stream", None))])
    for ptr in ("src", "out", "in_off", "out_off", "out_len"):
        assert call(**{ptr: None}) == -1, ptr
        assert b"null pointer" in lib.e2e_last_error()
    assert call(lw=None) == -1                                             # a bias without its weight
    assert call(n=0) == -1 and call(n=-2) == -1
    assert b"bad size" in lib.e2e_last_error()
    assert call(w=0) == -1 and call(stride=0) == -1
    assert call(g=3) == -1 and call(stride=3, g=2) == -1                   # g must be 1 or the stride
    assert call(in_pitch=639) == -1
    assert b"bad pitch" in lib.e2e_last_error()
    assert call(out_pitch=1279) == -1                                      # concat rows are g*W wide
    assert call(eps=0.0) == -1
    assert b"e2e_packed_subsample_ln" in lib.e2e_last_error()


def test_post_wrapper_has_no_cpu_path():
    from e2e_asr_pytorch_b200 import ops, _lib
    x = torch.zeros(6, 8)
    idx = torch.zeros(2, dtype=torch.int32)
    with pytest.raises(_lib.E2EError):
        ops.packed_subsample_ln(x, idx, idx, idx, 3, stride=2)
    with pytest.raises(_lib.E2EError):
        ops.packed_subsample_ln(x, idx, idx, idx, 3, stride=2, g=2, weight=torch.ones(8), bias=torch.zeros(8))


def test_decode_estimate_follows_the_time_reduction():
    """The default (4x: the VGG front end) is the estimate as it was; a 2x encoder sizes its buffers for twice the frames."""
    from e2e_asr_pytorch_b200 import shard
    assert shard.estimate_decode_bytes(2620, 3300, 31, 8, 12) == 67404331174
    assert shard.estimate_decode_bytes(300, 1000, 10000, 4, 0, num_head=2) == 23774980838
    args = (2620, 3300, 31, 8, 12)
    assert shard.estimate_decode_bytes(*args, time_reduction=4) == shard.estimate_decode_bytes(*args)
    assert shard.estimate_decode_bytes(*args, time_reduction=2) > shard.estimate_decode_bytes(*args)


def test_decode_estimate_holds_the_packed_first_layer_of_a_subsampling_encoder():
    """Without a front end the first recurrent layer runs over every input frame of the batch: its gates alone are
    U x l_max x 4*enc_dim fp32, which the estimate must hold whatever the output frame rate."""
    from e2e_asr_pytorch_b200 import shard
    u, l_max, enc_dim = 4096, 3300, 640
    gates = u * l_max * 4 * enc_dim * 4
    est = shard.estimate_decode_bytes(u, l_max, 31, 8, 12, time_reduction=2, front_reduction=1)
    assert est > gates + shard.estimate_decode_bytes(u, l_max, 31, 8, 12, time_reduction=2, front_reduction=2)
    # VGG + concat by 2: the first layer still runs at l_max / 4
    vgg8 = shard.estimate_decode_bytes(u, l_max, 31, 8, 12, time_reduction=8)
    assert vgg8 > u * (l_max // 4) * 4 * enc_dim * 4


def test_split_row_limit_matches_the_split_kernel():
    """model.SPLIT_MAX_ROWS is the row count e2e_lstm_split_rows refuses beyond (checked before any launch)."""
    from e2e_asr_pytorch_b200 import _lib
    from e2e_asr_pytorch_b200.model import SPLIT_MAX_ROWS
    lib = _lib.load()
    fake = ctypes.c_void_p(256)
    # e2e_lstm_split_rows(src, src_pitch, row_idx, n, w, dst, dst_pitch, K, off, stream)
    assert lib.e2e_lstm_split_rows(fake, 8, None, SPLIT_MAX_ROWS + 1, 8, fake, 24, 8, 0, None) == -3
    assert b"too many rows" in lib.e2e_last_error()
