"""Sub-sampling and LayerNorm encoder layers on the packed device path (B200): the post-processing kernel
(csrc/encoder_post.cu) against float64 LayerNorm and plain gathers, packed layers and whole encoders against batch-1
float64 module calls, and decodes of models with such encoders against the per-hypothesis oracle."""
import copy

import pytest
import torch
import torch.nn.functional as F

from tests.test_gpu_decode import _compare, _models, _oracle_nbest
from tests.test_gpu_kernels import copy_double

pytestmark = pytest.mark.gpu

LENS = [40, 33, 17, 9, 5, 4, 3, 2, 1] + [12 - (k % 5) for k in range(16)]       # 25 utterances, odd lengths, 1..3


def _ops():
    from e2e_asr_pytorch_b200 import ops, _lib
    return ops, _lib


def _randomize(module, seed):
    """Biases N(0, 0.3) as in the other packed tests; LayerNorm weight 1 + N(0, 0.1) and bias N(0, 0.1) (the reference's
    init zeroes every 1-D parameter, which would make a LayerNorm layer output zeros)."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in module.named_parameters():
            if "bias" in name and ".ln." not in "." + name:
                p.copy_(torch.randn(p.shape, generator=g) * 0.3)
        for m in module.modules():
            if isinstance(m, torch.nn.LayerNorm):
                m.weight.copy_(1 + torch.randn(m.weight.shape, generator=g) * 0.1)
                m.bias.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)


@pytest.mark.parametrize("ln", [False, True])
@pytest.mark.parametrize("style,rate", [("drop", 2), ("drop", 3), ("concat", 2), ("concat", 3), ("none", 1)])
@pytest.mark.parametrize("width", [32, 640, 768, 16, 320, 384])
def test_post_kernel_matches_gather_and_float64_layer_norm(cuda, ln, style, rate, width):
    """e2e_packed_subsample_ln over 25 ragged utterances (lengths 1, 2, 3 and odd ones; 'concat' leaves the short ones
    without rows): a plain gather is a bit-exact copy, with LayerNorm every row is within 5e-6 of float64 F.layer_norm of
    the gathered frame."""
    ops, _ = _ops()
    g = torch.Generator().manual_seed(width + rate)
    lens = torch.tensor(LENS)
    x = torch.randn(int(lens.sum()), width, generator=g) * 0.7 + 0.2
    w = 1 + torch.randn(width, generator=g) * 0.1
    b = torch.randn(width, generator=g) * 0.1
    out_len = (lens + rate - 1) // rate if style == "drop" else lens // rate
    gw = rate if style == "concat" else 1
    in_off = torch.cumsum(lens, 0) - lens
    out_off = torch.cumsum(out_len, 0) - out_len
    i32 = lambda t: t.to(torch.int32).to(cuda)
    got = ops.packed_subsample_ln(x.to(cuda), i32(in_off), i32(out_off), i32(out_len), int(out_len.sum()), stride=rate, g=gw,
                                  weight=w.to(cuda) if ln else None, bias=b.to(cuda) if ln else None, eps=1e-5).cpu()
    assert got.shape == (int(out_len.sum()), gw * width)
    src = torch.cat([in_off[n] + torch.arange(int(out_len[n]))[:, None] * rate + torch.arange(gw)[None, :]
                     for n in range(len(lens))]).reshape(-1)
    rows = x[src]
    if not ln:
        assert torch.equal(got, rows.reshape(-1, gw * width))
        return
    want = F.layer_norm(rows.double(), (width,), w.double(), b.double(), 1e-5).reshape(-1, gw * width)
    err = (got.double() - want).abs().max().item()
    assert err < 5e-6, err


def _layer(module, in_dim, h, rate, style, ln, proj, seed):
    from e2e_asr_pytorch_b200.model import RecurrentLayer, reference_init_
    torch.manual_seed(seed)
    layer = RecurrentLayer(in_dim, module, h, True, 0.0, ln, rate, style, proj)
    layer.apply(reference_init_)
    _randomize(layer, seed)
    return layer.eval()


LAYER_CASES = [(s, ln, m, pj) for s in ("drop", "concat") for ln in (False, True) for m in ("LSTM", "GRU")
               for pj in (False, True) if not (s == "concat" and pj)]     # a projection after 'concat' is no valid layer


@pytest.mark.parametrize("hidden,in_dim,rate,lens", [(16, 24, 2, [31, 22, 21, 9, 4, 3]), (320, 64, 2, [71, 41] + [33 - (k % 2) for k in range(20)]),
                                                     (16, 12, 3, [40, 29, 7, 3])])
@pytest.mark.parametrize("style,ln,module,proj", LAYER_CASES)
def test_packed_subsampling_layer_matches_float64(cuda, style, ln, module, proj, hidden, in_dim, rate, lens):
    """RecurrentLayer.forward_packed with sub-sampling (recurrence -> LayerNorm / drop / concat -> projection) vs the
    layer's own batch-1 forward in float64 on every row it returns (odd P included, so 'drop' keeps P' > X' rows)."""
    _ops()
    from e2e_asr_pytorch_b200.model import Encoder, subsample_lengths, packed_offsets
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    layer = _layer(module, in_dim, hidden, rate, style, ln, proj, hidden + rate)
    assert layer.packed_supported()
    g = torch.Generator().manual_seed(1)
    xs = [torch.randn(l, in_dim, generator=g) for l in lens]
    t_len = torch.tensor(lens)
    p2, x2 = subsample_lengths(t_len, t_len, rate, style)
    with torch.no_grad():
        ref = copy_double(layer)
        outs = [ref(x[None].double(), torch.tensor([x.shape[0]])) for x in xs]
        assert [o.shape[1] for o, _ in outs] == p2.tolist() and [int(l[0]) for _, l in outs] == x2.tolist()
        want = torch.cat([o[0] for o, _ in outs], dim=0)
        layer.to(cuda)
        off, lens32 = packed_offsets(t_len, cuda)
        first, rows = Encoder._groups(t_len)
        with _Fp32Math():
            got = layer.forward_packed(torch.cat(xs).to(cuda), off, lens32, torch.tensor(first, dtype=torch.int32, device=cuda),
                                       torch.tensor(rows, dtype=torch.int32, device=cuda), out_lens=p2)
    assert got.shape == want.shape
    err = (got.cpu().double() - want).abs().max().item()
    print("packed %s %s r=%d ln %s proj %s H=%d: max |gpu - fp64| = %.3g" % (module, style, rate, ln, proj, hidden, err))
    assert err < 5e-6


def test_layer_norm_only_layer_matches_float64(cuda):
    """LayerNorm without sub-sampling needs no output lengths: the post kernel keeps the recurrence's packing."""
    _ops()
    from e2e_asr_pytorch_b200.model import Encoder, packed_offsets
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    layer = _layer("LSTM", 20, 16, 1, "drop", True, True, 5)
    lens = [30, 22, 9, 1]
    g = torch.Generator().manual_seed(2)
    xs = [torch.randn(l, 20, generator=g) for l in lens]
    with torch.no_grad():
        ref = copy_double(layer)
        want = torch.cat([ref(x[None].double(), torch.tensor([x.shape[0]]))[0][0] for x in xs], dim=0)
        layer.to(cuda)
        t_len = torch.tensor(lens)
        off, lens32 = packed_offsets(t_len, cuda)
        first, rows = Encoder._groups(t_len)
        with _Fp32Math():
            got = layer.forward_packed(torch.cat(xs).to(cuda), off, lens32, torch.tensor(first, dtype=torch.int32, device=cuda),
                                       torch.tensor(rows, dtype=torch.int32, device=cuda))
    assert (got.cpu().double() - want).abs().max().item() < 5e-6


def test_split_gemm_takes_more_rows_than_one_split_launch(cuda):
    """An encoder without a front end projects every feature frame of the batch in one split_gemm_rows call (1.91 M frames
    of 160 bins for the 2620 dev-clean lengths): the rows go through the split kernel in blocks it accepts."""
    _ops()
    from e2e_asr_pytorch_b200.model import SPLIT_MAX_ROWS, split_gemm_rows
    from e2e_asr_pytorch_b200.stepper import SplitLinear
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    g = torch.Generator().manual_seed(4)
    x = torch.randn(SPLIT_MAX_ROWS + 1000, 8, generator=g)
    w = torch.randn(12, 8, generator=g)
    with torch.no_grad(), _Fp32Math():
        y = split_gemm_rows(x.to(cuda), SplitLinear(w.to(cuda))).cpu()
    assert (y.double() - x.double() @ w.double().t()).abs().max().item() < 1e-5


ENCODERS = {
    # config/librispeech_asr.yaml's structure: no VGG, the second layer drops every other frame
    "yaml_encoder": ({"vgg": 0, "sample_rate": [1, 2], "sample_style": "drop"}, [97, 92, 64, 41, 40, 13, 3]),
    # tests/test_oracle_vs_reference.py's concat_ln variant: VGG, frame concatenation, LayerNorm, no projection
    "concat_ln": ({"sample_rate": [2, 1], "sample_style": "concat", "layer_norm": [True, True], "proj": [False, False]},
                  [96, 92, 68, 44, 40, 12, 8]),
    "drop_2_2": ({"vgg": 0, "sample_rate": [2, 2], "sample_style": "drop"}, [97, 91, 66, 43, 40, 13, 2]),
}


def _asr(variant, peak=1.0):
    from e2e_asr_pytorch_b200 import synth
    cfg = copy.deepcopy(synth.TINY_ASR_CFG)
    cfg["encoder"].update(ENCODERS[variant][0])
    asr = synth.build_asr(31, cfg, seed=0, peak=peak)
    _randomize(asr.encoder, 7)
    return asr


@pytest.mark.parametrize("variant", sorted(ENCODERS))
def test_packed_subsampling_encoder_matches_batch1_calls(cuda, variant):
    """Encoder.forward_ragged_packed vs one batch-1 float64 Encoder call per utterance: rows [0, X) within 5e-6, enc_len
    == X, zeros beyond (odd lengths included, so a 'drop' layer walks P > X frames in the next layer).  Behind the VGG
    front end the bound is 4e-5: the front end's fp32-accurate split GEMMs sum in another order than the CPU, and a
    LayerNorm with no projection after it divides that difference by the standard deviation of its row.  Measured on a
    B200 for concat_ln: 3.4e-6 .. 1.8e-5 per utterance, against 1.6e-5 .. 2.9e-5 for the route this replaces
    (forward_ragged: the same front end, cuDNN layers), which is printed beside it (DESIGN.md §6.5)."""
    _ops()
    from e2e_asr_pytorch_b200 import synth
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    asr = _asr(variant)
    enc = asr.encoder
    lens = ENCODERS[variant][1]
    feat, fl = synth.padded_batch(list(range(len(lens))), lens)
    with torch.no_grad():
        ref = copy_double(enc)
        wants = [ref(feat[i:i + 1, :n].double(), fl[i:i + 1]) for i, n in enumerate(lens)]
        enc.to(cuda)
        enc.split_conv = True
        assert enc.packed_supported()
        with _Fp32Math():
            got, gl = enc.forward_ragged_packed(feat.to(cuda), fl.to(cuda), chunk=4)
            rag = enc.forward_ragged(feat.to(cuda), fl.to(cuda))[0] if enc.vgg else None
    assert gl.cpu().tolist() == [int(l[0]) for _, l in wants]
    assert got.shape[1] == max(int(l[0]) for _, l in wants)
    for i, (w, l) in enumerate(wants):
        x = int(l[0])
        err = (got[i, :x].cpu().double() - w[0, :x]).abs().max().item() if x else 0.0
        err_rag = (rag[i, :x].cpu().double() - w[0, :x]).abs().max().item() if x and rag is not None else 0.0
        print("%s utt %d: max |packed - fp64| = %.3g" % (variant, i, err)
              + (", max |forward_ragged - fp64| = %.3g" % err_rag if rag is not None else ""))
        assert err < (4e-5 if enc.vgg else 5e-6), (variant, i, err, err_rag)
        assert (got[i, x:] == 0).all()


def test_empty_utterance_is_refused_before_any_launch(cuda):
    from e2e_asr_pytorch_b200 import synth, ops
    asr = _asr("concat_ln").to(cuda)
    enc = asr.encoder
    enc.split_conv = True
    feat, fl = synth.padded_batch([0, 1], [40, 4])               # 4 frames -> 1 after the front end -> none after concat by 2
    before = ops.launch_count()
    with pytest.raises(ValueError, match="utterance 1"):
        enc.forward_ragged_packed(feat.to(cuda), fl.to(cuda))
    assert ops.launch_count() == before


@pytest.mark.parametrize("variant", ["yaml_encoder", "concat_ln"])
@pytest.mark.parametrize("beam,lm_w,ctc_w", [(1, 0.0, 0.0), (1, 0.3, 0.5), (4, 0.3, 0.5), (4, 0.0, 0.0), (8, 0.5, 0.5), (8, 0.0, 0.5)])
def test_subsampling_encoder_decode_matches_oracle(cuda, variant, beam, lm_w, ctc_w):
    """Models with the shipped encoder structure and with the concat + LayerNorm encoder decode through the packed
    encoder (forward_ragged is made to raise) to the oracle's 1-best, or a tie by its own scores, for all but at most
    one utterance.  The lengths keep P = X at every 'drop' layer: the oracle scores CTC over P frames, the device over X.
    The concat model reduces time 8x, so its hypotheses are capped at a twentieth of the input length, about half its
    encoder frames, as the usual fifth is for a 4x model (longer ones leave CTC no alignment, and the reference's search
    raises, src/decode.py:252, src/ctc.py:85)."""
    from e2e_asr_pytorch_b200 import BeamDecoder, synth
    asr = _asr(variant, peak=4.0)
    ratio = 0.2 if asr.encoder.sample_rate <= 4 else 0.05
    _, lm, lm_path, lm_cfg = _models()
    lens = [64, 120, 92, 148]
    feat, fl = synth.padded_batch(list(range(len(lens))), lens)

    def unpacked(*a, **k):
        raise AssertionError("the encoder left the packed path")
    asr.encoder.forward_ragged = unpacked
    dec = BeamDecoder(asr, None, beam, 0.01, ratio, lm_path=lm_path, lm_config=lm_cfg, lm_weight=lm_w, ctc_weight=ctc_w).to(cuda)
    out = dec.decode_batch(feat.to(cuda), fl.to(cuda))
    del asr.encoder.forward_ragged
    same = ties = 0
    for k, n in enumerate(lens):
        ora = _oracle_nbest(asr, lm, feat[k], n, beam, lm_w, ctc_w, max_ratio=ratio)
        assert len(out[k]) == len(ora)
        if not ora:
            continue
        s, t = _compare(out[k], ora, "%s beam %d lm %.1f ctc %.1f utt %d" % (variant, beam, lm_w, ctc_w, k))
        same, ties = same + s, ties + t
    print("%s beam %d lm_w %.1f ctc_w %.1f: identical 1-best %d/%d, ties %d" % (variant, beam, lm_w, ctc_w, same, len(lens), ties))
    assert same >= len(lens) - 1
