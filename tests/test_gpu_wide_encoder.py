"""Encoder recurrent layers wider than 384 units on the packed device path (B200): the thread-block cluster form of the
packed recurrence (csrc/lstm_seq.cu, e2e_lstm_sequence_wide / e2e_gru_sequence_wide) against the one-CTA form bit for
bit where both apply, wide packed layers and whole wide encoders against batch-1 float64 module calls, and decodes of
512-wide models against the per-hypothesis oracle."""
import copy
import re

import pytest
import torch

from tests.test_gpu_decode import _compare, _models, _oracle_nbest
from tests.test_gpu_encoder_subsample import _layer, _randomize
from tests.test_gpu_kernels import copy_double

pytestmark = pytest.mark.gpu


def _lib():
    from e2e_asr_pytorch_b200 import _lib as L
    return L, L.load()


def _run_entry(name, gates, out, off, lens, first, rows, h, dirs):
    from e2e_asr_pytorch_b200 import ops
    L, lib = _lib()
    n_g = 3 if "gru" in name else 4
    fw = dirs[0]
    bw = dirs[1] if len(dirs) == 2 else (None, None)
    L.check(getattr(lib, name)(L.ptr(gates), int(gates.stride(0)), L.ptr(out), int(out.stride(0)), L.ptr(off), L.ptr(lens),
                               L.ptr(first), L.ptr(rows), int(lens.numel()), h, int(first.numel()), len(dirs),
                               L.ptr(fw[0]), L.ptr(fw[1]), 0, 0, L.ptr(bw[0]), L.ptr(bw[1]), n_g * h, h, ops._stream()))


# ragged lengths with 1 among them, and groups of every template size, full and partial (the kernel picks R = 4, 8, 16
# from the group's row count)
BIT_LENS = [57, 40, 40, 33, 31, 29, 17, 17, 16, 12, 9, 9, 8, 5, 4, 3, 3, 2, 2, 1, 1, 1, 7, 6, 6, 5, 5, 4, 3, 2, 1, 1, 1]
BIT_GROUPS = [4, 3, 8, 5, 13]                    # 33 utterances: R = 4 (full, partial), 8 (full, partial), 16 (partial)


@pytest.mark.parametrize("module", ["lstm", "gru"])
@pytest.mark.parametrize("hidden", [256, 384])
@pytest.mark.parametrize("n_dirs", [1, 2])
def test_wide_entry_points_reproduce_the_narrow_ones_bit_for_bit(cuda, module, hidden, n_dirs):
    """At H = 256 and 384 the cluster form (2 CTAs of H / 2 units) writes the same bits as the one-CTA form."""
    g = torch.Generator().manual_seed(hidden + n_dirs)
    n_g = 3 if module == "gru" else 4
    lens = torch.tensor(BIT_LENS, dtype=torch.int32)
    f = int(lens.sum())
    gates = (torch.randn(f, 2 * n_g * hidden, generator=g) * 0.8).to(cuda)
    dirs = []
    for _ in range(n_dirs):
        bias = (torch.randn(4 * hidden, generator=g) * 0.3).to(cuda)
        w_t = torch.randn(hidden, hidden, 4, generator=g) / hidden ** 0.5
        if module == "gru":
            w_t[:, :, 3] = 0
        dirs.append((bias, w_t.contiguous().to(cuda)))
    off = (torch.cumsum(lens, 0) - lens).to(torch.int32).to(cuda)
    first = torch.tensor([sum(BIT_GROUPS[:i]) for i in range(len(BIT_GROUPS))], dtype=torch.int32, device=cuda)
    rows = torch.tensor(BIT_GROUPS, dtype=torch.int32, device=cuda)
    assert sum(BIT_GROUPS) == len(BIT_LENS)
    outs = []
    for name in ("e2e_%s_sequence" % module, "e2e_%s_sequence_wide" % module):
        out = torch.full((f, 2 * hidden), float("nan"), device=cuda)
        _run_entry(name, gates, out, off, lens.to(cuda), first, rows, hidden, dirs)
        outs.append(out.cpu())
    torch.cuda.synchronize()
    cols = slice(0, n_dirs * hidden)
    assert not outs[0][:, cols].isnan().any()
    assert torch.equal(outs[0][:, cols], outs[1][:, cols])


def _cudnn_error(layer, xs, want, cuda):
    """max |fp32 cuDNN - float64| of the layer's own batch-1 calls on the device, the same frames."""
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    with torch.no_grad(), _Fp32Math():
        got = torch.cat([layer(x[None].to(cuda), torch.tensor([x.shape[0]]))[0][0].cpu() for x in xs], dim=0)
    return (got.double() - want).abs().max().item()


@pytest.mark.parametrize("module", ["LSTM", "GRU"])
@pytest.mark.parametrize("hidden", [512, 768, 1024])
def test_wide_packed_layer_matches_float64(cuda, module, hidden):
    """RecurrentLayer.forward_packed (bidirectional, projection) at H = 512 / 768 / 1024, the cluster form with 2, 2 and 4
    CTAs, vs the layer's own batch-1 forward in float64, within 5e-6, or 1.5x the error of fp32 cuDNN on the same
    layer where that is larger (both printed).  Groups of 4, 8 and 16 utterances."""
    from e2e_asr_pytorch_b200.model import Encoder, packed_offsets
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    in_dim = 64
    layer = _layer(module, in_dim, hidden, 1, "drop", False, True, hidden)
    assert layer.packed_supported()
    lens = [610, 330, 320, 301, 300, 41, 40, 39, 38, 37, 36, 35] + [30 - k for k in range(10)] + [1]
    g = torch.Generator().manual_seed(1)
    xs = [torch.randn(l, in_dim, generator=g) for l in lens]
    t_len = torch.tensor(lens)
    with torch.no_grad():
        ref = copy_double(layer)
        want = torch.cat([ref(x[None].double(), torch.tensor([x.shape[0]]))[0][0] for x in xs], dim=0)
        layer.to(cuda)
        off, lens32 = packed_offsets(t_len, cuda)
        first, rows = Encoder._groups(t_len)
        assert rows == [4, 8, 11]
        with _Fp32Math():
            got = layer.forward_packed(torch.cat(xs).to(cuda), off, lens32, torch.tensor(first, dtype=torch.int32, device=cuda),
                                       torch.tensor(rows, dtype=torch.int32, device=cuda))
    err = (got.cpu().double() - want).abs().max().item()
    cudnn = _cudnn_error(layer, xs, want, cuda)
    bound = max(5e-6, 1.5 * cudnn)
    print("packed B%s H=%d: max |gpu - fp64| = %.3g, fp32 cuDNN %.3g, bound %.3g (groups %s)"
          % (module, hidden, err, cudnn, bound, sorted(set(rows))))
    assert err < bound


WIDE_ENCODERS = {
    "vgg_blstm": ({}, [96, 92, 64, 40, 40, 12]),
    # a 'drop' layer and LayerNorm on every layer, behind the VGG front end
    "vgg_drop_ln": ({"sample_rate": [2, 1], "sample_style": "drop", "layer_norm": [True, True]}, [96, 92, 68, 44, 40, 12, 8]),
}


def _wide_asr(variant=None, module="LSTM", peak=1.0):
    from e2e_asr_pytorch_b200 import synth
    cfg = copy.deepcopy(synth.TINY_WIDE_ASR_CFG)
    if variant:
        cfg["encoder"].update(WIDE_ENCODERS[variant][0])
    cfg["encoder"]["module"] = module
    asr = synth.build_asr(31, cfg, seed=0, peak=peak)
    return asr


@pytest.mark.parametrize("variant", sorted(WIDE_ENCODERS))
def test_wide_encoder_matches_batch1_calls(cuda, variant):
    """Encoder.forward_ragged_packed of a 512-wide encoder (split-GEMM VGG + cluster-form BLSTM layers) vs one batch-1
    float64 Encoder call per utterance: rows [0, X) within the 4e-5 bound of encoders behind the VGG front end (its
    split GEMMs sum in another order than the CPU), enc_len == X, zeros beyond."""
    from e2e_asr_pytorch_b200 import synth
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    asr = _wide_asr(variant)
    _randomize(asr.encoder, 7)
    enc = asr.encoder
    lens = WIDE_ENCODERS[variant][1]
    feat, fl = synth.padded_batch(list(range(len(lens))), lens)
    with torch.no_grad():
        ref = copy_double(enc)
        wants = [ref(feat[i:i + 1, :n].double(), fl[i:i + 1]) for i, n in enumerate(lens)]
        enc.to(cuda)
        enc.split_conv = True
        assert enc.packed_supported()
        with _Fp32Math():
            got, gl = enc.forward_ragged_packed(feat.to(cuda), fl.to(cuda), chunk=4)
    assert gl.cpu().tolist() == [int(l[0]) for _, l in wants]
    for i, (w, l) in enumerate(wants):
        x = int(l[0])
        err = (got[i, :x].cpu().double() - w[0, :x]).abs().max().item()
        print("%s utt %d: max |packed - fp64| = %.3g" % (variant, i, err))
        assert err < 4e-5, (variant, i, err)
        assert (got[i, x:] == 0).all()


@pytest.mark.parametrize("module", ["LSTM", "GRU"])
@pytest.mark.parametrize("beam,lm_w,ctc_w", [(1, 0.0, 0.0), (1, 0.3, 0.0), (1, 0.3, 0.5), (4, 0.3, 0.5), (4, 0.0, 0.0),
                                            (8, 0.5, 0.5), (8, 0.0, 0.5)])
def test_wide_model_decode_matches_oracle(cuda, module, beam, lm_w, ctc_w):
    """512-wide models (2 x 512 BLSTM or BGRU encoder, 512-wide speller) decode through the packed encoder
    (forward_ragged is made to raise) to the oracle's 1-best, or a tie by its own scores, for all but at most one
    utterance.  At beam 1 with CTC and the RNNLM these random-init models make the reference's own search fail (the
    winner is not among the CTC candidates, src/decode.py:252); the device must then report that failure for the
    utterance the oracle fails on."""
    from e2e_asr_pytorch_b200 import BeamDecoder, synth
    asr = _wide_asr(module=module, peak=4.0)
    _, lm, lm_path, lm_cfg = _models()
    lens = [64, 120, 92, 148]
    feat, fl = synth.padded_batch(list(range(len(lens))), lens)

    def unpacked(*a, **k):
        raise AssertionError("the encoder left the packed path")
    asr.encoder.forward_ragged = unpacked
    dec = BeamDecoder(asr, None, beam, 0.01, 0.2, lm_path=lm_path, lm_config=lm_cfg, lm_weight=lm_w, ctc_weight=ctc_w).to(cuda)
    try:
        out = dec.decode_batch(feat.to(cuda), fl.to(cuda))
    except ValueError as e:
        del asr.encoder.forward_ragged
        m = re.match(r"utterance (\d+): beam winner is not in the CTC candidate list", str(e))
        assert m, str(e)
        k = int(m.group(1))
        with pytest.raises(ValueError, match="not in list"):
            _oracle_nbest(asr, lm, feat[k], lens[k], beam, lm_w, ctc_w)
        print("wide %s beam %d lm_w %.1f ctc_w %.1f: utterance %d fails in the device search and in the oracle's" % (
            module, beam, lm_w, ctc_w, k))
        return
    del asr.encoder.forward_ragged
    same = ties = 0
    for k, n in enumerate(lens):
        ora = _oracle_nbest(asr, lm, feat[k], n, beam, lm_w, ctc_w)
        assert len(out[k]) == len(ora)
        if not ora:
            continue
        s, t = _compare(out[k], ora, "wide %s beam %d lm %.1f ctc %.1f utt %d" % (module, beam, lm_w, ctc_w, k))
        same, ties = same + s, ties + t
    print("wide %s beam %d lm_w %.1f ctc_w %.1f: identical 1-best %d/%d, ties %d" % (module, beam, lm_w, ctc_w, same, len(lens), ties))
    assert same >= len(lens) - 1
