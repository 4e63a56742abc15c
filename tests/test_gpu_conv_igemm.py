"""The VGG convolutions as one tcgen05 implicit split GEMM (csrc/conv_igemm.cu) against the unfold path
(csrc/conv_split.cu unfold + the three library GEMMs + bias_relu_mask(_pool)), which it must reproduce bit for bit:
first the GEMM core alone (raw epilogue vs mm/addmm/addmm on the unfolded operand), then whole layers with the fused
epilogue, then the front end and a decode."""
import pytest
import torch

pytestmark = pytest.mark.gpu

LAYERS = [(128, 128, True), (128, 256, False), (256, 256, True)]     # (Cin, Cout, pooled) of VGGFrontEnd's layers 2..4


def _front(cuda, seed=0):
    from e2e_asr_pytorch_b200.model import VGGFrontEnd
    torch.manual_seed(seed)
    return VGGFrontEnd(160).to(cuda)


def _conv(front, cin, cout):
    return next(m for m in front.extractor if isinstance(m, torch.nn.Conv2d) and m.in_channels == cin and m.out_channels == cout)


def _input(cuda, n, h, w, c, valid, seed=1):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, h, w, c, generator=g).abs() * 2.5                # ReLU outputs of the previous layer
    for i, v in enumerate(valid):
        x[i, v:] = 0
    return x.to(cuda), torch.tensor(valid, dtype=torch.int32, device=cuda)


def _library_gemm(front, conv, x, valid):
    """y [N*H*W, Cout] of the unfold path: unfold + split, then mm / addmm / addmm as VGGFrontEnd._conv_split runs them."""
    from e2e_asr_pytorch_b200 import ops
    n, h, w, c = x.shape
    k, total = 9 * c, n * h * w
    lin = front._split_weights(conv)
    a = torch.empty((total, 3 * k), dtype=torch.bfloat16, device=x.device)
    ops.conv3x3_unfold_split(x, valid, 0, total, a)
    y = torch.mm(a, lin.b2, out_dtype=torch.float32)
    torch.addmm(y, a[:, :2 * k], lin.b1, out_dtype=torch.float32, out=y)
    torch.addmm(y, a[:, :k], lin.b0, out_dtype=torch.float32, out=y)
    return y


def _ulps(a, b):
    ia, ib = a.view(torch.int32).long(), b.view(torch.int32).long()
    return int((ia - ib).abs().max())


# ragged batches: lengths 1..3 rows, full rows, and pixel counts that leave a partial last tile
SHAPES = [
    (3, 9, 40, [9, 3, 1]),
    (4, 7, 20, [7, 2, 5, 3]),
    (2, 5, 13, [5, 4]),
    (128, 48, 40, None),          # a bench-sized chunk of 128 utterances
    (128, 24, 20, None),
]


def _valid(n, h, lens, seed=3):
    if lens is not None:
        return lens
    g = torch.Generator().manual_seed(seed)
    return [int(v) for v in torch.randint(1, h + 1, (n,), generator=g)]


@pytest.mark.parametrize("cin,cout,pooled", LAYERS)
@pytest.mark.parametrize("n,h,w,lens", SHAPES)
def test_gemm_core_matches_library_gemms(cuda, cin, cout, pooled, n, h, w, lens):
    from e2e_asr_pytorch_b200 import ops
    front = _front(cuda)
    conv = _conv(front, cin, cout)
    x, valid = _input(cuda, n, h, w, cin, _valid(n, h, lens))
    ref = _library_gemm(front, conv, x, valid)
    got = ops.conv3x3_igemm(x, valid, front._igemm_weights(conv), None, "raw")
    torch.cuda.synchronize()
    assert torch.equal(got, ref), "max %d ulp" % _ulps(got, ref)


@pytest.mark.parametrize("cin,cout,pooled", LAYERS)
@pytest.mark.parametrize("n,h,w,lens", SHAPES)
def test_layer_matches_unfold_path(cuda, cin, cout, pooled, n, h, w, lens):
    front = _front(cuda)
    conv = _conv(front, cin, cout)
    x, valid = _input(cuda, n, h, w, cin, _valid(n, h, lens), seed=5)
    from e2e_asr_pytorch_b200 import ops
    front.conv_path = "unfold"
    ref = front._conv_split(x, valid, conv, pool=pooled)
    got = ops.conv3x3_igemm(x, valid, front._igemm_weights(conv), conv.bias.detach().float().contiguous(),
                            "pool" if pooled else "relu")
    torch.cuda.synchronize()
    assert got.shape == ref.shape
    assert torch.equal(got, ref), "max %d ulp" % _ulps(got, ref)


def test_front_end_routes_the_128_channel_layer(cuda, monkeypatch):
    from e2e_asr_pytorch_b200 import ops
    front = _front(cuda)
    seen = []
    real = ops.conv3x3_igemm
    monkeypatch.setattr(ops, "conv3x3_igemm", lambda x, *a, **k: seen.append(x.shape[3]) or real(x, *a, **k))
    feat = torch.randn(2, 40, 160, device=cuda)
    front.forward_masked_split(feat, torch.tensor([40, 17]))
    assert seen == [128]
    front.conv_path = "unfold"
    front.forward_masked_split(feat, torch.tensor([40, 17]))
    assert seen == [128]


def test_front_end_matches_unfold_path(cuda):
    front = _front(cuda, seed=7)
    g = torch.Generator().manual_seed(8)
    lens = torch.tensor([203, 4, 5, 6, 7, 150, 64, 12])             # 4..7 frames: 1 row after the first pool, ragged tails
    feat = torch.randn(len(lens), 203, 160, generator=g)
    for i, v in enumerate(lens):
        feat[i, v:] = 0
    feat = feat.to(cuda)
    front.conv_path = "unfold"
    ref, ref_len = front.forward_masked_split(feat, lens)
    front.conv_path = "igemm"
    got, got_len = front.forward_masked_split(feat, lens)
    torch.cuda.synchronize()
    assert torch.equal(got_len, ref_len)
    assert torch.equal(got, ref)


def test_decode_is_unchanged(cuda):
    from e2e_asr_pytorch_b200 import BeamDecoder, synth
    from tests.test_gpu_decode import _models
    asr, _, lm_path, lm_cfg = _models()
    lens = [64, 120, 92, 200, 76, 148, 36, 41]
    feat, fl = synth.padded_batch(list(range(len(lens))), lens)
    out = {}
    for path in ("unfold", "igemm"):
        dec = BeamDecoder(asr, None, 8, 0.01, 0.2, lm_path=lm_path, lm_config=lm_cfg, lm_weight=0.5, ctc_weight=0.5).to(cuda)
        dec.vgg_conv = path
        out[path] = dec.decode_batch(feat.to(cuda), fl.to(cuda), return_arrays=True)
        assert dec._stepper[2].asr.encoder.layers[0].conv_path == path
    for a, b in zip(out["unfold"], out["igemm"]):
        assert torch.equal(a, b)


def test_refuses_other_shapes(cuda):
    from e2e_asr_pytorch_b200 import ops, _lib
    assert ops.conv3x3_igemm_supported(128, 128) and ops.conv3x3_igemm_supported(256, 256)
    assert not ops.conv3x3_igemm_supported(64, 128) and not ops.conv3x3_igemm_supported(128, 192)
    x = torch.zeros(1, 4, 4, 64, device=cuda)
    w = torch.zeros(3, 128, 9 * 64, dtype=torch.bfloat16, device=cuda)
    with pytest.raises(_lib.E2EError):
        ops.conv3x3_igemm(x, torch.ones(1, dtype=torch.int32, device=cuda), w, torch.zeros(128, device=cuda), "relu")
