"""GRU models on the device path (B200): the fused GRU cell (csrc/lstm_step.cu), the fused GRU step stack of the
speller / RNNLM (stepper._FusedLstm over an nn.GRU), the packed bidirectional GRU recurrence of the encoder
(csrc/lstm_seq.cu) and whole all-GRU decodes against the per-hypothesis oracle."""
import os
import tempfile

import pytest
import torch
import yaml

from tests.test_gpu_decode import _compare, _oracle_nbest
from tests.test_gpu_kernels import copy_double

pytestmark = pytest.mark.gpu


def _ops():
    from e2e_asr_pytorch_b200 import ops, _lib
    return ops, _lib


@pytest.mark.parametrize("pieces", [3, 2])
@pytest.mark.parametrize("n,d,with_table,with_next,gather", [(33, 1024, True, True, True), (9, 300, False, True, True),
                                                             (4, 12, True, True, False), (6, 300, True, False, True)])
def test_gru_cell_matches_float64(cuda, pieces, n, d, with_table, with_next, gather):
    """h' within 1e-6 abs of a float64 GRU cell on the same gate pre-activations, h read through the parents' row index;
    the split of h' in the next layer's operand is bit-exact in both piece formats (D = 1024 and 300 take the 16-byte
    path; D = 12 with an odd next-operand offset takes the scalar one)."""
    ops, _ = _ops()
    from e2e_asr_pytorch_b200.stepper import _split3, _split2_f16, F16_ACT_SCALE
    g = torch.Generator().manual_seed(d + pieces)
    gates = torch.randn(n, 4 * d, generator=g) * 2
    bias = torch.randn(4 * d, generator=g)
    table = torch.randn(5, 4 * d, generator=g) if with_table else None
    tok = torch.randint(0, 5, (n,), generator=g) if with_table else None
    h_prev = torch.randn(n + 3, d, generator=g).tanh()
    idx = torch.randint(0, n + 3, (n,), generator=g) if gather else None
    z = gates.double() + bias.double() + (table.double()[tok] if with_table else 0)
    zr, zz, znx, znh = z.chunk(4, dim=-1)
    r, u = torch.sigmoid(zr), torch.sigmoid(zz)
    nn_ = torch.tanh(znx + r * znh)
    hp = h_prev.double()[idx] if gather else h_prev.double()[:n]
    want = (hp - nn_) * u + nn_
    dev = lambda t: None if t is None else t.to(cuda)
    h_new = torch.empty(n, d, device=cuda)
    off = 1 if d == 12 else 0
    k_next = 2 * d + off
    if pieces == 3:
        a_next = torch.zeros(n, 3 * k_next, dtype=torch.bfloat16, device=cuda) if with_next else None
        ops.gru_cell(dev(gates), dev(bias), dev(h_prev), dev(idx), n, h_new, table=dev(table), tok=dev(tok),
                     a_next=a_next, k_next=k_next if with_next else 0, off_next=off)
    else:
        gate_scale = 2.0 ** -3                       # the GEMM result carries 8x the gates; the kernel takes it out exactly
        a_next = torch.zeros(n, 2 * k_next, dtype=torch.float16, device=cuda) if with_next else None
        ops.gru_cell(dev(gates * 8), dev(bias), dev(h_prev), dev(idx), n, h_new, table=dev(table), tok=dev(tok),
                     a_next=a_next, k_next=k_next if with_next else 0, off_next=off, gate_scale=gate_scale, next_scale=F16_ACT_SCALE)
    assert (h_new.cpu().double() - want).abs().max().item() < 1e-6
    if with_next:
        parts = _split3(h_new) if pieces == 3 else _split2_f16(h_new, F16_ACT_SCALE)
        for p in range(pieces):
            assert torch.equal(a_next[:, p * k_next + off:p * k_next + off + d], parts[p])


@pytest.mark.parametrize("split", ["bf16x3", "fp16x2"])
def test_fused_gru_stack_matches_nn_gru(cuda, split):
    """Three steps of the device GRU stack (split kernel + split GEMMs on the 4-block gate form + GRU cell kernel, states
    read through the parents' row index) against torch.nn.GRU in float64 fed with the same parent permutation."""
    _ops()
    from e2e_asr_pytorch_b200.stepper import _FusedLstm
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    torch.manual_seed(3)
    cases = [(24, 16, 1, False), (24, 16, 2, False), (16, 16, 3, True), (16, 16, 1, True)]
    if split == "fp16x2":
        cases = [c for c in cases if c[3]]               # the fp16 format needs a tabled layer 0
    for in_dim, d, layers, table in cases:
        rnn = torch.nn.GRU(in_dim, d, num_layers=layers, batch_first=True)
        emb = torch.randn(7, in_dim)
        ref = torch.nn.GRU(in_dim, d, num_layers=layers, batch_first=True).double()
        ref.load_state_dict({k: v.double() for k, v in rnn.state_dict().items()})
        n = 10
        with torch.no_grad(), _Fp32Math():
            fused = _FusedLstm(rnn.to(cuda), emb.to(cuda) if table else None, split=split)
            assert fused.gru
            fused.start(n, cuda)
            assert fused.c is None
            h = torch.zeros(layers, n, d, dtype=torch.float64)
            g = torch.Generator().manual_seed(5)
            for step in range(3):
                tok = torch.randint(0, 7, (n,), generator=g)
                x = emb[tok] if table else torch.randn(n, in_dim, generator=g)
                top = fused.step(n, x0=None if table else x.to(cuda), tok=tok.to(cuda) if table else None)
                out, h = ref(x.double()[:, None, :], h)
                assert (top.cpu().double() - out[:, 0]).abs().max().item() < 2e-6, (in_dim, d, layers, table, step)
                perm = torch.randint(0, n, (n,), generator=g)           # survivors pick parents
                fused.reorder(perm.to(cuda))
                h = h[:, perm]
                assert (fused.hidden(n).cpu().double() - torch.cat(list(h), dim=1)).abs().max().item() < 2e-6


@pytest.mark.parametrize("hidden,in_dim,lens", [(16, 24, [30, 22, 22, 9, 1]), (320, 64, [70, 41] + [33] * 20), (40, 12, [700, 650, 310, 12])])
def test_gru_sequence_matches_nn_gru(cuda, hidden, in_dim, lens):
    """Packed bidirectional GRU layer (RecurrentLayer.forward_packed: split GEMM + persistent GRU kernel + projection) vs
    the layer's own per-utterance forward in float64; groups of 4 / 8 / 16 utterances are all exercised."""
    _ops()
    from e2e_asr_pytorch_b200.model import RecurrentLayer, Encoder, reference_init_
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    torch.manual_seed(hidden)
    layer = RecurrentLayer(in_dim, "GRU", hidden, True, 0.0, False, 1, "drop", True)
    layer.apply(reference_init_)
    for n, p in layer.named_parameters():
        if "bias" in n:
            p.data.normal_(0, 0.3)
    layer.eval()
    assert layer.packed_supported()
    g = torch.Generator().manual_seed(1)
    xs = [torch.randn(l, in_dim, generator=g) for l in lens]
    with torch.no_grad():
        ref = copy_double(layer)
        want = torch.cat([ref(x[None].double(), torch.tensor([x.shape[0]]))[0][0] for x in xs], dim=0)
        layer.to(cuda)
        t_len = torch.tensor(lens)
        off = (torch.cumsum(t_len, 0) - t_len).to(torch.int32).to(cuda)
        first, rows = Encoder._groups(t_len)
        with _Fp32Math():
            got = layer.forward_packed(torch.cat(xs).to(cuda), off, t_len.to(torch.int32).to(cuda),
                                       torch.tensor(first, dtype=torch.int32, device=cuda), torch.tensor(rows, dtype=torch.int32, device=cuda))
    err = (got.cpu().double() - want).abs().max().item()
    print("packed BGRU H=%d: max |gpu - fp64| = %.3g (groups %s)" % (hidden, err, sorted(set(rows))))
    assert err < 5e-6


def _gru_asr_cfg():
    import copy
    from e2e_asr_pytorch_b200 import synth
    cfg = copy.deepcopy(synth.TINY_ASR_CFG)
    cfg["encoder"]["module"] = "GRU"
    cfg["decoder"].update({"module": "GRU", "layer": 2})
    return cfg


def test_packed_gru_encoder_matches_per_utterance_calls(cuda):
    """Encoder.forward_ragged_packed of an all-GRU encoder (split-bf16 VGG + packed BGRU stack) vs one batch-1 float64
    call per utterance."""
    _ops()
    from e2e_asr_pytorch_b200 import synth
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    asr = synth.build_asr(31, _gru_asr_cfg(), seed=0)
    enc = asr.encoder
    lens = [96, 92, 64, 40, 40, 12]
    feat, fl = synth.padded_batch(list(range(len(lens))), lens)
    with torch.no_grad():
        ref = copy_double(enc)
        wants = [ref(feat[i:i + 1, :n].double(), fl[i:i + 1])[0][0] for i, n in enumerate(lens)]
        enc.to(cuda)
        enc.split_conv = True
        assert enc.packed_supported()
        with _Fp32Math():
            got, gl = enc.forward_ragged_packed(feat.to(cuda), fl.to(cuda), chunk=4)
    assert gl.cpu().tolist() == [n // 4 for n in lens]
    for i, w in enumerate(wants):
        err = (got[i, :w.shape[0]].cpu().double() - w).abs().max().item()
        assert err < 5e-6, (i, err)
        assert (got[i, w.shape[0]:] == 0).all()


def _gru_models():
    import copy
    from e2e_asr_pytorch_b200 import synth
    asr = synth.build_asr(31, _gru_asr_cfg(), seed=0, peak=4.0)
    lm_cfg = copy.deepcopy(synth.TINY_LM_CFG)
    lm_cfg["module"] = "GRU"
    lm = synth.build_lm(31, lm_cfg, seed=1)
    tmp = tempfile.mkdtemp()
    torch.save({"model": lm.state_dict()}, os.path.join(tmp, "lm.pth"))
    yaml.safe_dump({"model": lm_cfg}, open(os.path.join(tmp, "lm.yaml"), "w"))
    return asr, lm, os.path.join(tmp, "lm.pth"), os.path.join(tmp, "lm.yaml")


@pytest.mark.parametrize("beam,lm_w,ctc_w", [(1, 0.0, 0.0), (1, 0.3, 0.0), (4, 0.3, 0.5), (4, 0.0, 0.0), (8, 0.5, 0.5), (8, 0.0, 0.5)])
def test_all_gru_decode_matches_oracle(cuda, beam, lm_w, ctc_w):
    """All-GRU models (BGRU encoder, 2-layer GRU speller, GRU RNNLM) decode on the device path — fused GRU step stacks
    and the packed GRU encoder — to the oracle's 1-best, or a tie by its own scores, for all but at most one utterance."""
    from e2e_asr_pytorch_b200 import BeamDecoder, synth
    from e2e_asr_pytorch_b200.stepper import _FusedLstm
    asr, lm, lm_path, lm_cfg = _gru_models()
    lens = [64, 120, 92, 148]
    feat, fl = synth.padded_batch(list(range(len(lens))), lens)
    dec = BeamDecoder(asr, None, beam, 0.01, 0.2, lm_path=lm_path, lm_config=lm_cfg, lm_weight=lm_w, ctc_weight=ctc_w).to(cuda)
    out = dec.decode_batch(feat.to(cuda), fl.to(cuda))
    stepper = dec._stepper[2]
    assert isinstance(stepper.dec, _FusedLstm) and stepper.dec.gru and stepper.dec_fused
    if lm_w > 0:
        assert isinstance(stepper.lm_rnn, _FusedLstm) and stepper.lm_rnn.gru and stepper.lm_fused
    assert asr.encoder.packed_supported() and stepper.split_conv
    same = ties = 0
    for k, n in enumerate(lens):
        ora = _oracle_nbest(asr, lm, feat[k], n, beam, lm_w, ctc_w)
        assert len(out[k]) == len(ora)
        if not ora:
            continue
        s, t = _compare(out[k], ora, "all-GRU beam %d lm %.1f ctc %.1f utt %d" % (beam, lm_w, ctc_w, k))
        same, ties = same + s, ties + t
    print("all-GRU beam %d lm_w %.1f ctc_w %.1f: identical 1-best %d/%d, ties %d" % (beam, lm_w, ctc_w, same, len(lens), ties))
    assert same >= len(lens) - 1
