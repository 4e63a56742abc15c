"""Multi-head location-aware attention on the B200: e2e_attention_loc_heads against its CPU checker, and the batched
beam search of multi-head models against the per-hypothesis oracle."""
import copy

import pytest
import torch

from tests._attention_heads_oracle import loc_attention_full_heads
from tests.test_gpu_decode import _compare, _models, _oracle_nbest

pytestmark = pytest.mark.gpu


def _inputs(n_utts, beam, heads, t_len, dim, n_filt, half, e_dim, per_head, seed):
    g = torch.Generator().manual_seed(seed)
    n = n_utts * beam
    key = torch.tanh(torch.randn(n_utts, heads, t_len, dim, generator=g))
    value = torch.randn(n_utts, t_len, e_dim * (heads if per_head else 1), generator=g)
    query = torch.tanh(torch.randn(n, heads * dim, generator=g))
    enc_len = torch.tensor([max(1, t_len - 7 * i) for i in range(n_utts)], dtype=torch.int32)
    prev = torch.softmax(torch.randn(n, heads, t_len, generator=g) * 2, -1)
    for i in range(n):                                   # previous alignments are zero beyond the utterance
        prev[i, :, int(enc_len[i // beam]):] = 0
    conv_w = torch.randn(n_filt, heads, 2 * half + 1, generator=g) * 0.3 / heads ** 0.5
    w_proj = torch.randn(dim, n_filt, generator=g) / n_filt ** 0.5
    w_e = torch.randn(dim, generator=g) / dim ** 0.5 * 4
    return key, value, query, enc_len, prev, conv_w, w_proj, w_e


def _run(ops, cuda, key, value, query, enc_len, prev, conv_w, w_proj, w_e, beam, per_head, **kw):
    dev = lambda t: t.to(cuda)
    return ops.attention_loc_heads(dev(key).permute(0, 1, 3, 2).contiguous(), dev(value), dev(query), dev(prev), dev(enc_len),
                                   dev(conv_w), dev(w_proj), dev(w_e), 0.25, 0.5, beam, per_head, **kw)


@pytest.mark.parametrize("n_utts,beam,heads,t_len,dim,n_filt,half,e_dim,per_head", [
    (3, 8, 2, 180, 300, 10, 100, 640, False),            # the bench shape, values shared by the heads
    (3, 8, 2, 180, 300, 10, 100, 640, True),             # ... and per-head values (v_proj)
    (2, 1, 3, 37, 24, 4, 10, 17, True),                  # beam 1, T and E not multiples of 4
    (2, 1, 3, 37, 24, 4, 10, 40, False),
    (4, 32, 4, 300, 128, 12, 25, 96, False),             # beam 32, every slot's queries in one CTA
    (2, 32, 4, 61, 300, 12, 100, 33, True),              # the largest supported staging (B 32, H 4, A 300, W 201, K 12): CTA groups of 8 slots
    (2, 32, 2, 40, 300, 10, 100, 64, False),             # H 2: CTA groups of 28 / 24 / 20 slots at 1 / 2 / 4 slots a warp
    (2, 30, 4, 40, 300, 12, 100, 24, True),              # partial last group: 8 / 8 / 8 / 6 slots
    (2, 8, 4, 50, 32, 7, 3, 17, True),
    (1, 8, 4, 875, 300, 10, 100, 640, True),             # full-size dims, long form
])
def test_attention_loc_heads_matches_oracle(cuda, n_utts, beam, heads, t_len, dim, n_filt, half, e_dim, per_head):
    """attn within 5e-6 abs, context within 2e-5 abs of the fp32 CPU restatement; identical bits for every
    hypotheses-per-unit grouping; exact zeros beyond enc_len; only the first n_run utterances are written."""
    from e2e_asr_pytorch_b200 import ops
    key, value, query, enc_len, prev, conv_w, w_proj, w_e = _inputs(n_utts, beam, heads, t_len, dim, n_filt, half, e_dim, per_head,
                                                                     t_len + dim + heads)
    want_a, want_c = loc_attention_full_heads(key, value, query, prev, enc_len, conv_w, w_proj, w_e, 0.25, 0.5, beam, per_head)
    outs = []
    for nb in (0, 1, 2, 4):
        got_a, got_c = _run(ops, cuda, key, value, query, enc_len, prev, conv_w, w_proj, w_e, beam, per_head, hyps_per_unit=nb)
        outs.append((got_a.cpu(), got_c.cpu()))
    got_a, got_c = outs[0]
    assert got_a.shape == want_a.shape and got_c.shape == want_c.shape
    err_a, err_c = (got_a - want_a).abs().max().item(), (got_c - want_c).abs().max().item()
    print("attention heads U=%d B=%d H=%d T=%d A=%d E=%d per-head values %s: max |gpu-oracle| attn %.3g ctx %.3g"
          % (n_utts, beam, heads, t_len, dim, e_dim, per_head, err_a, err_c))
    assert err_a < 5e-6 and err_c < 2e-5
    for a, c in outs[1:]:
        assert torch.equal(a, got_a) and torch.equal(c, got_c)
    for u in range(n_utts):
        assert (got_a[u * beam:(u + 1) * beam, :, int(enc_len[u]):] == 0).all()
    if n_utts > 1:                                       # n_run: rows of later utterances stay untouched
        n = n_utts * beam
        attn = torch.full((n, heads, t_len), -7.0, device=cuda)
        ctx = torch.full((n, heads * e_dim), -7.0, device=cuda)
        _run(ops, cuda, key, value, query, enc_len, prev, conv_w, w_proj, w_e, beam, per_head, n_run=1, attn=attn, ctx=ctx)
        assert torch.equal(attn[:beam].cpu(), got_a[:beam]) and torch.equal(ctx[:beam].cpu(), got_c[:beam])
        assert (attn[beam:] == -7.0).all() and (ctx[beam:] == -7.0).all()


@pytest.mark.parametrize("n_utts,beam,t_len,dim,n_filt,half,e_dim", [(3, 8, 180, 300, 10, 100, 640), (2, 3, 37, 24, 4, 10, 17)])
def test_attention_loc_heads_one_head_is_the_single_head_kernel(cuda, n_utts, beam, t_len, dim, n_filt, half, e_dim):
    from e2e_asr_pytorch_b200 import ops
    key, value, query, enc_len, prev, conv_w, w_proj, w_e = _inputs(n_utts, beam, 1, t_len, dim, n_filt, half, e_dim, False, 7)
    dev = lambda t: t.to(cuda)
    for nb in (0, 1, 2, 4):
        a1, c1 = ops.attention_loc_full(dev(key[:, 0]).transpose(1, 2).contiguous(), dev(value), dev(query), dev(prev[:, 0]),
                                        dev(enc_len), dev(conv_w[:, 0]), dev(w_proj), dev(w_e), 0.25, 0.5, beam, hyps_per_unit=nb)
        ah, ch = _run(ops, cuda, key, value, query, enc_len, prev, conv_w, w_proj, w_e, beam, False, hyps_per_unit=nb)
        assert torch.equal(ah[:, 0], a1) and torch.equal(ch, c1)


def test_every_supported_shape_launches(cuda):
    """Every (beam, heads, filters) the shape query accepts at the full-size dims (A = 300, W = 201) runs."""
    from e2e_asr_pytorch_b200 import ops
    launched = 0
    for heads in range(1, 6):
        for n_filt in (4, 12):
            for beam in range(1, 34):
                if not ops.attention_loc_heads_supported(beam, heads, 300, n_filt, 201):
                    assert heads > 4 or beam > 32
                    continue
                key, value, query, enc_len, prev, conv_w, w_proj, w_e = _inputs(2, beam, heads, 12, 300, n_filt, 100, 8, True, beam)
                a, c = _run(ops, cuda, key, value, query, enc_len, prev, conv_w, w_proj, w_e, beam, True)
                assert torch.isfinite(a).all() and torch.isfinite(c).all()
                launched += 1
    torch.cuda.synchronize()
    assert launched == 4 * 2 * 32


@pytest.mark.parametrize("heads,mode,v_proj", [(2, "loc", False), (2, "loc", True), (4, "loc", False), (2, "dot", False), (5, "loc", False)])
def test_decode_multi_head_models_match_oracle(cuda, heads, mode, v_proj):
    """Multi-head models (attention.num_head = H) decode like the per-hypothesis oracle, beam 4 + RNNLM + CTC.  The
    location-aware cases with H <= 4 must have taken the fused kernel; scaled-dot attention and H = 5 take the plain
    PyTorch multi-head step."""
    from e2e_asr_pytorch_b200 import BeamDecoder, synth
    cfg = copy.deepcopy(synth.TINY_ASR_CFG)
    cfg["attention"].update({"mode": mode, "v_proj": v_proj, "num_head": heads})
    asr = synth.build_asr(31, cfg, seed=0, peak=4.0)
    _, lm, lm_path, lm_cfg = _models()
    lens = [64, 120, 92, 148]
    feat, fl = synth.padded_batch(list(range(len(lens))), lens)
    dec = BeamDecoder(asr, None, 4, 0.01, 0.2, lm_path=lm_path, lm_config=lm_cfg, lm_weight=0.3, ctc_weight=0.5).to(cuda)
    out = dec.decode_batch(feat.to(cuda), fl.to(cuda))
    assert dec._stepper[2].fused_step == (mode == "loc" and heads <= 4)
    same = ties = 0
    for k, n in enumerate(lens):
        ora = _oracle_nbest(asr, lm, feat[k], n, 4, 0.3, 0.5)
        assert len(out[k]) == len(ora)
        s, t = _compare(out[k], ora, "heads %d %s v_proj %s utt %d" % (heads, mode, v_proj, k))
        same, ties = same + s, ties + t
    print("heads %d, attention %s, v_proj %s: identical 1-best %d/%d, ties %d" % (heads, mode, v_proj, same, len(lens), ties))
    assert same >= len(lens) - 1
