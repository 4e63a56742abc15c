"""Embedding-fusion decoding on the B200: kernel (3a') e2e_emb_fuse_candidates against a float64 restatement of the
plug-in's formula, and whole decodes with the plug-in against the per-hypothesis CPU oracle (tests/_emb_fusion_oracle.py:
oracle/beam_oracle.py's search with the module called exactly as the reference's BeamDecoder calls it)."""
import numpy as np
import pytest
import torch

from tests.test_gpu_decode import _compare, _cpu_copy, _models

pytestmark = pytest.mark.gpu

# max |logp - float64 formula| of the kernel: 3.1e-6 measured over the shapes below on a B200 (the fp32 log of values
# down to the eps floor, log(1e-8) = -18.4, is one ulp of 1.9e-6 there)
LOGP_BOUND = 4e-6


def _ref64(dec, emb, scale, lam, eps):
    pd = torch.softmax(dec.double(), dim=-1)
    pe = torch.softmax(scale.double() * emb.double(), dim=-1)
    lam = lam.double()
    return torch.log((1 - lam) * pd + lam * pe + eps)


def _stable_topk(row, k):
    return np.argsort(-row, kind="stable")[:k]


@pytest.mark.parametrize("vocab", [31, 300, 10000])
@pytest.mark.parametrize("n_cand", [0, 3, 12, 24])
@pytest.mark.parametrize("per_entry", [False, True])
def test_kernel_matches_float64_and_picks_a_stable_top_c(cuda, vocab, n_cand, per_entry):
    from e2e_asr_pytorch_b200 import ops
    g = torch.Generator().manual_seed(vocab + n_cand + per_entry)
    u, b = 5, 8
    n_live = torch.tensor([8, 3, 8, 1, 0], dtype=torch.int32)
    dec = 4 * torch.randn(u * b, vocab, generator=g)
    emb = 3 * torch.randn(u * b, vocab, generator=g)
    if per_entry:
        scale = torch.relu(-0.5 + 2.5 * torch.rand(vocab, generator=g))          # some entries clamped to zero
        lam = torch.rand(vocab, generator=g)
        scale[5] = 1.0
    else:
        scale, lam = torch.tensor([1.7]), torch.tensor([0.3])
    # row 0: every entry but 5 falls to the eps floor, so the candidates past the first are ties broken by index
    dec[0].fill_(-100.0)
    dec[0, 5] = 100.0
    emb[0].fill_(-1000.0)
    emb[0, 5] = 1000.0
    eps = 1e-8
    logp = torch.full((u * b, vocab), 7.0, device=cuda)
    stats = torch.full((u * b, 2), 7.0, device=cuda)
    cand = torch.full((u * b, max(1, n_cand)), -7, dtype=torch.int32, device=cuda)
    ops.emb_fuse_candidates(dec.to(cuda), emb.to(cuda), u, b, vocab, n_cand, scale.to(cuda), lam.to(cuda), eps,
                            n_live.to(cuda), logp, stats, cand)
    torch.cuda.synchronize()
    logp, stats, cand = logp.cpu(), stats.cpu(), cand.cpu()
    want = _ref64(dec, emb, scale, lam, eps)
    live = torch.tensor([bb < int(n_live[uu]) for uu in range(u) for bb in range(b)])
    err = (logp[live].double() - want[live]).abs().max().item()
    print("V %d C %d per-entry %s: max |logp - float64| = %.3g" % (vocab, n_cand, per_entry, err))
    assert err <= LOGP_BOUND
    assert torch.all(stats[live] == 0)
    assert torch.all(logp[~live] == 7.0) and torch.all(stats[~live] == 7.0) and torch.all(cand[~live] == -7)
    floor = np.float32(np.log(np.float32(eps)))
    assert (logp[0] == logp[0, 0]).sum() == vocab - 1 and abs(float(logp[0, 0]) - float(floor)) < 1e-5
    for r in torch.nonzero(live).reshape(-1).tolist():
        if n_cand > 0:
            assert cand[r].tolist() == _stable_topk(logp[r].numpy(), n_cand).tolist(), r
    if n_cand > 0:
        assert cand[0].tolist() == [5] + [v for v in range(vocab) if v != 5][:n_cand - 1]


def _oracle_nbest(asr, lm, emb, feat, n, beam, lm_w, ctc_w, max_ratio, force=None):
    from tests import _emb_fusion_oracle as EO
    asr, lm, emb = _cpu_copy(asr), _cpu_copy(lm), _cpu_copy(emb)
    with torch.no_grad():
        nb = EO.decode_utterance(asr, emb, feat[None, :n], torch.LongTensor([n]), beam, 0.01, max_ratio, lm=lm if lm_w > 0 else None,
                                 lm_weight=lm_w, ctc_weight=ctc_w, force=force)
    return nb if force is not None else EO.nbest_as_arrays(nb)


CASES = [  # vocab, beam, fuse, temperature, fuse_normalize, ctc_w, lm_w, lazy_prefix
    (31, 4, 0.3, 2.0, False, 0.5, 0.3, True),
    (31, 8, -1, -1, True, 0.5, 0.0, False),
    (31, 4, -2, -2, False, 0.0, 0.3, True),       # CTC off, LM on: the aliased <eos> test reads the fused row + LM
    (31, 1, -2, -2, True, 0.0, 0.3, True),        # beam 1 (with CTC, one candidate: a blank winner is the reference's ValueError)
    (31, 4, -1, 1.0, False, 0.0, 0.0, True),
    (31, 8, 0.5, -2, True, 0.5, 0.5, False),
    (300, 8, -2, -2, False, 0.5, 0.5, True),      # wide rows: the streaming selection of (3a') and (3b)
]


@pytest.mark.parametrize("vocab,beam,fuse,temperature,normalize,ctc_w,lm_w,lazy", CASES)
def test_decode_with_embedding_fusion_matches_oracle(cuda, vocab, beam, fuse, temperature, normalize, ctc_w, lm_w, lazy):
    from e2e_asr_pytorch_b200 import BeamDecoder, synth
    asr, lm, lm_path, lm_cfg = _models(vocab=vocab)
    emb = synth.build_emb(vocab, asr.dec_dim, 30, fuse=fuse, temperature=temperature, fuse_normalize=normalize, seed=4)
    lens = [64, 120, 92, 148]
    max_ratio = 0.2
    feat, fl = synth.padded_batch(list(range(len(lens))), lens)
    dec = BeamDecoder(asr, emb, beam, 0.01, max_ratio, lm_path=lm_path, lm_config=lm_cfg, lm_weight=lm_w, ctc_weight=ctc_w).to(cuda)
    dec.lazy_prefix = lazy
    out = dec.decode_batch(feat.to(cuda), fl.to(cuda))
    same = ties = 0
    for k, n in enumerate(lens):
        ora = _oracle_nbest(asr, lm, emb, feat[k], n, beam, lm_w, ctc_w, max_ratio)
        assert len(out[k]) == len(ora)

        def rescore(ids, k=k, n=n):
            return _oracle_nbest(asr, lm, emb, feat[k], n, beam, lm_w, ctc_w, max_ratio, force=ids)[0].mean_score()
        s, t = _compare(out[k], ora, "emb fusion V %d beam %d fuse %s temp %s norm %s utt %d" % (vocab, beam, fuse, temperature,
                                                                                               normalize, k), rescore=rescore)
        same, ties = same + s, ties + t
    print("emb fusion V %d beam %d fuse %s temp %s norm %s ctc %.1f lm %.1f: identical 1-best %d/%d, ties %d"
          % (vocab, beam, fuse, temperature, normalize, ctc_w, lm_w, same, len(lens), ties))
    assert same >= len(lens) - 1


def test_dropin_calls_with_embedding_fusion_agree_with_decode_batch(cuda):
    from e2e_asr_pytorch_b200 import BeamDecoder, synth
    asr, lm, lm_path, lm_cfg = _models()
    emb = synth.build_emb(31, asr.dec_dim, 30, fuse=-2, temperature=-2, seed=4)
    lens = [64, 120, 92]
    feat, fl = synth.padded_batch(list(range(len(lens))), lens)
    dec = BeamDecoder(asr, emb, 4, 0.01, 0.2, lm_path=lm_path, lm_config=lm_cfg, lm_weight=0.3, ctc_weight=0.5).to(cuda)
    both = dec.decode_batch(feat.to(cuda), fl.to(cuda))
    host = dec.decode_batch_from_host(feat.pin_memory(), fl, cuda)
    for k, n in enumerate(lens):
        one = dec(feat[k:k + 1, :n].to(cuda), fl[k:k + 1].to(cuda))
        assert [h.outIndex for h in one] == [h.outIndex for h in both[k]], k
        assert [h.outIndex for h in host[k]] == [h.outIndex for h in both[k]], k
        assert [float(h.avgScore()) for h in host[k]] == [float(h.avgScore()) for h in both[k]], k
