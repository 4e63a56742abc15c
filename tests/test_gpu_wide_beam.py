"""Beams up to 64 on the B200: e2e_beam_combine_prune_wide against the narrow kernel (bit for bit at B <= 32) and
against the oracle's per-step pieces (B = 48, 64), the grouped fused attention at B > 32, and whole decodes against the
plain-C oracle — including beams 18 and 20 at V = 10000 on a small batch, whose fused prefix step takes the 16-frame tile."""
import copy
import types

import numpy as np
import pytest
import torch

from tests._attention_heads_oracle import loc_attention_full_heads
from tests.test_gpu_attention_heads import _inputs
from tests.test_gpu_beam_kernels import (_beam_from, _check_beam, _load_state, _oracle_step, _run_step,
                                         test_beam_combine_prune_hand_made_states, test_beam_kernels_replay_the_oracle_trace)
from tests.test_gpu_decode import _compare, _models, _oracle_nbest_c

pytestmark = pytest.mark.gpu


def _ops():
    from e2e_asr_pytorch_b200 import ops
    return ops


# ---- (3b) wide == narrow, bit for bit, at B <= 32 ------------------------------------------------------------------

def _random_state(ops, rng, U, beam, vocab, n_cand, step, dev):
    """A beam state of U utterances with everything the kernel branches on: few live hypotheses, an idle utterance, equal
    score sums and duplicated logit rows (equal keys across parents), <eos> far above (closes) or near the threshold,
    a top token missing from a parent's candidates (TOKEN_NOT_CAND), min_len gating."""
    n_steps = step + 3
    max_len = torch.tensor([n_steps] * (U - 1) + [step], dtype=torch.int32)        # the last utterance is idle
    min_len = torch.tensor([0, step + 1] + [0] * (U - 2), dtype=torch.int32)[:U]
    buf = ops.BeamBuffers(U, beam, n_cand, n_steps, min_len, max_len, dev)
    live = [beam, max(1, beam // 3)] + [beam] * (U - 2)
    buf.n_live.copy_(torch.tensor(live[:U], dtype=torch.int32))
    buf.n_active.copy_(buf.n_live)
    buf.last_tok.copy_(torch.from_numpy(rng.integers(2, vocab, (U, beam)).astype(np.int32)))
    buf.last_tok64.copy_(buf.last_tok.long())
    buf.prefix_len.fill_(step)
    buf.score_sum.copy_(torch.from_numpy((-rng.integers(1, 12, (U, beam)) * 0.25).astype(np.float32)))     # fp32-exact: ties
    buf.ctc_prob.copy_(torch.from_numpy((-rng.random((U, beam)) * 4).astype(np.float32)))
    att = torch.from_numpy(rng.standard_normal((U * beam, vocab)).astype(np.float32) * 3)
    if beam > 1:
        att[1] = att[0]                                                                 # equal keys
        buf.score_sum[0, 1] = buf.score_sum[0, 0]
    att[2, 1] = att[2].max() + 4.0                                                      # <eos> closes
    att[beam + 0, 1] = att[beam + 0].max() + 4.0                                        # ... but min_len blocks it
    if beam > 3:
        att[3, 1] = att[3].max() - 0.01                                                 # <eos> in the top-k, near the threshold
    lm = torch.from_numpy(rng.standard_normal((U * beam, vocab)).astype(np.float32) * 2)
    return buf, att.to(dev), lm.to(dev)


def _all_arrays(buf):
    names = ("n_live", "n_active", "last_tok", "prefix_len", "score_sum", "ctc_prob", "prev_lane", "parent_slot", "parent_row",
             "last_tok64", "parent_tok", "hist_tok", "hist_parent", "hist_score", "fin_count", "fin_step", "fin_parent",
             "fin_sum", "fin_score", "status")
    return {k: getattr(buf, k).cpu().clone() for k in names}


# with CTC, int(1.5 * B) candidates must exist: beam 32 needs 48 vocabulary entries (the reference cannot run it at V = 31)
@pytest.mark.parametrize("vocab,beam,ctc_w,lm_w", [(v, b, c, l) for v in (31, 300, 10000) for b in (1, 4, 8, 16, 32)
                                                   for c, l in ((0.5, 0.3), (0.0, 0.5), (0.5, 0.0), (0.0, 0.0))
                                                   if c == 0 or int(1.5 * b) <= v])
def test_wide_combine_prune_is_narrow_bit_for_bit(cuda, vocab, beam, ctc_w, lm_w):
    """Three consecutive steps of both entries from the same state and inputs: every output array is equal."""
    ops = _ops()
    U, step = 4, 2
    n_cand = int(1.5 * beam) if ctc_w > 0 else 0
    runs = []
    for narrow_max in (32, 0):                                    # the narrow entry, then the wide one
        rng = np.random.default_rng(vocab * 100 + beam)
        buf, att, lm = _random_state(ops, rng, U, beam, vocab, n_cand, step, cuda)
        for s in range(step, step + 3):
            ops.beam_candidates(att, U, beam, vocab, n_cand, buf.n_active, buf.att_stats, buf.cand)
            if ctc_w > 0:
                if s == step and beam > 1:
                    buf.cand[beam] = buf.cand[beam, 0]            # one distinct candidate: the top-B picks non-candidates
                buf.psi.copy_(torch.from_numpy((-rng.random(tuple(buf.psi.shape)) * 8).astype(np.float32)))
            keep = ops.BEAM_NARROW_MAX
            ops.BEAM_NARROW_MAX = narrow_max
            try:
                ops.beam_combine_prune(buf, att, lm if lm_w > 0 else None, vocab, s, ctc_w, lm_w, 1.5, n_run=U)
            finally:
                ops.BEAM_NARROW_MAX = keep
        runs.append(_all_arrays(buf))
    for k in runs[0]:
        assert torch.equal(runs[0][k], runs[1][k]), k
    if ctc_w > 0 and beam > 1:
        assert int(runs[1]["status"][1]) != 0                     # TOKEN_NOT_CAND was raised, by both
    assert int(runs[1]["fin_count"].sum()) > 0                    # some <eos> closed a hypothesis


# the oracle-replay and hand-made-state cases of test_gpu_beam_kernels, through the wide entry
@pytest.fixture
def wide_everywhere():
    ops = _ops()
    keep = ops.BEAM_NARROW_MAX
    ops.BEAM_NARROW_MAX = 0
    yield
    ops.BEAM_NARROW_MAX = keep


@pytest.mark.parametrize("beam,eos_bias,blank_bias,ctc_w,lm_w,n_frames,min_ratio",
                         [(4, 3.0, 6.0, 0.5, 0.3, 120, 0.01), (4, 4.0, 0.0, 0.0, 0.3, 92, 0.01), (8, 0.0, 0.0, 0.5, 0.5, 92, 0.01),
                          (4, 4.0, 6.0, 0.5, 0.3, 120, 0.08), (16, 2.0, 3.0, 0.5, 0.3, 148, 0.01)])
def test_wide_entry_replays_the_oracle_trace(cuda, wide_everywhere, beam, eos_bias, blank_bias, ctc_w, lm_w, n_frames, min_ratio):
    test_beam_kernels_replay_the_oracle_trace(cuda, beam, eos_bias, blank_bias, ctc_w, lm_w, n_frames, min_ratio)


@pytest.mark.parametrize("case,vocab", [("equal_keys", 31), ("few_live", 31), ("eos_closes", 31), ("eos_boundary_not_closed", 31),
                                        ("min_len_blocks", 31), ("lm_alias", 31), ("all_three", 300), ("lm_alias", 10000),
                                        ("all_three", 10000), ("equal_keys", 10000)])
def test_wide_entry_hand_made_states(cuda, wide_everywhere, case, vocab):
    test_beam_combine_prune_hand_made_states(cuda, case, vocab)


# ---- (3b) at B = 48, 64 against the oracle's per-step pieces ---------------------------------------------------------

@pytest.mark.parametrize("beam", [48, 64])
@pytest.mark.parametrize("vocab", [300, 10000])
@pytest.mark.parametrize("ctc_w,lm_w,n_live", [(0.5, 0.3, None), (0.0, 0.5, None), (0.5, 0.0, 5)])
def test_wide_combine_prune_matches_oracle_step(cuda, beam, vocab, ctc_w, lm_w, n_live):
    ops = _ops()
    rng = np.random.default_rng(beam + vocab)
    step = 3
    n = beam if n_live is None else n_live
    parents = [_beam_from(rng.integers(2, vocab, 3), -rng.integers(1, 8, 3) * 0.125) for _ in range(n)]
    att = torch.from_numpy(rng.standard_normal((n, vocab)).astype(np.float32) * 3)
    lml = torch.from_numpy(rng.standard_normal((n, vocab)).astype(np.float32) * 2)
    att[1] = att[0]
    parents[1] = _beam_from(parents[0].ids, [float(s) for s in parents[0].scores])        # equal keys across two parents
    att[2, 1] = att[2].max() + 4.0                                                         # one parent closes
    n_cand = int(1.5 * beam) if ctc_w > 0 else 0
    cands = psi = None
    if ctc_w > 0:
        # the candidates (3a) picks (at C = 96 of 10000 the CPU's top-k of torch's log-softmax may order near-equal
        # entries differently); the oracle step then scores exactly those
        tmp = ops.BeamBuffers(1, beam, n_cand, 1, torch.tensor([0]), torch.tensor([1]), cuda)
        tmp.n_active.fill_(n)
        pad = torch.zeros((beam, vocab))
        pad[:n] = att
        ops.beam_candidates(pad.to(cuda), 1, beam, vocab, n_cand, tmp.n_active, tmp.att_stats, tmp.cand)
        cands = tmp.cand.cpu()[:n, :n_cand].tolist()
        psi = [(-rng.random(n_cand) * 8 - 1).astype(np.float32) for _ in range(n)]
        for b, hyp in enumerate(parents):
            hyp.ctc_prob = np.float32(-0.5 * (b % 7 + 1))
    buf = ops.BeamBuffers(1, beam, n_cand, step + 2, torch.tensor([0]), torch.tensor([step + 2]), cuda)
    _load_state(buf, parents, step)
    parent_toks = [h.ids[-1] if h.ids else -1 for h in parents]
    live, closed = _oracle_step(parents, att.clone(), lml.clone(), cands, psi, beam, ctc_w, lm_w, step, 0)
    _run_step(ops, buf, att, lml if lm_w > 0 else None, cands, psi, vocab, step, ctc_w, lm_w, cuda)
    _check_beam(buf, live, parent_toks, step, ctc_w)
    assert int(buf.fin_count[0]) == len(closed) >= 1
    assert int(buf.status[0]) == 0


# ---- grouped fused attention at B > 32 -------------------------------------------------------------------------------

def _stepper_like(cuda, key, value, prev, enc_len, conv_w, w_proj, w_e, beam, heads):
    from e2e_asr_pytorch_b200.stepper import attention_groups
    dev = lambda t: t.to(cuda)
    key_t = dev(key).permute(0, 1, 3, 2).contiguous() if heads > 1 else dev(key[:, 0]).transpose(1, 2).contiguous()
    return types.SimpleNamespace(B=beam, _groups=attention_groups(beam), key_t=key_t, value=dev(value),
                                 prev_att=dev(prev if heads > 1 else prev[:, 0]).contiguous(), _enc_len32=dev(enc_len),
                                 _w_conv=dev(conv_w if heads > 1 else conv_w[:, 0]), _w_proj=dev(w_proj), _w_energy=dev(w_e),
                                 _b_energy=0.25, temperature=0.5)


@pytest.mark.parametrize("beam", [40, 64])
@pytest.mark.parametrize("heads", [1, 2])
def test_grouped_attention_matches_restatement_and_one_group_calls(cuda, beam, heads):
    """BatchedStepper._fused_attention at B > 32: within 5e-6 / 2e-5 of the CPU restatement, and the bits of the same
    hypotheses run as separate calls of at most 32 slots (here: groups of 8)."""
    from e2e_asr_pytorch_b200 import ops
    from e2e_asr_pytorch_b200.stepper import BatchedStepper
    n_utts, t_len, dim, n_filt, half, e_dim = 3, 61, 300, 10, 100, 64
    per_head = heads > 1                                                   # H = 2 with v_proj
    key, value, query, enc_len, prev, conv_w, w_proj, w_e = _inputs(n_utts, beam, heads, t_len, dim, n_filt, half, e_dim, per_head, beam + heads)
    want_a, want_c = loc_attention_full_heads(key, value, query, prev, enc_len, conv_w, w_proj, w_e, 0.25, 0.5, beam, per_head)
    st = _stepper_like(cuda, key, value, prev, enc_len, conv_w, w_proj, w_e, beam, heads)
    fn, extra = (ops.attention_loc_heads, (per_head,)) if heads > 1 else (ops.attention_loc_full, ())
    k = n_utts - 1                                                         # n_run: the last utterance is not advanced
    got_a, got_c = BatchedStepper._fused_attention(st, fn, query[:k * beam].to(cuda), k, *extra)
    n = k * beam
    want_a = want_a[:n] if heads > 1 else want_a[:n, 0]
    err_a, err_c = (got_a.cpu() - want_a).abs().max().item(), (got_c.cpu() - want_c[:n]).abs().max().item()
    print("grouped attention B=%d H=%d: max |gpu-restatement| attn %.3g ctx %.3g" % (beam, heads, err_a, err_c))
    assert err_a < 5e-6 and err_c < 2e-5
    st8 = copy.copy(st)
    st8._groups = [(lo, min(beam, lo + 8)) for lo in range(0, beam, 8)]
    a8, c8 = BatchedStepper._fused_attention(st8, fn, query[:k * beam].to(cuda), k, *extra)
    assert torch.equal(a8, got_a) and torch.equal(c8, got_c)


# ---- whole decodes against the plain-C oracle ------------------------------------------------------------------------

def _decode_vs_oracle(cuda, asr, lm, lm_path, lm_cfg, lens, seeds, beam, lm_w, ctc_w, max_ratio, what):
    from e2e_asr_pytorch_b200 import BeamDecoder, synth
    feat, fl = synth.padded_batch(seeds, lens)
    dec = BeamDecoder(asr, None, beam, 0.01, max_ratio, lm_path=lm_path if lm_w > 0 else '', lm_config=lm_cfg if lm_w > 0 else '',
                      lm_weight=lm_w, ctc_weight=ctc_w).to(cuda)
    out = dec.decode_batch(feat.to(cuda), fl.to(cuda))
    same = ties = 0
    for k, n in enumerate(lens):
        ora = _oracle_nbest_c(asr, lm, feat[k], n, beam, lm_w, ctc_w, max_ratio)
        assert len(out[k]) == len(ora)
        s, t = _compare(out[k], ora, "%s utt %d" % (what, k))
        same, ties = same + s, ties + t
    print("%s: identical 1-best %d/%d, ties %d" % (what, same, len(lens), ties))
    assert same + ties == len(lens)
    return dec


@pytest.mark.parametrize("beam", [48, 64])
@pytest.mark.parametrize("lm_w,ctc_w", [(0.3, 0.5), (0.3, 0.0)])
def test_decode_v300_wide_beams_match_oracle(cuda, beam, lm_w, ctc_w):
    asr, lm, lm_path, lm_cfg = _models(vocab=300)
    _decode_vs_oracle(cuda, asr, lm, lm_path, lm_cfg, [120, 92, 64], [0, 1, 2], beam, lm_w, ctc_w, 0.2,
                      "V 300 beam %d lm %.1f ctc %.1f" % (beam, lm_w, ctc_w))


def test_decode_v10000_beam40_matches_oracle(cuda):
    asr, lm, lm_path, lm_cfg = _models(vocab=10000)
    _decode_vs_oracle(cuda, asr, lm, lm_path, lm_cfg, [200, 148], [0, 1], 40, 0.5, 0.5, 0.07, "V 10000 beam 40")


def test_decode_two_head_model_beam40_matches_oracle(cuda):
    from e2e_asr_pytorch_b200 import synth
    cfg = copy.deepcopy(synth.TINY_ASR_CFG)
    cfg["attention"].update({"mode": "loc", "v_proj": True, "num_head": 2})
    asr = synth.build_asr(300, cfg, seed=0, peak=4.0)                  # beam 40 needs more than 40 vocabulary entries
    _, lm, lm_path, lm_cfg = _models(vocab=300)
    dec = _decode_vs_oracle(cuda, asr, lm, lm_path, lm_cfg, [120, 92, 64], [0, 1, 2], 40, 0.3, 0.0, 0.2, "2 heads beam 40")
    assert dec._stepper[2].fused_step


@pytest.mark.parametrize("beam", [18, 20])
def test_decode_v10000_beams_18_20_small_batch(cuda, beam):
    """Beams 18-23 at a subword vocabulary on a batch far below 1500 utterances: the fused prefix step's 32-frame
    column-gather tile does not fit, so it takes the 16-frame tile (before, the decode raised E2E_ERR_UNSUPPORTED)."""
    from e2e_asr_pytorch_b200 import ops
    assert ops.prefix_step_supported(10000, beam, int(1.5 * beam))
    asr, lm, lm_path, lm_cfg = _models(vocab=10000)
    _decode_vs_oracle(cuda, asr, lm, lm_path, lm_cfg, [200, 148, 120], [0, 1, 2], beam, 0.5, 0.5, 0.07, "V 10000 beam %d" % beam)
