"""Beams wider than 32 without a GPU: the decoder's beam range, the argument checks of e2e_beam_combine_prune_wide, the
fused prefix step's shape rule (it must launch whatever it calls supported, at every live count) and the memory estimate
at beam 64 against the peak measured on a B200."""
import json
import os

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def _decoder(beam, **kw):
    from e2e_asr_pytorch_b200 import BeamDecoder, synth
    asr = synth.build_asr(31, synth.TINY_ASR_CFG, seed=0)
    return BeamDecoder(asr, None, beam, 0.01, 0.2, **kw)


def test_decoder_accepts_beams_up_to_64():
    for beam in (1, 32, 33, 40, 48, 64):
        assert _decoder(beam, ctc_weight=0.5).beam_size == beam
    for beam in (0, 65, 128):
        with pytest.raises(ValueError, match="1..64"):
            _decoder(beam)


def _combine_args(lib, **over):
    """Arguments of e2e_beam_combine_prune(_wide) for one utterance: every pointer a dummy non-null address unless
    overridden (the checks run before anything is dereferenced)."""
    a = dict(att_logits=8, ld_att=300, att_stats=8, lm_logits=None, ld_lm=0, cand=None, psi=None, U=1, B=48, V=300, C=0, step=0,
             min_len=8, max_len=8, ctc_weight=0.0, lm_weight=0.0, eos_threshold=1.5, flags=0, n_live=8, n_active=8, last_tok=8,
             prefix_len=8, score_sum=8, ctc_prob=8, prev_lane=8, parent_slot=8, hist_tok=8, hist_parent=8, hist_score=8,
             fin_count=8, fin_step=8, fin_parent=8, fin_sum=8, fin_score=8, fin_cap=64, status=None, n_run=0, parent_row=None,
             last_tok64=None, parent_tok=None, stream=None)
    a.update(over)
    return list(a.values())


def test_wide_combine_prune_checks_its_arguments():
    from e2e_asr_pytorch_b200 import _lib as L
    lib = L.load()

    def refused(what, **over):
        assert lib.e2e_beam_combine_prune_wide(*_combine_args(lib, **over)) == -1, over         # E2E_ERR_ARG
        msg = lib.e2e_last_error()
        assert b"e2e_beam_combine_prune_wide" in msg and what in msg, (over, msg)

    for name in ("att_logits", "att_stats", "n_live", "parent_slot", "hist_score", "fin_score"):
        refused(b"null pointer", **{name: None})
    refused(b"lm_logits", flags=L.BEAM_USE_LM)                                 # LM on, no LM logits
    refused(b"cand+psi", flags=L.BEAM_USE_CTC, C=72)                           # CTC on, no candidates
    for bad in (0, 65, -1):
        refused(b"1..64", B=bad)
    refused(b"fin_cap", B=64, fin_cap=63)
    refused(b"fin_cap", B=40, fin_cap=39)
    # the narrow entry keeps its own range
    assert lib.e2e_beam_combine_prune(*_combine_args(lib, B=33)) == -1


def _lazy_layout_total(gather, lut, threads, vp, beam, tile):
    """lazy_smem_layout (csrc/prefix_lazy.cu), restated."""
    up = lambda x, a: (x + a - 1) // a * a
    off = up(65 * 8 * 16 if lut else 0, 128)
    off += 2 * tile * threads * 4 if gather else 4 * tile * vp * 4
    off = up(off, 128)
    off += 2 * (tile + 1) * beam * 8 + 2 * beam * (2 * tile + 2) * 4 + 2 * beam * tile * 8 + 2 * beam * (tile + 1) * 4 + 2 * beam * 4
    off = up(off, 8) + 32
    return up(off, 16)


@pytest.mark.parametrize("vocab", [31, 300, 10000])
def test_prefix_step_supported_exactly_when_a_tile_fits(vocab):
    """Every beam 1..64 with the decoder's candidate count int(1.5 * B): the fused step is supported exactly when it
    needs at most 32 warps per utterance and its 16-frame tile fits in 200 KB with the table log-add-exp (the largest
    layout) — so the launch, which falls back from the 32-frame to the 16-frame tile, never refuses a supported shape.
    With the column-gather form (V = 300, 10000) this includes beams 18-23, whose 32-frame tile does not fit."""
    from e2e_asr_pytorch_b200 import ops
    vp = ops.padded_vocab(vocab)
    gather = vp > 256
    n32_too_big = []
    for beam in range(1, 65):
        c = int(1.5 * beam)
        warps = 2 * ((beam + 7) // 8) + (beam * c + 31) // 32
        fits16 = warps <= 32 and _lazy_layout_total(gather, True, warps * 32, vp, beam, 16) <= 200 * 1024
        assert ops.prefix_step_supported(vocab, beam, c) == fits16, (vocab, beam)
        if warps <= 32 and _lazy_layout_total(gather, True, warps * 32, vp, beam, 32) > 200 * 1024:
            n32_too_big.append(beam)
    if gather:
        assert n32_too_big == list(range(18, 24)) and all(ops.prefix_step_supported(vocab, b, int(1.5 * b)) for b in n32_too_big)
    else:
        assert n32_too_big == []


def test_attention_groups_cover_the_beam():
    from e2e_asr_pytorch_b200.stepper import ATT_MAX_SLOTS, attention_groups
    assert attention_groups(8) == [(0, 8)] and attention_groups(32) == [(0, 32)]
    assert attention_groups(40) == [(0, 20), (20, 40)] and attention_groups(64) == [(0, 32), (32, 64)]
    for beam in range(1, 65):
        g = attention_groups(beam)
        assert g[0][0] == 0 and g[-1][1] == beam and all(a[1] == b[0] for a, b in zip(g, g[1:]))
        assert all(0 < hi - lo <= ATT_MAX_SLOTS for lo, hi in g) and len(g) == -(-beam // ATT_MAX_SLOTS)


def test_estimate_covers_the_measured_beam64_peak():
    """shard.estimate_decode_bytes at beam 64 against the peak allocation of the same decode on a B200
    (tools/bench_wide_beam.py)."""
    from e2e_asr_pytorch_b200 import shard
    rec = json.load(open(os.path.join(ROOT, "profiles", "r07_wide_beam.json")))["memory"]
    est = shard.estimate_decode_bytes(rec["n_utts"], rec["l_max"], rec["vocab"], rec["beam"], rec["n_cand"], **rec["estimate_kwargs"])
    assert est == rec["estimate_bytes"]
    assert est >= rec["peak_bytes"]
