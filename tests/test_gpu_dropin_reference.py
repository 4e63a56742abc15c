"""The drop-in proven through the REFERENCE'S OWN CALLER: ``e2e_asr_pytorch_b200.install()`` patches ``src.decode`` /
``src.ctc`` of the (unmodified) reference, then ``bin/test_asr.py``'s module-level ``beam_decode`` (:159-173) is driven the
way ``Solver.exec`` drives it (:80-82 construction with ``**config['decode']``, :108-109 deep copy inside
``functools.partial``) with a ``src.asr.ASR`` instance — the reference's own model class, not ``model.py`` — on the GPU.

The reference comes from ``oracle/_ref`` (its decode path byte-compiled by ``oracle/ref_stage.py``; built by
``__graft_entry__.build()`` in the build container, shipped with the snapshot) or from ``/root/reference`` where that
exists.  Expected N-best: the per-hypothesis CPU oracle with the same modules.
"""
import copy
import os
from functools import partial

import numpy as np
import pytest
import torch
import yaml

from oracle import refload

# the reference's own code is the caller under test: it is not part of this repository, so without it there is nothing to run
pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not (refload.available() or refload.staged_available()),
                                 reason="the reference's decode path (its source tree or oracle/_ref) is not present")]


def test_install_then_reference_beam_decode_on_the_gpu(cuda, tmp_path):
    from oracle import beam_oracle as BO
    from e2e_asr_pytorch_b200 import synth
    import e2e_asr_pytorch_b200 as P
    from tests.test_gpu_decode import _compare
    ref = refload.load()
    import src.ctc
    import src.decode
    saved = (src.ctc.CTCPrefixScore, src.decode.CTCPrefixScore, src.decode.BeamDecoder, src.decode.Hypothesis)
    try:
        P.install()
        test_asr = refload.load_test_asr(fresh=True)          # imported AFTER install(): `from src.decode import BeamDecoder` (bin/test_asr.py:10)
        assert test_asr.BeamDecoder is P.BeamDecoder and src.decode.CTCPrefixScore is P.CTCPrefixScore

        vocab = 31
        mine = synth.build_asr(vocab, synth.TINY_ASR_CFG, seed=0, peak=4.0)
        rasr = ref.ASR(synth.FEAT_DIM, vocab, True, **copy.deepcopy(synth.TINY_ASR_CFG)).eval()        # the reference's model class
        rasr.load_state_dict(mine.state_dict())
        lm = synth.build_lm(vocab, synth.TINY_LM_CFG, seed=1)
        lm_path, lm_cfg = str(tmp_path / "lm.pth"), str(tmp_path / "lm.yaml")
        torch.save({"model": lm.state_dict()}, lm_path)
        yaml.safe_dump({"model": synth.TINY_LM_CFG}, open(lm_cfg, "w"))
        decode_cfg = {"beam_size": 4, "min_len_ratio": 0.01, "max_len_ratio": 0.2, "lm_path": lm_path, "lm_config": lm_cfg,
                      "lm_weight": 0.3, "ctc_weight": 0.5}
        oracle_asr = copy.deepcopy(rasr)                                                            # stays on the CPU
        decoder = test_asr.BeamDecoder(rasr.cpu(), None, **decode_cfg)                              # bin/test_asr.py:80-81
        assert any("Beam size = 4" in m for m in decoder.create_msg())
        func = partial(test_asr.beam_decode, model=copy.deepcopy(decoder), device=cuda)             # bin/test_asr.py:108-109
        same = ties = 0
        lens = [64, 120, 92]
        for i, n in enumerate(lens):
            feat = synth.utterance(i, n)
            data = (["utt%d" % i], feat[None], torch.LongTensor([n]), torch.LongTensor([[5, 6, 7, 0]]))
            name, hyp_seqs, truth = func(data)                                                      # bin/test_asr.py:159-173
            assert name == "utt%d" % i and truth == [5, 6, 7, 0] and all(isinstance(t, int) for t in hyp_seqs[0])
            with torch.no_grad():
                nb = BO.decode_utterance(oracle_asr, feat[None], torch.LongTensor([n]), 4, 0.01, 0.2, lm=lm, lm_weight=0.3, ctc_weight=0.5)
            want = BO.nbest_as_arrays(nb)
            assert len(hyp_seqs) == len(want)
            hyps = func.keywords["model"](feat[None].to(cuda), torch.LongTensor([n]).to(cuda))      # the Hypothesis objects themselves
            assert [h.outIndex for h in hyps] == hyp_seqs
            s, t = _compare(hyps, want, "drop-in utt %d" % i)
            same, ties = same + s, ties + t
        print("drop-in through bin/test_asr.py::beam_decode with src.asr.ASR: identical 1-best %d/%d, ties %d" % (same, len(lens), ties))
        # the batched entry point with the reference's model object: its encoder is opaque to the stepper (one exact batch-1 call per utterance)
        dec = func.keywords["model"]
        feats, fl = synth.padded_batch([0, 1, 2], lens)
        both = dec.decode_batch(feats.to(cuda), fl.to(cuda))
        for i, n in enumerate(lens):
            one = dec(synth.utterance(i, n)[None].to(cuda), torch.LongTensor([n]).to(cuda))
            assert [h.outIndex for h in one] == [h.outIndex for h in both[i]], i
    finally:
        src.ctc.CTCPrefixScore, src.decode.CTCPrefixScore, src.decode.BeamDecoder, src.decode.Hypothesis = saved
