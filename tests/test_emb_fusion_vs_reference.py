"""Live pin of the embedding-fusion restatements against the UNMODIFIED reference (src/plugin.py and src/decode.py from
/root/reference): model.EmbeddingRegularizer loads into and from the reference's class and gives its log-probs bit for
bit on the CPU, and tests/_emb_fusion_oracle.py reproduces the reference BeamDecoder's N-best.  Skipped where the
reference tree is absent."""
import copy
import inspect
import sys
import types

import numpy as np
import pytest
import torch

from oracle import refload

pytestmark = pytest.mark.skipif(not refload.available(), reason="/root/reference not present")

CASES = [(0.3, 2.0, False), (-1, -1, True), (-2, -2, False), (-2, -2, True)]


def _load_plugin_class():
    """The reference's ``src.plugin.EmbeddingRegularizer`` from the live tree.  Its imports that decoding with a given
    table does not use are stood in for while it is imported: ``src.bert_embedding`` (pytorch_pretrained_bert is absent)
    and, where sentencepiece is missing, ``src.text``."""
    refload.load(staged=False)                       # the live tree on sys.path, matplotlib stub in place
    stubs = {"src.bert_embedding": {"BertEmbeddingPredictor": None}}
    try:
        import sentencepiece  # noqa: F401
    except ImportError:
        stubs["src.text"] = {"load_text_encoder": None}
    added = []
    for name, attrs in stubs.items():
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__dict__.update(attrs)
            sys.modules[name] = m
            added.append(name)
    try:
        from src.plugin import EmbeddingRegularizer
    finally:
        for name in added:
            sys.modules.pop(name, None)
    return EmbeddingRegularizer


def _reference_plugin(vocab, dec_dim, table, fuse, temperature, normalize):
    """The reference's EmbeddingRegularizer with ``table`` as its (fastText) embedding table."""
    cls = _load_plugin_class()
    mod = inspect.getmodule(cls)
    tok = types.SimpleNamespace(vocab_size=vocab)
    load = getattr(mod, "load_embedding", None)
    mod.load_embedding = lambda *a, **k: table.numpy().copy()
    try:
        kw = dict(tokenizer=tok, dec_dim=dec_dim, enable=True, src="unused", distance="CosEmb", weight=1.0, fuse=fuse,
                  temperature=temperature, freeze=True, fuse_normalize=normalize, dropout=0.0, bert=None)
        params = inspect.signature(cls.__init__).parameters
        emb = cls(**{k: v for k, v in kw.items() if k in params})
    finally:
        if load is not None:
            mod.load_embedding = load
    return emb.eval()


@pytest.mark.parametrize("fuse,temperature,normalize", CASES)
def test_module_loads_both_ways_and_matches_the_reference_bit_for_bit(fuse, temperature, normalize):
    from e2e_asr_pytorch_b200 import synth
    mine = synth.build_emb(31, 20, 30, fuse=fuse, temperature=temperature, fuse_normalize=normalize, seed=5)
    ref = _reference_plugin(31, 20, mine.emb_table.weight.detach(), fuse, temperature, normalize)
    ref.load_state_dict(mine.state_dict())
    back = copy.deepcopy(mine)
    back.load_state_dict(ref.state_dict())
    g = torch.Generator().manual_seed(1)
    x, y = torch.randn(5, 20, generator=g), 4 * torch.randn(5, 31, generator=g)
    with torch.no_grad():
        want = ref(x, y, return_loss=False)[1]
        assert torch.equal(mine(x, y, return_loss=False)[1], want)
        assert torch.equal(back(x, y, return_loss=False)[1], want)


@pytest.mark.parametrize("beam", [2, 8])
def test_oracle_emb_branch_reproduces_the_reference_decoder(tmp_path, beam):
    import yaml
    from tests import _emb_fusion_oracle as EO
    from e2e_asr_pytorch_b200 import synth
    ref = refload.load()
    torch.set_num_threads(4)
    mine = synth.build_asr(31, synth.TINY_ASR_CFG, seed=0, peak=4.0)
    rasr = ref.ASR(synth.FEAT_DIM, 31, True, **copy.deepcopy(synth.TINY_ASR_CFG)).eval()
    rasr.load_state_dict(mine.state_dict())
    emb = synth.build_emb(31, mine.dec_dim, 30, fuse=-2, temperature=-2, seed=4)
    remb = _reference_plugin(31, mine.dec_dim, emb.emb_table.weight.detach(), -2, -2, False)
    remb.load_state_dict(emb.state_dict())
    lm = synth.build_lm(31, synth.TINY_LM_CFG, seed=1)
    torch.save({"model": lm.state_dict()}, str(tmp_path / "lm.pth"))
    yaml.safe_dump({"model": synth.TINY_LM_CFG}, open(str(tmp_path / "lm.yaml"), "w"))
    lm_w = 0.3 if beam == 8 else 0.0
    n = 92
    feat, fl = synth.utterance(7, n)[None], torch.LongTensor([n])
    rdec = ref.BeamDecoder(rasr, remb, beam, 0.01, 0.2, lm_path=str(tmp_path / "lm.pth"), lm_config=str(tmp_path / "lm.yaml"),
                           lm_weight=lm_w, ctc_weight=0.5)
    with torch.no_grad():
        want = rdec(feat, fl)
        got = EO.decode_utterance(mine, emb, feat, fl, beam, 0.01, 0.2, lm=lm if lm_w > 0 else None, lm_weight=lm_w,
                                  ctc_weight=0.5)
    assert len(want) == len(got)
    for a, b in zip(want, got):
        assert a.outIndex == b.ids
        assert np.array_equal(np.array([float(s) for s in a.output_scores]), np.array([float(s) for s in b.scores]))
        assert float(a.avgScore()) == float(b.mean_score())
