"""Synthetic models, decode settings and utterance sets of the BASELINE configs
(SURVEY.md §8d).  No corpus or checkpoint is reachable, so every measurement and
parity run uses random-init weights of the reference architecture and seeded
Gaussian features; the same builders are used on both sides of every comparison.
"""
import copy

import numpy as np
import torch

from .model import ASR, RNNLM, EmbeddingRegularizer

# Dimensions of config/librispeech_asr.yaml:42-68 with the VGG front end switched
# on (vgg: 1, sample_rate [1,1,1,1] -> 4x time reduction), see SURVEY.md §8d.
ASR_MODEL_CFG = {
    "ctc_weight": 0.5,
    "encoder": {"vgg": 1, "vgg_freq": -1, "vgg_low_filt": -1, "module": "LSTM", "bidirection": True,
                "dim": [320, 320, 320, 320], "dropout": [0.2, 0.2, 0.2, 0.2],
                "layer_norm": [False, False, False, False], "proj": [True, True, True, True],
                "sample_rate": [1, 1, 1, 1], "sample_style": "drop"},
    "attention": {"mode": "loc", "dim": 300, "num_head": 1, "v_proj": False, "temperature": 0.5,
                  "loc_kernel_size": 100, "loc_kernel_num": 10},
    "decoder": {"module": "LSTM", "dim": 300, "layer": 1, "dropout": 0},
}
# config/librispeech_lm.yaml:23-29
LM_MODEL_CFG = {"emb_tying": True, "emb_dim": 1024, "module": "LSTM", "dim": 1024, "n_layers": 4, "dropout": 0.5}
FEAT_DIM = 160          # 80 fbank + delta (librispeech_asr.yaml:13,15)

# Small variant with the same topology for fast CPU tests / golden fixtures.
TINY_ASR_CFG = {
    "ctc_weight": 0.5,
    "encoder": {"vgg": 1, "vgg_freq": -1, "vgg_low_filt": -1, "module": "LSTM", "bidirection": True,
                "dim": [16, 16], "dropout": [0.2, 0.2], "layer_norm": [False, False], "proj": [True, True],
                "sample_rate": [1, 1], "sample_style": "drop"},
    "attention": {"mode": "loc", "dim": 24, "num_head": 1, "v_proj": False, "temperature": 0.5,
                  "loc_kernel_size": 10, "loc_kernel_num": 4},
    "decoder": {"module": "LSTM", "dim": 20, "layer": 1, "dropout": 0},
}
TINY_LM_CFG = {"emb_tying": True, "emb_dim": 32, "module": "LSTM", "dim": 32, "n_layers": 2, "dropout": 0.5}


def build_asr(vocab_size=31, cfg=None, seed=0, feat_dim=FEAT_DIM, peak=1.0):
    """Random-init ASR in eval mode.  ``peak`` > 1 scales the output layers
    (attention speller ``char_trans``, ``ctc_layer`` and nothing else) so that
    hypothesis scores are separated by more than fp32 noise (SURVEY.md §7.2-2);
    the same state dict is loaded on both sides of a comparison."""
    cfg = copy.deepcopy(cfg or ASR_MODEL_CFG)
    torch.manual_seed(seed)
    asr = ASR(feat_dim, vocab_size, True, **cfg).eval()
    if peak != 1.0:
        with torch.no_grad():
            asr.decoder.char_trans.weight.mul_(peak)
            asr.ctc_layer[0].weight.mul_(peak)
    return asr


def build_lm(vocab_size=31, cfg=None, seed=1, peak=1.0):
    cfg = copy.deepcopy(cfg or LM_MODEL_CFG)
    torch.manual_seed(seed)
    lm = RNNLM(vocab_size, **cfg).eval()
    if peak != 1.0:
        with torch.no_grad():
            lm.emb.weight.mul_(peak)
    return lm


def build_emb(vocab_size=31, dec_dim=300, emb_dim=300, fuse=0.5, temperature=1.0, fuse_normalize=False, seed=3,
              perturb=True):
    """Random-init embedding-fusion plug-in (model.EmbeddingRegularizer) in eval mode: an N(0, 1) table [V, E] and the
    default Linear init of emb_net.  ``perturb`` moves the learnable weights away from their init values (seeded): a
    learnable ``fuse_lambda`` to N(0, 1) logits, a learnable scalar ``temp`` to U(0.5, 2), an elementwise ``temp`` to
    U(-0.5, 2) per entry with entry 2 set to -1, so that the ReLU clamps some of them to zero."""
    g = torch.Generator().manual_seed(int(seed))
    table = torch.randn(vocab_size, emb_dim, generator=g)
    torch.manual_seed(seed)
    emb = EmbeddingRegularizer(vocab_size, dec_dim, table=table, fuse=fuse, temperature=temperature,
                               fuse_normalize=fuse_normalize).eval()
    if perturb and emb.apply_fuse:
        with torch.no_grad():
            if emb.fuse_learnable:
                emb.fuse_lambda.copy_(torch.randn(emb.fuse_lambda.shape, generator=g))
            if temperature == -1:
                emb.temp.copy_(0.5 + 1.5 * torch.rand(1, generator=g))
            elif temperature == -2:
                t = -0.5 + 2.5 * torch.rand(vocab_size, generator=g)
                t[min(2, vocab_size - 1)] = -1.0
                emb.temp.copy_(t)
    return emb


def utterance(i, n_frames, feat_dim=FEAT_DIM):
    """Seeded Gaussian features of utterance ``i``: [n_frames, feat_dim] fp32."""
    g = torch.Generator().manual_seed(1000 + int(i))
    return torch.randn(int(n_frames), feat_dim, generator=g)


def devclean_lengths(n_utts=2620, seed=2):
    """Input lengths (frames at 100/s, multiples of 4) with a LibriSpeech
    dev-clean-like duration distribution: log-normal around 6.4 s, clipped to
    [1.5, 33] s (SURVEY.md §8d, cfg2)."""
    rng = np.random.default_rng(seed)
    dur = np.clip(np.exp(rng.normal(np.log(6.4), 0.55, size=n_utts)), 1.5, 33.0)
    return (4 * np.round(25.0 * dur)).astype(np.int64)


def padded_batch(ids, lengths, feat_dim=FEAT_DIM, pin=False):
    """Zero-padded [U, Lmax, D] features + [U] lengths for utterances ``ids``."""
    lmax = int(max(lengths))
    feat = torch.zeros(len(ids), lmax, feat_dim)
    for k, (i, n) in enumerate(zip(ids, lengths)):
        feat[k, :int(n)] = utterance(i, n, feat_dim)
    lens = torch.as_tensor(np.asarray(lengths), dtype=torch.long)
    if pin:
        feat, lens = feat.pin_memory(), lens.pin_memory()
    return feat, lens
