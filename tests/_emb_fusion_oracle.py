"""The per-hypothesis CPU oracle (oracle/beam_oracle.py) for models decoded with the word-embedding fusion plug-in
(src/plugin.py EmbeddingRegularizer, or model.EmbeddingRegularizer).

``decode_utterance`` is ``oracle.beam_oracle.decode_utterance`` with the one branch the reference's BeamDecoder takes
when it holds an ``emb_decoder`` (src/decode.py:~118-122): the attention log-softmax is replaced by the plug-in's fused
log-probs, ``_, cur_prob = self.emb_decoder(d_state, cur_prob, return_loss=False)``, and everything downstream (CTC
candidate pre-prune, CTC / LM blend, <eos> threshold, prune) sees them in its place.  The search steps are
beam_oracle's own helpers.  ``trace`` records also hold the plug-in's emb logits (x_emb @ table^T), for teacher
forcing."""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import beam_oracle as BO
from oracle import ctc_prefix_oracle as cpo

nbest_as_arrays = BO.nbest_as_arrays


def emb_logits(emb_decoder, d_state):
    """x_emb @ table^T of the plug-in (row-normalised operands with fuse_normalize)."""
    x_emb = emb_decoder.emb_net(d_state)
    table = emb_decoder.emb_table.weight
    if emb_decoder.fuse_normalize:
        return F.linear(F.normalize(x_emb, dim=-1), F.normalize(table, dim=-1))
    return F.linear(x_emb, table)


def decode_utterance(asr, emb_decoder, feat, feat_len, beam_size, min_len_ratio, max_len_ratio,
                     lm=None, lm_weight=0.0, ctc_weight=0.0, trace=None, scorer_cls=None, force=None):
    """beam_oracle.decode_utterance (same arguments, same ``force`` rescoring) with the plug-in's fused log-probs."""
    assert feat.shape[0] == 1, "Batchsize == 1 is required for beam search"
    assert asr.enable_att
    use_ctc, use_lm = ctc_weight > 0, lm_weight > 0
    if use_ctc:
        assert asr.ctc_weight > 0, "ASR was not trained with CTC decoder"
        n_cand = int(BO.CTC_BEAM_RATIO * beam_size)
    device = feat.device
    scorer_cls = scorer_cls or cpo.PrefixScorerOracle

    dec_state0 = asr.decoder.init_state(1)
    asr.attention.reset_mem()
    n_in = feat_len.cpu().item()
    max_steps = int(np.ceil(n_in * max_len_ratio))
    min_steps = int(np.ceil(n_in * min_len_ratio))
    keep_att = asr.attention.mode == "loc"

    enc, enc_len = asr.encoder(feat, feat_len)
    scorer, state0 = None, None
    if use_ctc:
        post = F.log_softmax(asr.ctc_layer(enc), dim=-1)
        scorer = scorer_cls(post.detach().cpu().numpy())
        state0 = scorer.init_state()

    live = [BO.Beam([], [], dec_state0, None, None, state0, 0)]
    done = []
    for step in range(max_steps if force is None else len(force)):
        pool = []
        for hyp in live:
            tok_prev = torch.LongTensor([hyp.tokens[-1] if hyp.tokens else 0]).to(device)
            att_prev = hyp.att_map.to(device) if hyp.att_map is not None else None
            lm_prev = hyp.lm_state
            if isinstance(lm_prev, tuple):
                lm_prev = (lm_prev[0].to(device), lm_prev[1].to(device))
            elif lm_prev is not None:
                lm_prev = lm_prev.to(device)
            asr.set_state(hyp.dec_state, att_prev)

            attn, context = asr.attention(asr.decoder.get_query(), enc, enc_len)
            dec_in = torch.cat([asr.pre_embed(tok_prev), context], dim=-1)
            logits, d_state = asr.decoder(dec_in)
            _, score = emb_decoder(d_state, logits, return_loss=False)           # [1, V] fused log-probs
            att_logp = score.squeeze(0)

            cands = psi = new_state = lm_state = None
            rec = None
            if trace is not None:
                rec = {"step": step, "prefix": hyp.ids, "att_logits": logits.detach().clone(),
                       "emb_logits": emb_logits(emb_decoder, d_state).detach().clone()}
            if use_ctc:
                _, cand_t = score.squeeze(0).topk(n_cand, dim=-1)
                cands = cand_t.cpu().tolist()
                psi, new_state = scorer.cheap_compute(hyp.ids, hyp.ctc_state, cands)
                score = BO.blend_ctc(score, cands, psi, hyp.ctc_prob, ctc_weight)
                if rec is not None:
                    rec.update(cands=list(cands), psi=np.array(psi), parent_psi=np.float32(hyp.ctc_prob))
            if use_lm:
                lm_out, lm_state = lm(tok_prev.unsqueeze(1), torch.ones([1]), hidden=lm_prev)
                lm_out = lm_out.squeeze(0)
                score = BO.add_lm(score, lm_out, lm_weight)
                if rec is not None:
                    rec["lm_logits"] = lm_out.detach().clone()

            if force is None:
                top_vals, top_ids = score.squeeze(0).topk(beam_size)
            else:
                top_ids = torch.LongTensor([int(force[step])]).to(device)
                top_vals = score.squeeze(0)[top_ids]
            att_map = asr.attention.att_layer.prev_att.cpu() if keep_att else None
            if rec is not None:
                rec.update(top_ids=top_ids.clone(), top_vals=top_vals.clone(), att_logp=att_logp.detach().clone())
                trace.append(rec)
            closed, children = BO._expand(hyp, top_ids, top_vals, asr.decoder.get_state(), att_map, lm_state,
                                          new_state, psi, cands, att_logp)
            if closed is not None and step >= min_steps:
                done.append(closed)
                if beam_size == 1:
                    return done
            pool.extend(children)
            if force is not None and closed is not None:
                return [closed]
        live = BO.prune(pool, beam_size)

    if force is not None:
        return live
    done += live
    done.sort(key=lambda b: b.mean_score(), reverse=True)
    return done[:beam_size]
