"""CPU restatement of one multi-head location-aware attention step (TEST INFRASTRUCTURE), the checker of
``e2e_attention_loc_heads``.  It follows model.py's ``LocationAwareAttention`` / ``Attention`` with num_head = H at
batch 1 per hypothesis (how the per-hypothesis decode calls them), in the style of
oracle/attention_oracle.py::loc_attention_full, and is itself checked against ``model.Attention`` in
tests/test_attention_heads_host.py.  It lives with the tests rather than in oracle/: the modules there are the
restatements pinned to the reference (tests/test_oracle_vs_reference.py) and kept unchanged while the kernels under
them change, and the multi-head branch has no reference tree here to be pinned against."""
import numpy as np
import torch


def loc_attention_full_heads(key, value, query, prev_att, enc_len, w_conv, w_proj, w_energy, b_energy, temperature, beam,
                             per_head_values):
    """The location features come from ALL H previous alignments (Conv1d H->K, zero padded, no bias) and are shared by
    the heads; each head has its own keys, queries and (with ``per_head_values``) values.
    key [U,H,T,A], value [U,T,E] (shared) or [U,T,H*E], query [N,H*A], prev_att [N,H,T], w_conv [K,H,W]
    -> (attn [N,H,T], ctx [N,H*E], the input of merge_head)."""
    key, value, query, prev_att, w_conv, w_proj, w_energy = (torch.as_tensor(a, dtype=torch.float32) for a in
                                                             (key, value, query, prev_att, w_conv, w_proj, w_energy))
    n, h, t = prev_att.shape
    u_of = torch.arange(n) // beam
    feat = torch.nn.functional.conv1d(prev_att, w_conv, padding=w_conv.shape[2] // 2)        # [N,K,T]
    loc = torch.tanh(feat.transpose(1, 2) @ w_proj.t())                                      # [N,T,A]
    q = query.view(n, h, -1)
    mix = torch.tanh(key[u_of] + q[:, :, None, :] + loc[:, None])                            # [N,H,T,A]
    energy = mix @ w_energy + b_energy                                                       # [N,H,T]
    pad = torch.arange(t)[None, :] >= torch.as_tensor(enc_len).long()[u_of][:, None]
    attn = torch.softmax((energy / temperature).masked_fill(pad[:, None, :], -np.inf), dim=-1)
    if per_head_values:
        val = value.view(value.shape[0], t, h, -1).permute(0, 2, 1, 3)[u_of]                  # [N,H,T,E]
    else:
        val = value[u_of][:, None].expand(n, h, t, value.shape[2])                           # every head: its own utterance
    ctx = (attn[:, :, None, :] @ val).squeeze(2)                                             # [N,H,E]
    return attn, ctx.reshape(n, -1)
