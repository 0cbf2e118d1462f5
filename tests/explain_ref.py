"""Host reference of the split of SUE's click score over the interest clusters (CorpusScorer.explain).

``sue_explain`` restates ``oracle.nnr_oracle.sue_forward`` (eval mode) with the oracle's own pieces, and returns the
intermediate tensors the forward drops: score = user . cand = sum_c beta_c (f_c . cand).  It runs in any dtype (fp64 for
the exact split, fp32 on the oracle's cached news vectors).
"""
import math

import torch
import torch.nn.functional as F

from oracle.nnr_oracle import gcn_forward, scatter_softmax, scatter_sum


def sue_explain(p, cfg, history_embedding, graph, category_mask, category_indices, candidate, pre='user_encoder.'):
    """(alpha [B,n,H] intra-cluster weights in history order, beta [B,n,C1] inter-cluster weights, f.cand [B,n,C1], user
    [B,n,D]), applying intraCluster_K.bias where the variant has one.  SUE_wo_HCA: (its additive attention's weights
    over the history expanded over the candidates [B,n,H], None, None, user)."""
    B, H, D = history_embedding.shape
    n = candidate.shape[1]
    C1 = cfg.category_num + 1
    category_mask = category_mask.clone()
    category_mask[:, -1] = 1                                                       # userEncoders.py:73
    if cfg.user_encoder == 'SUE_wo_GCN':
        g = history_embedding
    else:
        x0 = torch.cat([history_embedding, p[pre + 'proxy_node_embedding'].unsqueeze(0).expand(B, -1, -1)], dim=1)
        g = (gcn_forward(p, cfg, x0, graph, pre + 'gcn.') + x0)[:, :H, :]
    if cfg.user_encoder == 'SUE_wo_HCA':                                           # layers.py:167-175 without the pooling
        u = torch.tanh(g @ p[pre + 'attention.affine1.weight'].t() + p[pre + 'attention.affine1.bias'])
        w = F.softmax((u @ p[pre + 'attention.affine2.weight'].t()).squeeze(2), dim=1)                   # [B,H]
        user = torch.bmm(w.unsqueeze(1), g).expand(-1, n, -1)
        return w.unsqueeze(1).expand(-1, n, -1), None, None, user
    Au = p[pre + 'intraCluster_K.weight'].shape[0]
    K = g @ p[pre + 'intraCluster_K.weight'].t()
    if (pre + 'intraCluster_K.bias') in p:                                         # SUE_wo_GCN
        K = K + p[pre + 'intraCluster_K.bias']
    Q = candidate @ p[pre + 'intraCluster_Q.weight'].t() + p[pre + 'intraCluster_Q.bias']
    a = torch.einsum('bha,bka->bkh', K, Q) / math.sqrt(float(Au))
    idx = category_indices.unsqueeze(1).expand(-1, n, -1)
    alpha = scatter_softmax(a, idx, 2)                                             # [B,n,H]
    intra = scatter_sum(alpha.unsqueeze(3) * g.unsqueeze(1), idx, 2, C1)           # [B,n,C1,D]
    f = F.relu(intra @ p[pre + 'clusterFeatureAffine.weight'].t() + p[pre + 'clusterFeatureAffine.bias']) + intra
    pa = pre + 'interClusterAttention.'                                            # scaled_dot_candidate_attention
    k = f @ p[pa + 'K.weight'].t()
    q = candidate @ p[pa + 'Q.weight'].t() + p[pa + 'Q.bias']
    logits = torch.einsum('bkca,bka->bkc', k, q) / math.sqrt(float(k.shape[3]))
    beta = F.softmax(logits.masked_fill(category_mask.unsqueeze(1) == 0, -1e9), dim=2)       # [B,n,C1]
    user = torch.einsum('bkc,bkcd->bkd', beta, f)
    return alpha, beta, torch.einsum('bkcd,bkd->bkc', f, candidate), user
