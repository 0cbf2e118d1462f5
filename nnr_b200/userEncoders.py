"""Drop-in ``UserEncoder`` / ``SUE`` (reference userEncoders.py:12-98) on the nnr_b200 CUDA path."""
import math

import torch
import torch.nn as nn

from . import engine
from .layers import GCN, ScaledDotProduct_CandidateAttention
from .newsEncoders import NewsEncoder


class UserEncoder(nn.Module):
    def __init__(self, news_encoder: NewsEncoder, config):
        super().__init__()
        self.news_embedding_dim = news_encoder.news_embedding_dim
        self.news_encoder = news_encoder
        self.device = torch.device('cuda')
        self.auxiliary_loss = None

    def forward(self, *args):
        raise Exception('Function forward must be implemented at sub-class')


class SUE(UserEncoder):
    hca = True
    use_gcn = True

    def __init__(self, news_encoder: NewsEncoder, config):
        super().__init__(news_encoder, config)
        self.attention_dim = max(config.attention_dim, self.news_embedding_dim // 4)
        self.proxy_node_embedding = nn.Parameter(torch.zeros([config.category_num, self.news_embedding_dim]))
        self.gcn = GCN(in_dim=self.news_embedding_dim, out_dim=self.news_embedding_dim, hidden_dim=self.news_embedding_dim,
                       num_layers=config.gcn_layer_num, dropout=config.dropout_rate / 2, residual=not config.no_gcn_residual,
                       layer_norm=config.gcn_layer_norm)
        self.intraCluster_K = nn.Linear(self.news_embedding_dim, self.attention_dim, bias=False)
        self.intraCluster_Q = nn.Linear(self.news_embedding_dim, self.attention_dim, bias=True)
        self.clusterFeatureAffine = nn.Linear(self.news_embedding_dim, self.news_embedding_dim, bias=True)
        self.interClusterAttention = ScaledDotProduct_CandidateAttention(self.news_embedding_dim, self.news_embedding_dim, self.attention_dim)
        self.dropout_rate = config.dropout_rate
        self.dropout = nn.Dropout(p=config.dropout_rate, inplace=True)
        self.dropout_ = nn.Dropout(p=config.dropout_rate, inplace=False)
        self.category_num = config.category_num + 1  # extra one category index for padding news
        self.max_history_num = config.max_history_num
        self.gcn_layer_num = config.gcn_layer_num
        self.gcn_residual = not config.no_gcn_residual
        self.gcn_layer_norm = bool(config.gcn_layer_norm)
        self.attention_scalar = math.sqrt(float(self.attention_dim))

    def initialize(self):
        self.gcn.initialize()
        nn.init.zeros_(self.proxy_node_embedding)
        nn.init.xavier_uniform_(self.intraCluster_K.weight)
        nn.init.xavier_uniform_(self.intraCluster_Q.weight)
        nn.init.zeros_(self.intraCluster_Q.bias)
        nn.init.xavier_uniform_(self.clusterFeatureAffine.weight, gain=nn.init.calculate_gain('relu'))
        nn.init.zeros_(self.clusterFeatureAffine.bias)
        self.interClusterAttention.initialize()

    def _params(self):
        cached = self.__dict__.get('_param_list')      # see newsEncoders.CNE._params
        if cached is None:
            ln = getattr(self, 'gcn_layer_norm', False)
            names = ((engine.sue_param_names(self.gcn_layer_num, ln) if self.hca else engine.sue_wo_hca_param_names(self.gcn_layer_num, ln))
                     if self.use_gcn else engine.sue_wo_gcn_param_names())
            sd = {k: v for k, v in self.named_parameters() if not k.startswith('news_encoder.')}
            cached = [sd[k] for k in names]
            self.__dict__['_param_list'] = cached
        return cached

    def forward(self, user_title_text, user_title_mask, user_title_entity, user_content_text, user_content_mask, user_content_entity,
                user_category, user_subCategory, user_history_mask, user_history_graph, user_history_category_mask,
                user_history_category_indices, user_embedding, candidate_news_representation):
        history_embedding = self.news_encoder(user_title_text, user_title_mask, user_title_entity, user_content_text,
                                              user_content_mask, user_content_entity, user_category, user_subCategory,
                                              user_embedding)                     # [B, H, D]  (its own pairing domain)
        return self.encode_user(history_embedding, user_history_graph, user_history_category_mask,
                                user_history_category_indices, candidate_news_representation)

    def encode_user(self, history_embedding, user_history_graph, user_history_category_mask, user_history_category_indices,
                    candidate_news_representation):
        """userEncoders.py:73-97 given the already encoded history (Model.forward encodes candidates and history
        with one CNE schedule, see CNE.encode_calls)."""
        user_history_category_mask[:, -1] = 1                                    # userEncoders.py:73 (in place, like the reference)
        return engine.SUEFunction.apply(self._meta(), history_embedding, candidate_news_representation, user_history_graph,
                                        user_history_category_mask, user_history_category_indices.long(), *self._params())

    def _meta(self):
        return dict(hca=self.hca, gcn=self.use_gcn, gcn_layers=self.gcn_layer_num, residual=self.gcn_residual,
                    layer_norm=getattr(self, 'gcn_layer_norm', False),
                    training=self.training, p_drop=float(self.dropout_rate), category_num=self.category_num - 1 if self.hca else 0)

    def user_side(self, history_embedding, user_history_graph, user_history_category_mask, user_history_category_indices,
                  factored=False):
        """inference (eval mode): the part of encode_user that depends on the history alone, computed once for every tile of
        candidates scored against these users with ``tile_scores`` (``tile_scores_factored`` with ``factored=True``;
        engine.sue_user_side)"""
        user_history_category_mask[:, -1] = 1
        return engine.sue_user_side(self._meta(), history_embedding, user_history_graph, user_history_category_mask,
                                    user_history_category_indices.long(), *self._params(), factored=factored)

    def tile_scores(self, user_side, candidate_news_representation):
        """click scores [B, T] of candidates [B, T, D] for the users of ``user_side``: equal, bit for bit, to
        RowDot(encode_user(...), candidates) on the same inputs (engine.sue_tile_scores)"""
        return engine.sue_tile_scores(self._meta(), user_side, candidate_news_representation, *self._params())

    def tile_explain(self, user_side, candidate_news_representation):
        """tile_scores and the explanation of each score: (scores [B, T], alpha [B, T, H], beta [B, T, C1],
        beta * (f . cand) [B, T, C1]), the model's own attention weights and per-cluster score terms; SUE_wo_HCA:
        (scores, its pooled attention's weights [B, T, H], None, None) (engine.sue_tile_explain)"""
        return engine.sue_tile_explain(self._meta(), user_side, candidate_news_representation, *self._params())

    def tile_scores_factored(self, user_side, candidate_rows):
        """click scores [B, T] of candidates [T, D] shared by the users of ``user_side(..., factored=True)``, through the
        factored cluster tail: equal to tile_scores on the expanded candidates in real arithmetic, not bit for bit
        (engine.sue_tile_scores_factored)"""
        return engine.sue_tile_scores_factored(self._meta(), user_side, candidate_rows, *self._params())

    def packed_scores_factored(self, user_side, candidate_rows, row_off, out):
        """click scores of per-user candidate lists for the users of ``user_side(..., factored=True)``: user b's candidates
        are candidate_rows [row_off[b], row_off[b + 1]) (row_off [B + 1] int32 on the device), the score of its j-th goes
        to out[b, j] and the rest of out is left as it is; returns out.  The factored cluster tail, as in
        tile_scores_factored (engine.sue_packed_scores_factored)"""
        return engine.sue_packed_scores_factored(self._meta(), user_side, candidate_rows, row_off, out, *self._params())

    def packed_explain_factored(self, user_side, candidate_rows, row_off, out, alpha, beta, contrib):
        """packed_scores_factored that also writes the explanation of each score: alpha [B, n, H], beta and
        beta * (f . cand) [B, n, C1], past the counts left as they are; returns (out, alpha, beta, contrib)
        (engine.sue_packed_explain_factored)"""
        return engine.sue_packed_explain_factored(self._meta(), user_side, candidate_rows, row_off, out, alpha, beta, contrib,
                                                  *self._params())
