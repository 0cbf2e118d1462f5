"""Ablation variants that run through the same kernels (reference variantEncoders.py:263-339, 393-419)."""
import torch.nn as nn

from .layers import GCN, Attention, ScaledDotProduct_CandidateAttention
from .newsEncoders import CNE
from .userEncoders import SUE, UserEncoder


class CNE_wo_CA(CNE):
    """CNE without cross attention: output [title_self | content_self]; gate weights Xavier with gain 1."""
    cross_attention = False
    gate_gain = None


class CNE_wo_CS(CNE):
    """CNE without the cross-selective gate (variantEncoders.py:190-260): both attentions read the LSTM states."""
    selective_gate = False


class CNE_Title(CNE):
    """title LSTM + self attention only (variantEncoders.py:14-55): output [title_self | category | subCategory]"""
    modalities = ('title',)
    cross_attention = False
    selective_gate = False


class CNE_Content(CNE):
    """abstract LSTM + self attention only (variantEncoders.py:58-99)"""
    modalities = ('content',)
    cross_attention = False
    selective_gate = False


class SUE_wo_GCN(UserEncoder):
    """SUE without the graph convolution (variantEncoders.py:342-390): the hierarchical cluster attention runs on the
    history embedding itself; the graph input is ignored.  intraCluster_K has a bias in this variant."""
    hca = True
    use_gcn = False
    _params = SUE._params
    forward = SUE.forward
    encode_user = SUE.encode_user
    _meta, user_side, tile_scores = SUE._meta, SUE.user_side, SUE.tile_scores
    tile_scores_factored, packed_scores_factored = SUE.tile_scores_factored, SUE.packed_scores_factored
    tile_explain, packed_explain_factored = SUE.tile_explain, SUE.packed_explain_factored

    def __init__(self, news_encoder, config):
        super().__init__(news_encoder, config)
        import math
        self.attention_dim = max(config.attention_dim, self.news_embedding_dim // 4)
        self.intraCluster_K = nn.Linear(self.news_embedding_dim, self.attention_dim, bias=True)
        self.intraCluster_Q = nn.Linear(self.news_embedding_dim, self.attention_dim, bias=True)
        self.clusterFeatureAffine = nn.Linear(self.news_embedding_dim, self.news_embedding_dim, bias=True)
        self.interClusterAttention = ScaledDotProduct_CandidateAttention(self.news_embedding_dim, self.news_embedding_dim, self.attention_dim)
        self.dropout_rate = config.dropout_rate
        self.dropout = nn.Dropout(p=config.dropout_rate, inplace=True)
        self.category_num = config.category_num + 1
        self.max_history_num = config.max_history_num
        self.gcn_layer_num = 0
        self.gcn_residual = True
        self.attention_scalar = math.sqrt(float(self.attention_dim))

    def initialize(self):
        nn.init.xavier_uniform_(self.intraCluster_K.weight)
        nn.init.zeros_(self.intraCluster_K.bias)
        nn.init.xavier_uniform_(self.intraCluster_Q.weight)
        nn.init.zeros_(self.intraCluster_Q.bias)
        nn.init.xavier_uniform_(self.clusterFeatureAffine.weight, gain=nn.init.calculate_gain('relu'))
        nn.init.zeros_(self.clusterFeatureAffine.bias)
        self.interClusterAttention.initialize()


class SUE_wo_HCA(UserEncoder):
    """GCN + plain additive attention over the history rows (no mask), repeated over candidates."""
    hca = False
    use_gcn = True
    _params = SUE._params
    forward = SUE.forward
    encode_user = SUE.encode_user
    _meta, user_side, tile_scores = SUE._meta, SUE.user_side, SUE.tile_scores
    tile_scores_factored, packed_scores_factored = SUE.tile_scores_factored, SUE.packed_scores_factored
    tile_explain, packed_explain_factored = SUE.tile_explain, SUE.packed_explain_factored

    def __init__(self, news_encoder, config):
        super().__init__(news_encoder, config)
        import torch
        self.max_history_num = config.max_history_num
        self.proxy_node_embedding = nn.Parameter(torch.zeros([config.category_num, self.news_embedding_dim]))
        self.gcn = GCN(in_dim=self.news_embedding_dim, out_dim=self.news_embedding_dim, hidden_dim=self.news_embedding_dim,
                       num_layers=config.gcn_layer_num, dropout=config.dropout_rate / 2, residual=not config.no_gcn_residual,
                       layer_norm=config.gcn_layer_norm)
        self.attention = Attention(self.news_embedding_dim, config.attention_dim)
        self.dropout_rate = config.dropout_rate
        self.dropout_ = nn.Dropout(p=config.dropout_rate, inplace=False)
        self.gcn_layer_num = config.gcn_layer_num
        self.gcn_residual = not config.no_gcn_residual
        self.gcn_layer_norm = bool(config.gcn_layer_norm)

    def initialize(self):
        nn.init.zeros_(self.proxy_node_embedding)
        self.gcn.initialize()
        self.attention.initialize()
