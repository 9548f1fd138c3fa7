"""Exp1 (reference src/model/Exp1/__init__.py:7-80): NRMS's text encoder over the title (and abstract), element
encoders over category / subcategory, a final additive attention over those vectors, and a user encoder with a
position embedding.  Same constructor, methods, sub-module names and state_dict keys as the reference; every
arithmetic step runs in libnrms_b200 (sm_100a)."""
import torch

from .news_encoder import NewsEncoder
from .user_encoder import UserEncoder
from ..general.click_predictor.dot_product import DotProductClickPredictor


class Exp1(torch.nn.Module):
    def __init__(self, config, pretrained_word_embedding=None):
        super().__init__()
        self.config = config
        self.news_encoder = NewsEncoder(config, pretrained_word_embedding)
        self.user_encoder = UserEncoder(config)
        self.click_predictor = DotProductClickPredictor()

    def set_precision(self, name):
        """"tf32" (tcgen05) or "fp32" (CUDA cores, reference-exact)."""
        self.news_encoder.precision = name
        self.user_encoder.precision = name
        return self

    def forward(self, candidate_news, clicked_news):
        """candidate_news: [{"category": B, "subcategory": B, "title": B x L, ...}] * (1+K); clicked_news: the same * N
        -> click_probability B x (1+K).

        The reference runs the news encoder 1+K+N times (:36-41); the encoder is row-wise, so every attribute is
        stacked first and the 1+K+N batches are encoded in one launch sequence."""
        n_cand = len(candidate_news)
        items = list(candidate_news) + list(clicked_news)
        merged = {name: torch.stack([x[name] for x in items], dim=1) for name in self.news_encoder.attributes()}
        B, T = next(iter(merged.values())).shape[:2]
        flat = {name: v.reshape(B * T, *v.shape[2:]) for name, v in merged.items()}
        vec = self.news_encoder(flat).view(B, T, -1)
        user_vector = self.user_encoder(vec[:, n_cand:])
        return self.click_predictor(vec[:, :n_cand], user_vector)

    def forward_rows(self, news_table, cand_rows, hist_rows):
        """Index-only minibatch: news_table {attribute: device column} with N + 1 rows (title [N+1, num_words_title],
        abstract [N+1, num_words_abstract], category / subcategory [N+1]; row N is the pad, as
        NewsTable.token_table_with_pad builds it),
        cand_rows [B, 1+K] and hist_rows [B, N_clicked] news-row indices -> logits [B, 1+K]."""
        B, n_cand = cand_rows.shape
        dev = next(iter(news_table.values())).device
        rows = torch.cat([cand_rows.to(dev, non_blocking=True), hist_rows.to(dev, non_blocking=True)], dim=1)
        vec = self.news_encoder.forward_rows(news_table, rows.reshape(-1).long()).view(B, rows.shape[1], -1)
        user_vector = self.user_encoder(vec[:, n_cand:])
        return self.click_predictor(vec[:, :n_cand], user_vector)

    def get_news_vector(self, news):
        """news: {"title": B x L, "category": B, ...} -> B x word_embedding_dim"""
        return self.news_encoder(news)

    def get_user_vector(self, clicked_news_vector):
        """clicked_news_vector: B x N x word_embedding_dim -> B x word_embedding_dim"""
        return self.user_encoder(clicked_news_vector)

    def get_prediction(self, news_vector, user_vector):
        """news_vector: C x X, user_vector: X -> C"""
        return self.click_predictor(news_vector.unsqueeze(dim=0), user_vector.unsqueeze(dim=0)).squeeze(dim=0)
