"""LSTUR (reference src/model/LSTUR/__init__.py): a CNN title encoder plus raw category rows (900-wide news vectors), a
GRU user encoder over the click history started from (ini) or concatenated with (con) a learned per-user embedding,
and the dot-product click predictor.  Same constructor, methods, sub-module names and state_dict keys as the reference;
every arithmetic step runs in libnrms_b200 (sm_100a)."""
import torch
import torch.nn as nn

from ... import ops
from .news_encoder import NewsEncoder, _check_ids
from .user_encoder import UserEncoder
from ..general.click_predictor.dot_product import DotProductClickPredictor
from ..Exp1.news_encoder import TextEncoder as _Exp1TextEncoder


class LSTUR(nn.Module):
    def __init__(self, config, pretrained_word_embedding=None):
        super().__init__()
        self.config = config
        self.news_encoder = NewsEncoder(config, pretrained_word_embedding)
        self.user_encoder = UserEncoder(config)
        self.click_predictor = DotProductClickPredictor()
        assert int(config.num_filters * 1.5) == config.num_filters * 1.5
        self.user_embedding = nn.Embedding(
            config.num_users,
            config.num_filters * 3 if config.long_short_term_method == 'ini' else int(config.num_filters * 1.5),
            padding_idx=0)
        self._masking_calls = 0
        self.dropout_seed = 0x1057

    _seed = _Exp1TextEncoder._seed

    def set_precision(self, name):
        """"tf32" (tcgen05) or "fp32" (CUDA cores, reference-exact)."""
        self.news_encoder.precision = name
        self.user_encoder.precision = name
        return self

    def _user(self, user, masked):
        """user_embedding(user), under F.dropout2d(p=masking_probability) in training when `masked`: whole user rows
        are zeroed with probability p and the others scaled by 1 / (1 - p)."""
        _check_ids(user, self.user_embedding.num_embeddings, "user")
        user = torch.as_tensor(user).to(self.user_embedding.weight.device, non_blocking=True)
        p = float(self.config.masking_probability) if (masked and self.training) else 0.0
        offset = 0
        if p > 0.0:
            offset = self._masking_calls
            self._masking_calls += user.numel()
        return ops.embedding_rows(user, self.user_embedding.weight, padding_idx=0, dropout_p=p, seed=self._seed(),
                                  offset=offset)

    def forward(self, user, clicked_news_length, candidate_news, clicked_news):
        """
        Args:
            user: batch_size,
            clicked_news_length: batch_size,
            candidate_news: [{"category": B, "subcategory": B, "title": B x num_words_title}] * (1 + K)
            clicked_news: the same * num_clicked_news_a_user
        Returns:
            click_probability: batch_size, 1 + K
        The reference encodes the 1 + K + N news batches one by one; the encoder is row-wise, so they are stacked
        and encoded in one launch sequence."""
        n_cand = len(candidate_news)
        items = list(candidate_news) + list(clicked_news)
        merged = {name: torch.stack([x[name] for x in items], dim=1) for name in ("category", "subcategory", "title")}
        B, T = merged["title"].shape[:2]
        flat = {name: v.reshape(B * T, *v.shape[2:]) for name, v in merged.items()}
        vec = self.news_encoder(flat).view(B, T, -1)
        user_vector = self.user_encoder(self._user(user, True), clicked_news_length, vec[:, n_cand:])
        return self.click_predictor(vec[:, :n_cand], user_vector)

    def forward_rows(self, news_table, cand_rows, hist_rows, user, clicked_news_length):
        """Index-only minibatch: news_table {"category": [N+1], "subcategory": [N+1], "title": [N+1, L]} device
        columns (row N the pad), cand_rows [B, 1+K] and hist_rows [B, N_clicked] news-row indices, user [B],
        clicked_news_length [B] -> logits [B, 1+K]."""
        B, n_cand = cand_rows.shape
        dev = news_table["title"].device
        rows = torch.cat([cand_rows.to(dev, non_blocking=True), hist_rows.to(dev, non_blocking=True)], dim=1)
        vec = self.news_encoder.forward_rows(news_table, rows.reshape(-1).long()).view(B, rows.shape[1], -1)
        user_vector = self.user_encoder(self._user(user, True), clicked_news_length, vec[:, n_cand:])
        return self.click_predictor(vec[:, :n_cand], user_vector)

    def get_news_vector(self, news):
        """news: {"category": B, "subcategory": B, "title": B x num_words_title} -> B x num_filters * 3"""
        return self.news_encoder(news)

    def get_user_vector(self, user, clicked_news_length, clicked_news_vector):
        """user: batch_size; clicked_news_length: batch_size; clicked_news_vector: batch_size, num_clicked_news_a_user,
        num_filters * 3 -> batch_size, num_filters * 3.  No masking of the user embedding."""
        return self.user_encoder(self._user(user, False), clicked_news_length, clicked_news_vector)

    def get_prediction(self, news_vector, user_vector):
        """news_vector: candidate_size, X; user_vector: X -> candidate_size"""
        return self.click_predictor(news_vector.unsqueeze(dim=0), user_vector.unsqueeze(dim=0)).squeeze(dim=0)
