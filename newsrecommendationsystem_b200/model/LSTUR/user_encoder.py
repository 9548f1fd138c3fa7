"""LSTUR UserEncoder (reference src/model/LSTUR/user_encoder.py) on libnrms_b200: nn.GRU(900, 900 (ini) or 450 (con))
over pack_padded_sequence(clicked_news_vector, clicked_news_length, batch_first=True, enforce_sorted=False), started
from the user vector (ini) or from zero and concatenated with it (con).  One library call, nrms_gru_fwd / _bwd.

As in the reference, the GRU reads rows [0, length) of the history, and the history is left-padded: a user with n
clicks runs over 50 - n padding rows and then the first 2n - 50 clicks, and with n <= 25 only over padding."""
import torch
import torch.nn as nn

from ... import ops
from ...config import resolve_mode


def gru_lengths(clicked_news_length, T):
    """clicked_news_length (integer [B], host or device) as a new host tensor with 0 read as 1 -- what the reference's
    `clicked_news_length[clicked_news_length == 0] = 1` does, without writing into the caller's tensor."""
    lengths = torch.as_tensor(clicked_news_length).detach().reshape(-1).cpu().long()
    if lengths.numel() and (int(lengths.min()) < 0 or int(lengths.max()) > T):
        raise ValueError(f"clicked_news_length must lie in 0..{T}, got [{int(lengths.min())}, {int(lengths.max())}]")
    return lengths.clamp(min=1)


class UserEncoder(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.config = config
        assert int(config.num_filters * 1.5) == config.num_filters * 1.5
        self.gru = nn.GRU(config.num_filters * 3, config.num_filters * 3 if config.long_short_term_method == 'ini'
                          else int(config.num_filters * 1.5))
        self.precision = None

    def _params(self):
        g = self.gru
        return g.weight_ih_l0, g.weight_hh_l0, g.bias_ih_l0, g.bias_hh_l0

    def _finish(self, h, user):
        return h if self.config.long_short_term_method == 'ini' else ops.concat_rows(h, user)

    def forward(self, user, clicked_news_length, clicked_news_vector):
        """
        Args:
            user:
                ini: batch_size, num_filters * 3
                con: batch_size, num_filters * 1.5
            clicked_news_length: batch_size,
            clicked_news_vector: batch_size, num_clicked_news_a_user, num_filters * 3
        Returns:
            (shape) batch_size, num_filters * 3
        clicked_news_length is not written into: lengths of 0 are read as 1 in a copy.
        """
        lengths = gru_lengths(clicked_news_length, clicked_news_vector.shape[1])
        h0 = user if self.config.long_short_term_method == 'ini' else None
        h = ops.gru(clicked_news_vector, lengths, h0, *self._params(), mode=resolve_mode(self.config, self.precision))
        return self._finish(h, user)

    @torch.no_grad()
    def forward_indexed(self, user, clicked_news_length, table, rows):
        """Inference over rows of a news-vector table: table fp32 [n_rows, 900] on the device, rows integer [U, T]
        (host rows are range-checked against the table) -> [U, 900].  The GRU's input projection runs once over the table rows and each step reads its
        sequence's projected row."""
        lengths = gru_lengths(clicked_news_length, rows.shape[1])
        h0 = user if self.config.long_short_term_method == 'ini' else None
        h = ops.gru_indexed(table, rows, lengths, h0, *self._params(),
                            mode=resolve_mode(self.config, self.precision))
        return self._finish(h, user)
