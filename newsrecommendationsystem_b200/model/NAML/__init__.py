"""NAML (reference src/model/NAML/__init__.py:7-93): CNN text encoders over title and abstract, element encoders over
category / subcategory, a final additive attention over those vectors, and an additive-attention user encoder.  Same
constructor, methods, sub-module names and state_dict keys as the reference; every arithmetic step runs in
libnrms_b200 (sm_100a).  forward / forward_rows / get_* are Exp1's: the news encoder is row-wise, so the 1+K+N batches
are encoded in one launch sequence."""
from .news_encoder import NewsEncoder
from .user_encoder import UserEncoder
from ..Exp1 import Exp1
from ..general.click_predictor.dot_product import DotProductClickPredictor


class NAML(Exp1):
    def __init__(self, config, pretrained_word_embedding=None):
        super(Exp1, self).__init__()
        self.config = config
        self.news_encoder = NewsEncoder(config, pretrained_word_embedding)
        self.user_encoder = UserEncoder(config)
        self.click_predictor = DotProductClickPredictor()
