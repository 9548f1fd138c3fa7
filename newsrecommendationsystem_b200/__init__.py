"""B200-native NRMS hot path (news encoder -> user encoder -> dot-product click predictor).

Drop-in for the reference's `src/model/NRMS` module API; all arithmetic runs in the
hand-written sm_100a library `libnrms_b200.so` through the C-ABI in `include/nrms_b200.h`.
Importing the package does not load CUDA; the first op call does, and raises if the library
is missing (there is no CPU fallback).
"""
from .config import NRMSConfig, NRMSLNConfig, Exp1Config, NAMLConfig, LSTURConfig, BaseConfig  # noqa: F401

__all__ = ["NRMSConfig", "NRMSLNConfig", "Exp1Config", "NAMLConfig", "LSTURConfig", "BaseConfig", "NRMS", "Exp1", "NAML",
           "LSTUR", "NewsEncoder",
           "UserEncoder", "DotProductClickPredictor"]


def __getattr__(name):
    if name == "NRMS":
        from .model.NRMS import NRMS
        return NRMS
    if name == "Exp1":
        from .model.Exp1 import Exp1
        return Exp1
    if name == "NAML":
        from .model.NAML import NAML
        return NAML
    if name == "LSTUR":
        from .model.LSTUR import LSTUR
        return LSTUR
    if name == "NewsEncoder":
        from .model.NRMS.news_encoder import NewsEncoder
        return NewsEncoder
    if name == "UserEncoder":
        from .model.NRMS.user_encoder import UserEncoder
        return UserEncoder
    if name == "DotProductClickPredictor":
        from .model.general.click_predictor.dot_product import DotProductClickPredictor
        return DotProductClickPredictor
    raise AttributeError(name)
