"""Configuration objects with the reference's attribute names (reference src/config.py:10-45).

The B200 modules read ONLY attributes the reference modules read (`num_words`,
`word_embedding_dim`, `num_attention_heads`, `query_vector_dim`, `dropout_probability`,
`num_words_title`, `num_clicked_news_a_user`), so a reference `NRMSConfig` object can be passed
unchanged.  Two optional extra attributes are honoured when present:
  precision: "tf32" (tcgen05 tensor cores, default) | "fp32" (CUDA-core reference-exact mode)
  use_layernorm: True adds nn.LayerNorm(300) on the self-attention context of both encoders (the "+LN" of the
      reference README's config-5 row, which has no code in the tree; builder-defined, see DESIGN.md section 1)
"""
import os


class BaseConfig:
    num_epochs = 2
    num_batches_show_loss = 100
    num_batches_validate = 1000
    batch_size = 128
    learning_rate = 0.0001
    num_workers = 4
    num_clicked_news_a_user = 50
    num_words_title = 20
    num_words_abstract = 50
    word_freq_threshold = 1
    entity_freq_threshold = 2
    entity_confidence_threshold = 0.5
    negative_sampling_ratio = 2
    dropout_probability = 0.2
    num_words = 1 + 70975
    num_categories = 1 + 274
    num_entities = 1 + 12957
    num_users = 1 + 50000
    word_embedding_dim = 300
    category_embedding_dim = 100
    entity_embedding_dim = 100
    query_vector_dim = 200


class NRMSConfig(BaseConfig):
    dataset_attributes = {"news": ['title'], "record": []}
    num_attention_heads = 15


class NRMSLNConfig(NRMSConfig):
    """BASELINE configs[4]: NRMS + LayerNorm, trained with AdamW + cosine decay (optim.FusedAdam(adamw=True),
    optim.cosine_lr)."""
    use_layernorm = True


class Exp1Config(BaseConfig):
    """reference src/config.py:99-107"""
    dataset_attributes = {"news": ['category', 'subcategory', 'title'], "record": []}
    num_attention_heads = 15
    ensemble_factor = 1


class NAMLConfig(BaseConfig):
    """reference src/config.py (NAMLConfig): CNN text encoders over title and abstract, element encoders over category
    and subcategory."""
    dataset_attributes = {"news": ['category', 'subcategory', 'title', 'abstract'], "record": []}
    num_filters = 300
    window_size = 3


class LSTURConfig(BaseConfig):
    """reference src/config.py (LSTURConfig): NAML's CNN title encoder plus raw category rows, and a GRU user encoder
    started from (ini) or concatenated with (con) a learned per-user embedding."""
    dataset_attributes = {"news": ['category', 'subcategory', 'title'], "record": ['user', 'clicked_news_length']}
    num_filters = 300
    window_size = 3
    long_short_term_method = 'ini'
    # See paper for more detail
    masking_probability = 0.5


def resolve_mode(config=None, override=None):
    from . import _lib
    name = override or getattr(config, "precision", None) or os.environ.get("NRMS_B200_PRECISION", "tf32")
    if name not in _lib.MODES:
        raise ValueError(f"unknown precision {name!r}; expected one of {sorted(_lib.MODES)}")
    return _lib.MODES[name]
