"""mot_b200 -- B200-native (sm_100a) byte-mix embedding path of mixture-of-tokenizers.

Host side in Python/PyTorch mirroring the reference's module interfaces; all
compute goes through the C ABI of libmot_b200.so (include/mot_b200.h)."""
from .ops import MixSpec, mot_embed, mot_embed_proj, mot_embed_byte_fc, split_residual, ttb_expand, pull_from_left, pull_from_right, tokens_to_digits, tok_gather, mixout_copy, mixout_split, set_custom_ops, launch_count, reset_launch_count, FP32_EPS  # noqa: F401
from . import _lib  # noqa: F401
from . import data  # noqa: F401
from . import ttb  # noqa: F401
from .modules import MoTEmbedding, MoTProjEmbedding, SptByteMixEmbedding, DigitMixinEmbedding, MoTByteFcEmbedding, MoTSplitResidualEmbedding, TokenValueEmbeddings, MoTValueEmbeddings, RUN_VARIANTS, PROJ_VARIANTS  # noqa: F401
