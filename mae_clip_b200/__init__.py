"""mae_clip_b200: B200-native training-loss hot path of ykojima4020/mae_clip.

Drop-in names: ``CLIPModel``, ``ProjectionHead``, ``cross_entropy`` (reference ``CLIP.py`` /
``modules.py``) plus the MAE ops the north_star names (``random_masking``, ``masked_mse_loss``).
Everything runs in ``libmae_clip_b200.so`` (hand-written sm_100a CUDA behind a C ABI); importing
this package never imports the oracle and has no CPU fallback.
"""
from . import config  # noqa: F401
from .CLIP import CLIPModel, cross_entropy  # noqa: F401
from .functional import clip_contrastive_loss, projection_head  # noqa: F401
from .mae import (masked_mse_loss, patchify, random_masking, random_masking_with_ids,  # noqa: F401
                  restore_tokens)
from .inference import (evaluate_retrieval, find_matches, get_image_embeddings, retrieval_ranks,  # noqa: F401
                        retrieval_recall, retrieval_topk, similarity_topk)
from .modules import ImageEncoder, ProjectionHead, TextEncoder  # noqa: F401

__version__ = "0.1.0"
