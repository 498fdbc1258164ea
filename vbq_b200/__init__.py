"""vbq_b200 — B200-native implementation of VBQ's per-coordinate rate-distortion quantization path
(reference: mandt-lab/vbq, img-compression/quantizer.py and the word-embedding notebook).

Importing the package loads libvbq_b200.so; if it has not been built this raises (no CPU fallback)."""
from . import _lib

_lib.load()

from . import ops, utils, sharding, serialize                        # noqa: E402
from .quantizer import ChannelwisePriorCDFQuantizer                  # noqa: E402
from .learned_prior import BMSHJ2018Prior                            # noqa: E402
from .vae_models import StandardGaussianPrior, FactoredGaussianPrior, GaussianVAE   # noqa: E402
from .word_embeddings import GaussianCodebook, CompressedEmbedding   # noqa: E402
from .word_embeddings import ranks, analogy_ranks, analogy_metrics   # noqa: E402
from .evaluation import evaluate_compression_quantizer               # noqa: E402

__all__ = ["ops", "utils", "sharding", "serialize", "ChannelwisePriorCDFQuantizer", "BMSHJ2018Prior",
           "StandardGaussianPrior", "FactoredGaussianPrior", "GaussianVAE", "GaussianCodebook", "CompressedEmbedding",
           "ranks", "analogy_ranks", "analogy_metrics", "evaluate_compression_quantizer"]
