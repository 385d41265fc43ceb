"""mdir_b200 -- B200-native (sm_100a) implementation of jenicek/mdir's post-backbone retrieval
hot path behind the reference's own plug-in surface (SURVEY.md section 8).

    layers    GeM / MAC / SPoC / L2N modules + POOLING registry     (cirtorch/layers)
    wrappers  CirMultiscaleAggregation, CirtorchWhiten, whitenapply, RetrievalHead
    clahe     clahe_u8, ChannelClahe / ImageClahe / ApplyClahe ...  (mdir transforms)
    search    rank(), Index, ShardedIndex, ranks_from_scores, topk_from_scores
    qe        alpha-QE / DBA (not in the reference; parity unpinned)
    diffusion Diffusion: re-ranking on a mutual kNN graph of the database; DiffusionTable: its offline table;
              GraphedDiffusion / DiffusionPipeline: either one served from CUDA graphs (not in the reference; parity
              unpinned)
    extract   batched extract_vectors (no per-image sync)            (cirtorch/networks/imageretrievalnet.py)
    evaluate  compute_map / compute_map_and_print on the device      (cirtorch/utils/evaluate.py)
    score     CirDatasetAp replacement + install()

All arithmetic runs in hand-written CUDA kernels (mdir_b200/csrc) reached through the C ABI in
include/mdir_b200.h; there is no CPU or PyTorch fallback -- a missing library raises."""
from ._lib import MdirError, lib  # noqa: F401
from .layers import GeM, MAC, SPoC, L2N, POOLING, gem, mac, spoc, l2n  # noqa: F401
from .wrappers import CirMultiscaleAggregation, CirtorchWhiten, RetrievalHead, whitenapply  # noqa: F401
from .clahe import clahe_u8, image_clahe, ChannelClahe, ImageClahe, ApplyClahe, AddClaheFromRgb, CreateClahedImage  # noqa: F401
from .search import (Index, ShardedIndex, GraphedSearch, SearchPipeline, GraphedRangeSearch, RangePipeline, rank,  # noqa: F401
                     ranks_from_scores, topk_from_scores)
from .diffusion import Diffusion, DiffusionTable, GraphedDiffusion, DiffusionPipeline  # noqa: F401
from .extract import extract_vectors, extract_from_tensors  # noqa: F401
from .evaluate import compute_map, compute_map_and_print  # noqa: F401
from .score import install  # noqa: F401
from .mining import mine_hard_negatives, search_hard_negatives  # noqa: F401
from .whiten_learn import whitenlearn, pcawhitenlearn, gemm_f64  # noqa: F401

__version__ = "0.1.0"
