"""Movie-movie similarity on the GPU.

``factor_cosine_topk`` is config 4 of BASELINE.json: cosine similarity of the (row-normalised)
item factors an ALS run produced, top-k per movie, as a tensor-core GEMM fused with the
selection (csrc/similarity.cu).  The reference has no factor-based similarity -- its
``SimilarMovieFinder`` (python/full_data/build_similar_movies_db.py:21-221) scores co-rating
vectors -- so this entry point is an extension; its results are bit-exact against the written-down
CPU definition in oracle/ls_oracle.c (ids and scores).
"""
import ctypes

import numpy

from . import _lib

_dll = _lib.dll


def kernel_kind():
    """Which candidate kernel ``factor_cosine_topk`` runs (``MRB_SIM_KERNEL=dmma`` selects the
    fp64 mma.sync kernel the tcgen05 one replaced; kept for A/B runs)."""
    import os
    if os.environ.get("MRB_SIM_KERNEL") == "dmma":
        return "fp64 DMMA (mma.sync m8n8k4)"
    return "tcgen05.mma kind::tf32 (TMA operands, TMEM accumulators)"


def padded_k(num_factors):
    """Contraction length the candidate GEMM really executes."""
    import os
    if os.environ.get("MRB_SIM_KERNEL") == "dmma":
        ks = (num_factors + 3) // 4
        return 4 * (4 if ks <= 4 else 8 if ks <= 8 else 13 if ks <= 13 else 16)
    return 8 * ((num_factors + 7) // 8)


def factor_cosine_topk(item_factors, num_factors=None, topk=50, q_lo=0, q_hi=None):
    """Top-``topk`` most similar movies of every query movie ``q_lo <= q < q_hi``.

    :param item_factors: ``(num_items, num_factors)`` array, or the flat ``num_items*num_factors``
        array ``cpp_ls.als`` returns together with ``num_factors``; 1 to 160 factors (every rank
        the exact ALS solvers train; 1 to 64 with ``MRB_SIM_KERNEL=dmma``)
    :param topk: 1 to 56
    :return: ids ``int32[q, topk]`` (-1 padded), scores ``float64[q, topk]``, ``SimInfo``
    """
    M = numpy.ascontiguousarray(item_factors, dtype=numpy.double)
    if M.ndim == 1:
        M = M.reshape(-1, num_factors)
    n, k = M.shape
    q_hi = n if q_hi is None else q_hi
    nq = q_hi - q_lo
    ids = numpy.full((max(nq, 0), topk), -1, dtype=numpy.int32)
    scores = numpy.zeros((max(nq, 0), topk), dtype=numpy.double)
    info = _lib.SimInfo()
    _lib.check(_dll.mrb_cosine_topk(_lib.dp(M), n, k, topk, q_lo, q_hi, _lib.ip(ids),
                                    _lib.dp(scores), ctypes.byref(info)))
    return ids, scores, info
