"""rassengine_b200: B200-native retrieval hot path of RASSEngine (kNN + hybrid query behind the
OpenSearchIndexer surface).  Host code is Python over a C-ABI CUDA library; see DESIGN.md."""
from ._capi import (METRIC_COSINE, METRIC_L2, KEEP_FP32, BF16_ONLY, NO_INT8_SHADOW, PATH_AUTO, PATH_STREAM, PATH_UMMA,
                    PATH_EXACT, PATH_GEMM, PATH_UMMA8, RassError, RassStats)
from .engine import Engine

__all__ = ["Engine", "RassError", "RassStats", "METRIC_COSINE", "METRIC_L2", "KEEP_FP32", "BF16_ONLY",
           "NO_INT8_SHADOW", "PATH_AUTO", "PATH_STREAM", "PATH_UMMA", "PATH_EXACT", "PATH_GEMM", "PATH_UMMA8"]
