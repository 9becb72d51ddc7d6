"""graphlearninglayer_b200 -- B200 (sm_100a) implementation of the GraphLearningLayer hot path.

    from graphlearninglayer_b200 import LaplaceLearningSparseHard, knn_sym_dist, stable_conjgrad
    from graphlearninglayer_b200 import laplace_learning        # utils.laplace on GPU features, no host round trip
    from graphlearninglayer_b200 import laplace_learning_batched  # the same over B independent graphs (B, n, d)
    from graphlearninglayer_b200 import laplace_learning_trials  # T labeled sets on one graph (n, d)
    from graphlearninglayer_b200 import LaplaceLearningSparseHardBatched  # B independent graphs (B, n, d) in one call

The names resolve lazily so that ``python -m graphlearninglayer_b200.build`` can run before the shared library
exists; the first access loads libgll_b200.so through ctypes and fails loudly if it is missing or stale.  There is no
CPU or PyTorch fallback.
"""
__all__ = ["LaplaceLearningSparseHard", "LaplaceLearningSparseHardNormalized", "LaplaceLearningSparseHardBatched", "knn_sym_dist", "stable_conjgrad", "last_info", "GLL",
           "GraphedStep", "BaseSetEvaluator", "laplace_learning", "LaplaceResult",
           "laplace_learning_batched", "laplace_learning_trials"]
_ELSEWHERE = {"GraphedStep": ".graphed", "BaseSetEvaluator": ".evalcache", "laplace_learning": ".laplace_eval",
              "LaplaceResult": ".laplace_eval", "laplace_learning_batched": ".laplace_eval",
              "laplace_learning_trials": ".laplace_eval"}


def __getattr__(name):
    if name in _ELSEWHERE:
        import importlib

        return getattr(importlib.import_module(_ELSEWHERE[name], __name__), name)
    if name in __all__:
        import importlib

        mod = importlib.import_module(".GLL", __name__)
        return mod if name == "GLL" else getattr(mod, name)
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")
