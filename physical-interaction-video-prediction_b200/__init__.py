"""B200-native hot path of kristofbc/physical-interaction-video-prediction (the training step of
``src/models/train_model.py``): reference-named links over hand-written sm_100a kernels in libpivp.so.

Import as ``pivp_b200`` (alias module at the repo root) -- the directory name carries a hyphen.
"""
from ._lib import lib, PivpError, parse_header, LIBPATH, HEADER          # noqa: F401
from . import layout                                                      # noqa: F401


def __getattr__(name):
    # torch-dependent modules are imported lazily so that `import pivp_b200` works in a build-only environment
    if name in ("functions", "links", "engine", "tensorcore", "parallel", "train", "data", "serializers", "rollout", "train_loop",
                "predictor", "planner"):
        import importlib
        return importlib.import_module("." + name, __name__)
    if name in ("Model", "Adam", "BasicConvLSTMCell", "LayerNormalizationConv2D", "StatelessCDNA", "StatelessDNA",
                "StatelessSTP", "concat_examples", "scheduled_sample", "peak_signal_to_noise_ratio",
                "num_ground_truth", "scheduled_sample_mask"):
        from . import links
        return getattr(links, name)
    if name == "TrainStep":
        from .train import TrainStep
        return TrainStep
    if name in ("Rollout", "predict"):
        from . import rollout
        return getattr(rollout, name)
    if name == "Predictor":
        from .predictor import Predictor
        return Predictor
    if name == "CEMPlanner":
        from .planner import CEMPlanner
        return CEMPlanner
    if name in ("save_npz", "load_npz"):
        from . import serializers
        return getattr(serializers, name)
    if name == "BatchPrefetcher":
        from .train import BatchPrefetcher
        return BatchPrefetcher
    raise AttributeError(name)
