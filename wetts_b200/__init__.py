"""wetts_b200: B200-native (sm_100a) VITS inference hot path with the WeTTS interface.

Scope (SURVEY.md §8): SynthesizerTrn.infer = TextEncoder -> duration predictor -> length
regulation -> flow inversion -> HiFi-GAN generator, as hand-written CUDA kernels behind the
C ABI in include/wetts_b200.h.  Importing the package does not load the CUDA library;
constructing a model does, and fails loudly if it is missing.
"""
from .hparams import HParams, builtin_config, get_hparams_from_file  # noqa: F401
from .checkpoint import load_checkpoint  # noqa: F401
from .models import (Generator, PosteriorEncoder, ResidualCouplingTransformersBlock,  # noqa: F401
                     SynthesizerTrn, TextEncoder)
from ._lib import WettsError  # noqa: F401

__version__ = "0.1.0"


def build_model(hps, n_vocab, n_speakers, state_dict=None, device="cuda"):
    """Construct exactly as the reference's inference.py:65-80 does."""
    spec_channels = hps.data.filter_length // 2 + 1
    if "use_mel_posterior_encoder" in hps.model.keys() and hps.model.use_mel_posterior_encoder:
        spec_channels = hps.data.n_mel_channels   # VITS2 mel posterior encoder (inference.py:67-71)
    net = SynthesizerTrn(n_vocab, spec_channels, hps.train.segment_size // hps.data.hop_length,
                         n_speakers=n_speakers, **hps.model).eval()
    if state_dict is not None:
        net.load_state_dict(state_dict)
    return net.to(device)
