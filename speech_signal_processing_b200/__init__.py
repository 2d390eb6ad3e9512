"""speech_signal_processing_b200 -- the MFCC -> diag-GMM-UBM hot path of
kleinzcy/speech_signal_processing on B200 (sm_100a) behind the reference's own entry points.

Nothing here imports ``oracle`` and nothing falls back to the CPU: the CUDA library
(``libssp_b200.so``, built by ``python -m speech_signal_processing_b200.build``) is loaded on the
first call that needs it and a missing library or device raises.
"""
from . import synth  # noqa: F401  (host-side synthetic inputs)
from . import dtw  # noqa: F401  (MFCC_DTW.py template matching)
from . import vad  # noqa: F401  (reference VAD.py entry points)
from .frontend import (FrontEnd, MFCC, MFCC_lib, MelDbFrontEnd, PlpFrontEnd, Recipe, delta, extract_feature,  # noqa: F401
                       librosa_mfcc, librosa_recipe, mfcc, mfccInitFilterBanks, plp, plp_recipe, preprocessing, processing_recipe, psf_recipe,
                       scale, sidekit_recipe)
from .dtw import accelerated_dtw, dtw_identify, dtw_matrix  # noqa: F401
from .mixture import GaussianMixture, ModelSet, SharedModelSet, fit_batch, score_matrix  # noqa: F401
from .ubm import (GMM, chunk_features, chunk_identify, identify, identify_pcm, install, list_wavs, load_batch, load_data, load_extract,  # noqa: F401
                  main, map_adapt, map_enrol)
from .wavio import PcmBatch, read_wav_batch  # noqa: F401

__all__ = ["FrontEnd", "Recipe", "sidekit_recipe", "psf_recipe", "processing_recipe", "mfcc", "plp", "plp_recipe", "PlpFrontEnd", "MFCC", "MFCC_lib", "mfccInitFilterBanks",
           "librosa_mfcc", "librosa_recipe", "MelDbFrontEnd", "delta", "scale",
           "preprocessing", "extract_feature", "GaussianMixture", "ModelSet", "SharedModelSet", "score_matrix", "fit_batch", "GMM", "identify", "identify_pcm", "chunk_features", "chunk_identify",
           "map_adapt", "map_enrol", "install", "load_data", "load_batch", "list_wavs", "read_wav_batch", "PcmBatch", "load_extract", "main", "synth", "vad",
           "dtw", "accelerated_dtw", "dtw_matrix", "dtw_identify"]
