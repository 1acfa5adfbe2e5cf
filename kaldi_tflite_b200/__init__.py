"""
kaldi_tflite_b200 -- B200-native (sm_100a CUDA) implementation of kaldi-tflite's
wav -> x-vector hot path behind the reference's Python API.

    import kaldi_tflite_b200 as ktf          # or: import kaldi_tflite as ktf (alias package)
    ktf.layers.Framing / Windowing / FilterBank / DCT / MFCC / VAD / CMVN / BatchNorm / TDNN /
               StatsPooling / PLDA
    ktf.models.XvectorExtractorFromConfig / XvectorExtractor / SequentialFromConfig
    ktf.io.KaldiNnet3Reader / KaldiPldaReader / ReadKaldiArray / KaldiObjReader
    ktf.diarization.agglomerative_cluster
"""

from . import diarization  # noqa: F401
from . import io  # noqa: F401  (numpy only)
from . import kaldi_numpy  # noqa: F401
from . import layers  # noqa: F401
from . import models  # noqa: F401
from . import parallel  # noqa: F401
from ._native import KtfNativeError, launch_count  # noqa: F401

__version__ = "0.1.0"
