"""Run the UNMODIFIED reference modules of the upstream KoeMorph project (a checkout named by KOEMORPH_REFERENCE).

TEST INFRASTRUCTURE ONLY -- used by ``tests/golden/make_golden.py`` to produce the
committed golden vectors and by ``bench.py --impl reference``; the test suite
reads those stored vectors and never imports the reference itself.

The reference cannot be imported as-is in this image: ``librosa`` and
``opensmile`` are not installed (SURVEY.md section 8c).  Following SURVEY.md
section 7 step 1 we pre-seed ``sys.modules`` with two minimal stand-ins and
then import ``src.model.*`` unchanged:

* ``librosa``  -- only ``feature.melspectrogram``, ``power_to_db``, ``filters.mel``,
  backed by the restatement in ``oracle/koemorph_oracle.py`` (so the mel stage of
  these goldens is a restatement, NOT librosa itself: parity unpinned there).
* ``opensmile`` -- a ``Smile`` whose ``process_signal`` returns an 88-column frame,
  enough for ``OpenSMILEeGeMAPSExtractor.__init__`` (opensmile_extractor.py:227-235).

``extract_emotion_features`` is replaced by ``Linear(264->256)(egemaps)`` with the
seeded compression layer, because the reference creates that layer unseeded and
outside ``state_dict`` (opensmile_extractor.py:586-592) and the path's inputs are
synthetic eGeMAPS windows (BASELINE.json north_star).
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np
import torch

from . import koemorph_oracle as O

# /root/reference in the build container; on the GPU box the byte-identical copies staged by oracle/stage_reference.py
# (oracle/_ref, git-ignored, shipped with the gpurun snapshot)
_STAGED_ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
REFERENCE_ROOT = os.environ.get("KOEMORPH_REFERENCE", "/root/reference")
if not os.path.isdir(os.path.join(REFERENCE_ROOT, "src", "model")) and os.path.isdir(os.path.join(_STAGED_ROOT, "src", "model")):
    REFERENCE_ROOT = _STAGED_ROOT


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "src", "model"))


def reference_kind() -> str:
    """"tree" (the reference checkout itself), "staged" (oracle/_ref copies) or "absent"."""
    if not reference_available():
        return "absent"
    return "staged" if REFERENCE_ROOT == _STAGED_ROOT else "tree"


def _install_stubs():
    if "librosa" not in sys.modules:
        lib = types.ModuleType("librosa")
        lib.__version__ = "0.10.restated"
        feat = types.ModuleType("librosa.feature")
        filt = types.ModuleType("librosa.filters")

        def melspectrogram(y=None, sr=22050, n_fft=2048, hop_length=512, win_length=None, n_mels=128,
                           fmin=0.0, fmax=None, power=2.0, center=True, pad_mode="constant", **kw):
            assert win_length in (None, n_fft)
            return O.melspectrogram(np.asarray(y), sr=sr, n_fft=n_fft, hop_length=hop_length, n_mels=n_mels,
                                    fmin=fmin, fmax=fmax if fmax is not None else sr / 2, power=power,
                                    center=center, pad_mode=pad_mode)

        def power_to_db(S, ref=1.0, amin=1e-10, top_db=80.0):
            assert ref is np.max, "only ref=np.max is on the path"
            return O.power_to_db(S, amin=amin, top_db=top_db)

        def mel(sr, n_fft, n_mels=128, fmin=0.0, fmax=None, **kw):
            return O.mel_filterbank(sr, n_fft, n_mels, fmin, fmax if fmax is not None else sr / 2)

        feat.melspectrogram = melspectrogram
        filt.mel = mel
        lib.feature = feat
        lib.filters = filt
        lib.power_to_db = power_to_db
        sys.modules["librosa"] = lib
        sys.modules["librosa.feature"] = feat
        sys.modules["librosa.filters"] = filt
    if "opensmile" not in sys.modules:
        import pandas as pd

        osm = types.ModuleType("opensmile")

        class FeatureSet:
            eGeMAPSv02 = "eGeMAPSv02"
            GeMAPS = "GeMAPS"

        class FeatureLevel:
            Functionals = "Functionals"
            LowLevelDescriptors = "LowLevelDescriptors"

        class Smile:
            def __init__(self, feature_set=None, feature_level=None):
                self.feature_set, self.feature_level = feature_set, feature_level

            def process_signal(self, signal, sampling_rate):
                return pd.DataFrame(np.zeros((1, 88), np.float32), columns=[f"f{i}" for i in range(88)])

        osm.FeatureSet, osm.FeatureLevel, osm.Smile = FeatureSet, FeatureLevel, Smile
        sys.modules["opensmile"] = osm


def import_reference():
    """-> (SimplifiedDualStreamModel, SequentialDualStreamModel, DualStreamCrossAttention, MelSlidingWindowExtractor)"""
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    _install_stubs()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    from src.model.simplified_dual_stream_model import SimplifiedDualStreamModel
    from src.model.sequential_dual_stream_model import SequentialDualStreamModel
    from src.model.dual_stream_attention import DualStreamCrossAttention
    from src.features.mel_sliding_window import MelSlidingWindowExtractor
    return SimplifiedDualStreamModel, SequentialDualStreamModel, DualStreamCrossAttention, MelSlidingWindowExtractor


_EMO_CFG = {"backend": "opensmile", "use_concatenation": True, "enable_caching": False, "device": "cpu",
            "sample_rate": 16000, "context_window": 20.0, "update_interval": 0.3}


def build_reference_model(weights, fps: int = 30, sequential: bool = True, stride_frames: int = 1):
    """Instantiate the reference model on CPU, load ``weights`` and wire the synthetic eGeMAPS input.
    Call ``model.set_egemaps(egemaps264)`` before ``model(audio)``."""
    Simple, Seq, _, _ = import_reference()
    kw = dict(d_model=256, num_heads=8, num_blendshapes=52, sample_rate=16000, target_fps=fps,
              mel_sequence_length=256 if fps == 30 else 512, emotion_config=dict(_EMO_CFG), device="cpu")
    model = Seq(stride_frames=stride_frames, **kw) if sequential else Simple(**kw)
    assert model.emotion_dim == 256, "opensmile stub did not take the concatenation path"
    missing = model.load_state_dict(O.model_state_dict(weights), strict=True)
    model.eval()
    comp = torch.nn.Linear(264, 256)
    with torch.no_grad():
        comp.weight.copy_(torch.from_numpy(weights["compression.weight"]))
        comp.bias.copy_(torch.from_numpy(weights["compression.bias"]))
    state = {}

    def set_egemaps(e):
        state["e"] = torch.as_tensor(np.asarray(e), dtype=torch.float32).reshape(-1, 264)

    def extract_emotion_features(audio):
        with torch.no_grad():
            return comp(state["e"]), {"backend_used": "opensmile", "processing_time": 0.0}

    model.set_egemaps = set_egemaps
    model.extract_emotion_features = extract_emotion_features
    return model
