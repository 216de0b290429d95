"""B200-native embedding-vs-gallery matcher: the hot path of
bharatlytics/faceRecognition_InfrenceEngine (the per-face np.dot loop of infrenceServer.py /
peopleCount.py and the in-process gallery cache behind it), rebuilt as hand-written sm_100a CUDA
behind a C ABI (include/frg.h).  See DESIGN.md for scope and INTEGRATION.md for the binding.

Importing the package requires the built library (no CPU fallback):
    python -m facerecognition_infrenceengine_b200.build
"""
from . import _native
from ._native import NativeError
from .gallery import GalleryStore, StaleRows
from .matcher import (CAMPUS_THRESHOLD, CAMPUS_UNKNOWN, LIVE_THRESHOLD, CameraProcessor,
                      FaceRecognitionProcessor, Matcher, MatchResult, RangeResult)
from .manager import BroadcastSource, EmbeddingManager, GalleryView, ListSource
from .enrol import EnrolmentChecker, EnrolmentGallery, find_duplicate_pairs
from .clustering import UnknownClusterer
from .aggregator import BatchAggregator

__all__ = ["GalleryStore", "Matcher", "MatchResult", "RangeResult", "find_duplicate_pairs", "FaceRecognitionProcessor", "CameraProcessor",
           "EmbeddingManager", "GalleryView", "ListSource", "BroadcastSource", "EnrolmentChecker", "EnrolmentGallery", "StaleRows", "UnknownClusterer",
           "BatchAggregator", "NativeError", "LIVE_THRESHOLD",
           "CAMPUS_THRESHOLD", "CAMPUS_UNKNOWN"]
