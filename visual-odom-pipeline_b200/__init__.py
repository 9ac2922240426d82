"""B200-native pyramidal Lucas-Kanade tracking: drop-in for the cv2.calcOpticalFlowPyrLK hot path
of JonasFrey96/Visual-Odom-Pipeline (src/extractor/extractor.py:44,45,65,66) and, next to it, the Shi-Tomasi
detection step (cv2.goodFeaturesToTrack, src/extractor/extractor.py:110-111), the loader's pre-filter
(cv2.bilateralFilter, src/loader/loader.py:86) and contrast-limited equalisation of the frames (cv2.createCLAHE).

Import name: ``visual_odom_pipeline_b200`` (the on-disk directory is ``visual-odom-pipeline_b200``).
"""
from ._lib import (KLT_MAX_CLAHE_TILES, KLT_MAX_SUBPIX_WIN, KLTLibraryError, LIB_PATH, OPTFLOW_LK_GET_MIN_EIGENVALS, OPTFLOW_USE_INITIAL_FLOW,
                   TERM_COUNT, TERM_EPS, Context, default_context)
from .corners import cornerMinEigenVal, cornerSubPix, detectNewFeatures, goodFeaturesToTrack
from .filters import bilateralFilter, createCLAHE
from .lk import buildOpticalFlowPyramid, calcOpticalFlowPyrLK, error, pinned_empty, trackBidirectional

__all__ = ["calcOpticalFlowPyrLK", "buildOpticalFlowPyramid", "trackBidirectional", "goodFeaturesToTrack", "cornerMinEigenVal", "cornerSubPix", "detectNewFeatures", "bilateralFilter", "createCLAHE", "error", "pinned_empty", "Context", "default_context",
           "KLTLibraryError", "LIB_PATH", "TERM_COUNT", "TERM_EPS", "OPTFLOW_USE_INITIAL_FLOW",
           "OPTFLOW_LK_GET_MIN_EIGENVALS", "KLT_MAX_SUBPIX_WIN", "KLT_MAX_CLAHE_TILES"]
__version__ = "0.1.2"
