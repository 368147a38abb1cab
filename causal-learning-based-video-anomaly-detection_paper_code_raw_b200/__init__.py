"""cvad_b200 -- B200-native (sm_100a) hot path of the causal video-anomaly-detection reference.

The directory name follows the project convention and is not a valid Python identifier; import it through the
root-level ``cvad_b200`` alias module (``import cvad_b200``).

Public surface (mirrors the reference's Python seam, SURVEY.md 8b):
  mb.CausalAnomalyDetector / mb.ImprovedMiniCausalVAD / mb.MiniCausalVAD      avenue_training_script2.py, script1.py
  mc.SimpleVideoAnomalyDetector / mc.StableTrainer                           minicausal_vad_complete3.py
  ma.CausalAnomalyDetector / ma.train_model / ma.test_model                  causal_anomaly_detection.py
  ma0.CausalAnomalyDetector / ma0.train_model / ma0.test_model               video_anomaly_detection.py
  ma0.StreamingWindowScorer (sliding windows over a frame stream: each frame's backbone pass is computed once)
  infer.GraphedStreamingScorer / infer.FrozenBackbone (the same windows, one CUDA graph replay per push; eval BatchNorm folded into the convolutions)
  infer.MultiStreamScorer (many cameras or the videos of a test set: one push and one CUDA graph replay per tick for all streams)
  infer.MultiStreamClipScorer (the same service for the 3-D clip models M-B, M-C and M-E from raw camera frames)
  md.VideoAutoEncoder / md.train_model / md.calculate_anomaly_scores         causal_anomaly_detection1.py
  infer.MultiStreamAutoEncoderScorer (many camera streams for M-D, one replay per tick; each frame encoded once)
  me.CausalAnomalyDetector / me.predict_anomaly_for_clip / me.score_windows  avenue_training_script_bbox.py
  train.train_improved_minicausal_vad (s2:339-468 driver with real resume, async checkpoints, history JSON)
  frames.DeviceFrames (uint8 frame cache on the device: cv2-exact bilinear resize, clip / sliding-window gather)
  evaltail (device-side percentile / AUC / evaluation metrics / smoothing: the numpy + sklearn code after the hot path)
  ops (autograd glue over include/cvad_b200.h), arena.FusedAdam, parallel.DataParallel
There is no CPU fallback: importing the package loads libcvad_b200.so and raises if it is missing.
"""
from . import _lib

_lib.lib()   # fail loudly when the CUDA extension has not been built

from . import arena, evaltail, frames, graphs, infer, ma, ma0, ma_ops, mb, mc, md, me, noise, ops, parallel, tc, train  # noqa: E402,F401

__all__ = ["arena", "evaltail", "frames", "graphs", "infer", "ma", "ma0", "ma_ops", "mb", "mc", "md", "me", "noise", "ops", "parallel", "tc", "train"]
