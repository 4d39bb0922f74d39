"""B200-native batched UKF + URTSS for ship tracks.

A from-scratch, sm_100a-only implementation of the one data-parallel hot path of
NOC-OI/ship-track-estimators: the fp64 Unscented Kalman Filter with geodetic dynamics and the
unscented Rauch-Tung-Striebel smoother, behind the reference's own Python surface
(``kalman_filters``, ``ship_track``, ``utils``, ``cli``) plus the many-track entry point
:mod:`ship_track_estimators_b200.batch`.  The arithmetic lives in ``csrc/libste_ukf.so`` (C ABI in
``include/ste_ukf.h``); importing this package does not load it, calling a filter does.
"""
__version__ = "0.1.0"

__all__ = ["__version__", "kalman_filters", "utils", "constants", "ship_track", "performance_metrics", "batch", "batch_n", "synthetic", "sharding", "cli"]
