"""swraytracing_b200 -- B200-native engine for SWRaytracing's packet hot path (see DESIGN.md)."""
from .engine import (Engine, QGFlow, QG2Flow, SwrtError, load_library, interpolate_dev, g2k_dev, k2g_dev,
                     MODE_SPECTRAL, MODE_LAGRANGE6, MODE_NUFFT, SCHEME_LEAPFROG, SCHEME_RK4_PACKET, SCHEME_RK4_XKA,
                     HIST_INTRINSIC, HIST_ABSOLUTE, FLAG_RHS_GH, EVENT_X, EVENT_Y, EVENT_K, EVENT_L, EVENT_KMAG,
                     EVENT_OMEGA, MAX_EVENTS, Q_XMOD, Q_YMOD, Q_K, Q_L, Q_KMAG, Q_THETA, Q_OMEGA, Q_OMEGA_ABS,
                     W_ACTION, W_ENERGY, W_PSEUDO_K, W_PSEUDO_L, MAX_WEIGHTS, fixed_sums_to_double)

__all__ = ["Engine", "QGFlow", "QG2Flow", "SwrtError", "load_library", "interpolate_dev", "g2k_dev", "k2g_dev",
           "MODE_SPECTRAL", "MODE_LAGRANGE6", "MODE_NUFFT", "SCHEME_LEAPFROG", "SCHEME_RK4_PACKET", "SCHEME_RK4_XKA",
           "HIST_INTRINSIC", "HIST_ABSOLUTE", "FLAG_RHS_GH", "EVENT_X", "EVENT_Y", "EVENT_K", "EVENT_L", "EVENT_KMAG",
           "EVENT_OMEGA", "MAX_EVENTS", "Q_XMOD", "Q_YMOD", "Q_K", "Q_L", "Q_KMAG", "Q_THETA", "Q_OMEGA", "Q_OMEGA_ABS",
           "W_ACTION", "W_ENERGY", "W_PSEUDO_K", "W_PSEUDO_L", "MAX_WEIGHTS", "fixed_sums_to_double"]
