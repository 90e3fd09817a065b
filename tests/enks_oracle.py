"""Reference of the ensemble Kalman smoother in gain form (no transform, no Woodbury), for the tests of txh_enks_smooth
and Muskingum.run_assimilating(smooth_lag=...)."""
import numpy as np


def enks_gain(A_past, HA, dz, S):
    """Ensemble Kalman smoother gain of one update for a past state (the ensemble counterpart of the RTS smoother,
    da.py:139-264): the sample cross-covariance of the past anomalies with the predicted observations of the update,
    times S^-1 dz, evaluated with an explicit inverse as oracle.enkf_update does (da.py:119).

    A_past : [k][M] anomalies of the past state (already smoothed by the updates before this one)
    HA     : [m][M] forecast anomalies at the gauges of the update
    dz     : [m][M] its innovations Zp - O[s]
    S      : [m][m] its innovation covariance HA HA^T/(M-1) + Q[s,s] + R
    Q[:, s] is not part of the cross-covariance: model noise added at the update is uncorrelated with earlier states.
    Returns the gain [k][M] to add to the past state."""
    A_past = np.asarray(A_past, dtype=np.float64)
    HA = np.asarray(HA, dtype=np.float64)
    M = HA.shape[1]
    return (A_past @ HA.T / (M - 1)) @ np.linalg.inv(np.asarray(S, dtype=np.float64)) @ np.asarray(dz, dtype=np.float64)


def smooth_transforms(rec, T_hist, nupd, every, rec_every, lag):
    """The definition txh_enks_smooth implements, by a loop: slot j (after step (j+1) rec_every) takes, in increasing
    u, every update u (after step (u+1) every) with s_j < t_u <= s_j + lag as X <- X + (X - mean) T_u."""
    out = np.array(rec, dtype=np.float64, copy=True)
    for j in range(out.shape[0]):
        s = (j + 1) * rec_every
        for u in range(nupd):
            t = (u + 1) * every
            if s < t <= s + lag:
                X = out[j]
                out[j] = X + (X - X.mean(axis=1, keepdims=True)) @ T_hist[u]
    return out
