"""shared helpers for the parity tests (test infrastructure)"""
import numpy as np

NOM = ("t", "q", "R", "p", "v", "ba", "bg", "g")


def random_states(batch, rng, t0=1.0):
    """random but plausible filter states in the fbus_state_soa layout (dict of [n][B] arrays)"""
    from fbus_ekf_b200 import capi
    import fbus_oracle_np as onp
    st = capi.alloc_state(batch, True)
    for b in range(batch):
        A = rng.normal(size=(18, 18))
        P = A @ A.T * 1e-3 + np.diag(rng.uniform(1e-4, 1.0, 18))
        P[15:, 15:] += np.eye(3) * rng.uniform(0, 100.0)
        P = (P + P.T) / 2
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        q2 = q + 1e-3 * rng.normal(size=4)  # carried rotation slightly stale (SURVEY A.3-2)
        q2 /= np.linalg.norm(q2)
        st["q"][:, b] = q
        st["R"][:, b] = onp.q2R(q2).ravel()
        st["p"][:, b] = rng.normal(size=3) * 0.3
        st["v"][:, b] = rng.normal(size=3) * 0.2
        st["ba"][:, b] = rng.normal(size=3) * 0.05
        st["bg"][:, b] = rng.normal(size=3) * 2e-3
        st["g"][:, b] = [9.8, 0, 0]
        st["P"][:, b] = P.ravel()
    st["t"][:] = t0
    st["initialised"][:] = 1
    return st


def cov_close(P, Pref, rtol=1e-9):
    """SURVEY 7 'hard parts' 2: max|dP| <= rtol*max|P| and per-entry relative rtol where |P_ij| >= 1e-6 max|P|.
    P, Pref: [324][B]"""
    P = np.asarray(P)
    Pref = np.asarray(Pref)
    scale = np.abs(Pref).max(axis=0, keepdims=True)
    d = np.abs(P - Pref)
    ok_abs = (d <= rtol * scale).all()
    big = np.abs(Pref) >= 1e-6 * scale
    ok_rel = (d[big] <= rtol * np.abs(Pref)[big]).all()
    worst = float((d / scale).max())
    return bool(ok_abs and ok_rel), worst


IX6 = [0, 1, 2, 6, 7, 8]  # (position, attitude): the block of P that the 6-dof NEES inverts


def _cov18(P):
    """one filter's covariance ([324] or 18x18, float64 or an object array of mpmath numbers) -> 18x18 object array of mpf"""
    import mp_reference as mpr
    return mpr.mpa(np.asarray(P).reshape(18, 18))


def cov_whitened_err(P, Pref):
    """max |L^-1 (P6 - P6ref) L^-T| with L = chol(P6ref), P6 = P[IX6, IX6], evaluated in mpmath.  It bounds the relative
    error of any e^T P6^-1 e (NEES) computed from P6 instead of P6ref, whatever P6's scale and conditioning, which cov_close's
    max|P|-scaled measure does not.  P, Pref: one filter, [324] or 18x18; Pref may be an mpmath object array (exact)."""
    import mp_reference as mpr
    D = (_cov18(P) - _cov18(Pref))[np.ix_(IX6, IX6)]
    Li = mpr._inv(mpr._chol(_cov18(Pref)[np.ix_(IX6, IX6)]))
    return float(np.abs(mpr.to_np(Li @ D @ Li.T)).max())


def cov_corr_err(P, Pref):
    """max |P_ij - Pref_ij| / sqrt(Pref_ii Pref_jj) over all 18x18 entries: the error relative to the correlation scale of each
    entry, so small variances (a converged pose block) weigh as much as the gravity block.  Same arguments as cov_whitened_err."""
    import mp_reference as mpr
    A, B = _cov18(P), _cov18(Pref)
    d = np.sqrt(np.abs(np.diag(mpr.to_np(B))))
    return float((np.abs(mpr.to_np(A - B)) / np.outer(d, d)).max())


def state_close(a, b, rtol=1e-9, fields=NOM):
    worst = 0.0
    ok = True
    for f in fields:
        x, y = np.asarray(a[f], dtype=np.float64), np.asarray(b[f], dtype=np.float64)
        scale = np.maximum(np.abs(y), 1.0)
        e = float((np.abs(x - y) / scale).max())
        worst = max(worst, e)
        ok = ok and e <= rtol
    return ok, worst
