"""numpy restatement of the log densities of a fitted map (DESIGN.md section 1) on top of the CPU oracle's
OracleMap -- test infrastructure only.  The reference never defined these quantities (its evaluators assert separable
monotonicity and return exp(...)), so there are no golden fixtures: the anchors are identities (the objective, the
normalisation, pushforward(pullback) = Gaussian) and the reference's own evaluator where its quirks vanish."""

import numpy as np


def log_dS(om, k, Xs):
    """l_k = log dS_k/dx~_c of OracleMap `om` on standardised samples Xs (n, Dtot)."""
    b = om.coeffs_mon[k]
    if om.monotonicity == "integrated rectifier":
        r = np.dot(om.fun_mon(k, Xs), b[:, None])[..., 0]
        if om.rectifier_type == "exponential" and om.delta == 0:
            return r
        return np.log(om.rect.evaluate(r) + om.delta)
    return np.log(np.dot(om.der_fun_mon(k, Xs), b[:, None])[..., 0])


def _check_x_star(om, X_star):
    if X_star is not None and (om.skip_dimensions == 0 or X_star.shape[-1] != om.skip_dimensions):
        raise ValueError("X_star must hold the skip_dimensions conditioning columns of a partial map")


def _standardised(om, X, X_star):
    """[X_star | X] standardised, and log sigma_c of every component."""
    _check_x_star(om, X_star)
    if X_star is not None:
        X = np.column_stack((X_star, X))
    X = np.array(X, dtype=np.float64)
    if not om.standardize_samples:
        return X, np.zeros(om.D)
    c = np.arange(om.D) + om.skip_dimensions
    return (X - om.X_mean) / om.X_std, np.log(om.X_std[c])


def log_pullback_density(om, X, X_star=None):
    """sum_k [-S_k(x~)^2/2 - log(2 pi)/2 + l_k(x~) - log sigma_c]."""
    Xs, logsig = _standardised(om, X, X_star)
    out = np.zeros(Xs.shape[0])
    for k in range(om.D):
        S = om.s(Xs, k)
        out += -0.5 * S ** 2 - 0.5 * np.log(2 * np.pi) + log_dS(om, k, Xs) - logsig[k]
    return out


def log_pushforward_density(om, Z, log_target_pdf, X_star=None):
    """log_target_pdf(x) - sum_k [l_k(x~) - log sigma_c], x = om.inverse_map(Z, X_star)."""
    _check_x_star(om, X_star)
    X = om.inverse_map(Z, X_star)
    out = np.array(log_target_pdf(X), dtype=np.float64)
    Xs, logsig = _standardised(om, X, X_star)
    for k in range(om.D):
        out -= log_dS(om, k, Xs) - logsig[k]
    return out
