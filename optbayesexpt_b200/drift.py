"""Time-varying parameters: the random-walk step the engine applies to its cloud after every update.

``drift`` is the per-parameter standard deviation of one step (a scalar or one value per parameter) or the full
covariance ``Q`` of one step.  The device applies ``x <- x + F z`` with ``z ~ N(0, I)`` and ``F`` the
lower-triangular factor computed here on the host, ``F F^T = Q``.
"""
import numpy as np

#: ``Q`` counts as symmetric when ``|Q - Q^T| <= SYMMETRY_TOL * max|Q|`` elementwise ...
SYMMETRY_TOL = 1e-12
#: ... and as positive semidefinite when its smallest eigenvalue is ``>= -PSD_TOL * max|Q|``
PSD_TOL = 1e-12


def semidefinite_cholesky(q):
    """Lower-triangular ``L`` with ``L L^T = q`` for a symmetric positive SEMIdefinite ``q``.

    Cholesky without pivoting, so that ``L`` stays lower-triangular, in which a pivot at the rounding level of its
    own diagonal entry (``<= 4 d eps q_jj``) counts as zero and leaves column j of ``L`` zero: for a semidefinite
    ``q`` the whole column of the Schur complement vanishes with its pivot.  A parameter with zero variance (a zero
    row and column of ``q``) therefore gets an all-zero row of ``L``, exactly."""
    q = np.asarray(q, dtype=np.float64)
    d = q.shape[0]
    eps = np.finfo(np.float64).eps
    low = np.zeros((d, d))
    for j in range(d):
        s = q[j, j] - low[j, :j] @ low[j, :j]
        if not s > 4.0 * d * eps * q[j, j]:
            continue
        low[j, j] = np.sqrt(s)
        for i in range(j + 1, d):
            low[i, j] = (q[i, j] - low[i, :j] @ low[j, :j]) / low[j, j]
    return low


def drift_factor(drift, n_dims):
    """The lower-triangular factor ``F`` (n_dims, n_dims) of a ``drift`` argument, or None for ``drift=None``.

    Raises ``ValueError`` for a shape that is neither a scalar, ``(n_dims,)`` nor ``(n_dims, n_dims)``, non-finite
    values, a negative standard deviation, or a covariance that is not symmetric or not positive semidefinite within
    ``SYMMETRY_TOL`` / ``PSD_TOL``."""
    if drift is None:
        return None
    try:
        a = np.array(drift, dtype=np.float64)
    except (TypeError, ValueError) as exc:
        raise ValueError(f'drift must be a number, {n_dims} standard deviations or an ({n_dims}, {n_dims}) '
                         f'covariance, got {drift!r}') from exc
    if a.ndim > 2 or (a.ndim == 1 and a.shape != (n_dims,)) or (a.ndim == 2 and a.shape != (n_dims, n_dims)):
        raise ValueError(f'drift must be a number, {n_dims} standard deviations or an ({n_dims}, {n_dims}) '
                         f'covariance, got shape {a.shape}')
    if not np.all(np.isfinite(a)):
        raise ValueError(f'drift must be finite, got {drift!r}')
    if a.ndim < 2:
        std = np.broadcast_to(a, (n_dims,))
        if np.any(std < 0.0):
            raise ValueError(f'drift standard deviations must be >= 0, got {drift!r}')
        return np.diag(std)
    scale = float(np.max(np.abs(a)))
    if np.any(np.abs(a - a.T) > SYMMETRY_TOL * scale):
        raise ValueError('the drift covariance must be symmetric')
    q = 0.5 * (a + a.T)
    if scale > 0.0 and np.linalg.eigvalsh(q)[0] < -PSD_TOL * scale:
        raise ValueError('the drift covariance must be positive semidefinite')
    return semidefinite_cholesky(q)


def batched_drift_factors(drift, n_instances, n_dims):
    """The factors of a batched engine's ``drift``: None for ``drift=None``, one ``(n_dims, n_dims)`` F shared by all
    instances for every form ``drift_factor`` takes, or ``(n_instances, n_dims, n_dims)`` factors for an
    ``(n_instances, n_dims, n_dims)`` array of covariances (per-instance standard deviations are passed as diagonal
    covariances).  Each slice is validated like the single engine's ``drift``; ``ValueError`` names the instance."""
    if drift is None:
        return None
    try:
        a = np.array(drift, dtype=np.float64)
    except (TypeError, ValueError) as exc:
        raise ValueError(f'drift must be a number, {n_dims} standard deviations, an ({n_dims}, {n_dims}) covariance or '
                         f'({n_instances}, {n_dims}, {n_dims}) covariances, got {drift!r}') from exc
    if a.ndim < 3:
        return drift_factor(a, n_dims)
    if a.shape != (n_instances, n_dims, n_dims):
        raise ValueError(f'per-instance drift covariances must have shape ({n_instances}, {n_dims}, {n_dims}), got '
                         f'{a.shape}')
    out = np.empty_like(a)
    for b in range(n_instances):
        try:
            out[b] = drift_factor(a[b], n_dims)
        except ValueError as exc:
            raise ValueError(f'drift of instance {b}: {exc}') from None
    return out
