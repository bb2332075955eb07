"""Estimator-protocol mirror of what stage_1 uses from scikit-learn.

``B200LinearRegression`` keeps the constructor / ``fit`` / ``predict`` / attribute contract of
``sklearn.linear_model.LinearRegression`` as the reference uses it
(stage_1_train_model.py:105-107: ``LinearRegression(fit_intercept=True)``, ``.fit(X_train, y_train)``,
``.predict(X_test)``), with the arithmetic on the B200 through libb2gram.so.  ``alpha`` adds the
ridge term (alpha = 0 == the reference).

``to_sklearn()`` returns a genuine ``sklearn.linear_model.LinearRegression`` carrying our
coefficients: stage_2_serve_model.py:65,78,79 un-pickles the model with only sklearn / numpy /
joblib importable, calls ``.predict`` and ``str(model)`` -- a custom class could not be loaded there.
"""
from __future__ import annotations

from typing import Optional

import numpy as np

from . import _native as native

_shared_ctx: Optional[native.Context] = None


def default_context() -> native.Context:
    global _shared_ctx
    if _shared_ctx is None or _shared_ctx._h is None:
        _shared_ctx = native.Context(0)
    return _shared_ctx


_F64_UPLOAD_LIMIT = 64 << 30     # float64 host rows larger than this (as fp32, bytes) are converted and streamed block-wise

# Smallest sqrt(lambda_min / lambda_max) of the centred Gram, scaled to unit diagonal, that a statistic from an inexact
# kernel resolves.  The kernels' error is entrywise relative, |dA_ij| <= eps sqrt(A_ii A_jj) (tests/test_gpu_hard_data.py:
# tensor core ~3e-5, narrow ~3e-7), i.e. eps in the scaled matrix, whatever the column scales; the limits are ~sqrt of
# eps * D.  Below them the small eigenvalues are noise of either sign, so neither the LDL^T pivots nor rank_ can be
# trusted.
_RESOLVABLE = {native.KERNEL_NARROW: 3e-3, native.KERNEL_TCGEN05: 1e-2}
_RESOLVABLE_BF16_OPERAND = 1e-1      # the tensor core's single-operand mode (PRECISION_BF16)


def _as_f32_matrix(X) -> np.ndarray:
    X = np.asarray(X)
    if X.ndim == 1:
        X = X.reshape(-1, 1)
    if X.ndim != 2:
        raise ValueError(f"Expected 2D array, got {X.ndim}D array instead")
    if X.shape[1] > native.MAX_D:
        raise ValueError(f"at most {native.MAX_D} features are supported, got {X.shape[1]}")
    return np.ascontiguousarray(X, dtype=np.float32)


class B200LinearRegression:
    """The statistic S = [X 1 y]^T [X 1 y] of a fit lives in the (shared) context while the fit runs; whatever an
    estimator needs of it later -- the next ``partial_fit``, a deferred ``singular_`` / ``rank_`` -- is kept per
    estimator (``_S``) or guarded by the context's serial number, so two estimators on one context never see each
    other's rows."""

    def __init__(self, *, fit_intercept: bool = True, alpha: float = 0.0, tol: float = 1e-6,
                 ctx: Optional[native.Context] = None):
        self.fit_intercept = fit_intercept
        self.alpha = float(alpha)
        self.tol = tol
        self._ctx = ctx
        self._S: Optional[np.ndarray] = None     # this estimator's statistic (set by partial_fit / deferred attributes)
        self._serial = -1                        # ctx.serial right after this estimator's last fit

    @property
    def ctx(self) -> native.Context:
        return self._ctx if self._ctx is not None else default_context()

    # -- fit -------------------------------------------------------------------------------------
    def _set_solution(self, coef, b0, d: int) -> None:
        if not (np.all(np.isfinite(coef)) and np.isfinite(b0)):
            # sklearn's check_array refuses such input up front; here it shows up in the statistic
            raise ValueError("Input X or y contains NaN, infinity or a value too large for dtype('float32').")
        self.coef_ = coef
        self.intercept_ = np.float64(b0 if self.fit_intercept else 0.0)
        self.n_features_in_ = int(d)

    def _spectrum(self, d: int, need_coef: bool):
        """singular_ / rank_ of the statistic resident in the context (eigenvalues only, b2_solve_eigvals); when the
        centred Gram is numerically rank deficient (or the factorisation failed) also the minimum-norm coefficients
        gelsd would return (b2_solve_spectral, device Jacobi)."""
        ctx = self.ctx
        sing, rank, rows = ctx.solve_eigvals(cond=self.tol, fit_intercept=self.fit_intercept)
        self.singular_ = sing[: min(rows, d)]
        self.rank_ = int(rank)
        if (need_coef or (rank < min(rows, d) and self.alpha == 0.0)) and d > 0:
            coef, b0, sing_j, rank_j = ctx.solve_spectral(cond=self.tol, fit_intercept=self.fit_intercept)
            self.singular_ = sing_j[: min(rows, d)]
            self.rank_ = int(rank_j)
            self._set_solution(coef, b0, d)

    def _drop_spectrum(self) -> None:
        for name in ("singular_", "rank_"):
            if hasattr(self, name):
                delattr(self, name)

    def _unresolved(self) -> bool:
        """Did an inexact kernel build the resident statistic, and is its centred Gram closer to singular than that
        kernel resolves?  Judged on the Gram scaled to unit diagonal (the kernels' error is relative to the columns' own
        scales), so a well-conditioned design whose columns differ in scale -- age beside income -- keeps the fast
        statistic.  With a communicator the decision must be the same on every rank (the rebuild all-reduces): it then
        depends on the all-reduced S alone and takes the largest limit, whichever kernels this rank's shard used."""
        ctx = self.ctx
        if ctx.comm_info()["n_ranks"] > 1:
            limit = max(max(_RESOLVABLE.values()), _RESOLVABLE_BF16_OPERAND)
        else:
            used = ctx.gram_kernels()
            limits = [lim for k, lim in _RESOLVABLE.items() if used & (1 << k)]
            if used & (1 << native.KERNEL_TCGEN05) and ctx.precision == native.PRECISION_BF16:
                limits.append(_RESOLVABLE_BF16_OPERAND)
            if not limits:
                return False
            limit = max(limits)
        s = np.asarray(getattr(self, "singular_", ()))
        if s.size < 2 or not s[0] > 0.0 or s[-1] >= limit * np.sqrt(s.size) * s[0]:
            return False       # van der Sluis: kappa(scaled) <= D kappa(unscaled), so the scaled Gram is resolved too
        # the unscaled spectrum is near singular: look at the scaled one (host eigvalsh of a D x D matrix, ~1 ms at 128)
        S = ctx.gram_export()
        d = S.shape[0] - 2
        n = S[d, d]
        if self.fit_intercept:
            xm = S[:d, d] / n
            A = S[:d, :d] - n * np.outer(xm, xm)
        else:
            A = S[:d, :d].copy()
        dg = np.diag(A).copy()
        # a column whose centred variance is at the fp64 rounding of its raw moment is constant: no scale to judge by
        if np.any(dg <= 64.0 * np.finfo(np.float64).eps * np.abs(np.diag(S)[:d])):
            return True
        r = 1.0 / np.sqrt(dg)
        lam = np.linalg.eigvalsh(0.5 * (A + A.T) * np.outer(r, r))
        return not lam[0] > (limit ** 2) * lam[-1]

    def _refit_exact(self, X, y, row_mask, mask_keep, d: int) -> None:
        """Rebuild the statistic of the same rows on the exact fp64 kernel and solve again."""
        ctx = self.ctx
        kernel = ctx.kernel
        ctx.set_kernel(native.KERNEL_SIMT)
        try:
            ctx.gram_reset(d)
            ctx.gram_accumulate(X, y, row_mask, mask_keep)
            ctx.gram_allreduce()
        finally:
            ctx.set_kernel(kernel)
        self._drop_spectrum()
        singular = False
        try:
            coef, b0 = ctx.solve(alpha=self.alpha, fit_intercept=self.fit_intercept)
            self._set_solution(coef, b0, d)
        except np.linalg.LinAlgError:
            singular = True
        self._serial = ctx.serial
        self._spectrum(d, need_coef=singular)

    def fit(self, X, y, row_mask=None, mask_keep: int = 1, with_spectrum: bool = True) -> "B200LinearRegression":
        """X: (n, D) host array (any float dtype; staged as fp32) or a ``DeviceArray`` (f32 / bf16).
        ``row_mask`` (uint8 per row) restricts the fit to rows equal to ``mask_keep``.
        ``with_spectrum=False`` defers ``singular_`` / ``rank_`` (computed on first use, e.g. by ``to_sklearn``).

        When the tensor-core or narrow kernel built the statistic and its spectrum shows the centred Gram closer to
        singular than that kernel resolves (s_min / s_max below ~sqrt of its error), the rows are accumulated again on
        the exact fp64 kernel and solved from that statistic: rank_, coef_ and singular_ are then gelsd's even for an
        exactly collinear design (one-hot blocks with the intercept, x2 = 3 x1, ...).  "Near singular" is judged on the
        Gram scaled to unit diagonal: well-conditioned fits never pay for it, however different their columns' scales.  The check needs the spectrum: with ``with_spectrum=False`` the fit keeps the inexact statistic's
        solution (and the deferred spectrum is that statistic's); ``partial_fit`` and ``solve_resident`` no longer hold
        the earlier tranches' rows and likewise solve what the kernels accumulated."""
        ctx = self.ctx
        owned = []                  # device buffers this call created (float64 host rows: converted on the way up)
        if isinstance(X, native.DeviceArray):
            d = X.shape[1]
        else:
            Xh = np.asarray(X)
            if Xh.ndim == 2 and Xh.dtype == np.float64 and 0 < Xh.shape[1] <= native.MAX_D and Xh.shape[0] >= 65_536 \
                    and Xh.size * 4 <= _F64_UPLOAD_LIMIT:
                # what scikit-learn users hand over: float64 rows.  numpy's astype(float32) is one thread; b2_upload_columns
                # converts with the host threads of the bounce ring beside the H2D copies and leaves the rows resident
                if np.asarray(y).size != Xh.shape[0]:
                    raise ValueError(f"Found input variables with inconsistent numbers of samples: "
                                     f"[{Xh.shape[0]}, {np.asarray(y).size}]")
                X = ctx.upload_columns([Xh[:, j] for j in range(Xh.shape[1])])
                y = ctx.to_device(np.ascontiguousarray(np.asarray(y).ravel(), dtype=np.float32))
                owned = [X, y]
                if row_mask is not None and not isinstance(row_mask, native.DeviceArray):
                    row_mask = ctx.to_device(np.ascontiguousarray(row_mask, dtype=np.uint8))
                    owned.append(row_mask)
            else:
                X = _as_f32_matrix(X)
                y = np.ascontiguousarray(np.asarray(y).ravel(), dtype=np.float32)
                if y.shape[0] != X.shape[0]:
                    raise ValueError(f"Found input variables with inconsistent numbers of samples: "
                                     f"[{X.shape[0]}, {y.shape[0]}]")
            d = X.shape[1]
        self._S = None
        self._drop_spectrum()
        try:
            singular = False
            try:
                coef, b0 = ctx.fit(X, y, row_mask, mask_keep, alpha=self.alpha, fit_intercept=self.fit_intercept)
                self._set_solution(coef, b0, d)
            except np.linalg.LinAlgError:
                singular = True     # rank deficient and alpha == 0: the minimum-norm solution gelsd would return
            self._serial = ctx.serial
            if with_spectrum or singular:
                self._spectrum(d, need_coef=singular)
                if self._unresolved():
                    self._refit_exact(X, y, row_mask, mask_keep, d)
        finally:
            for a in owned:
                a.free()
        return self

    def partial_fit(self, X, y, with_spectrum: bool = False) -> "B200LinearRegression":
        """Fold one more tranche into THIS estimator's running statistic and re-solve (incremental daily refit)."""
        ctx = self.ctx
        Xh = X if isinstance(X, native.DeviceArray) else _as_f32_matrix(X)
        d = Xh.shape[1]
        if not isinstance(Xh, native.DeviceArray):
            y = np.ascontiguousarray(np.asarray(y).ravel(), dtype=np.float32)
        if self._S is not None and self._S.shape[0] == d + 2:
            ctx.gram_import(self._S)
        elif hasattr(self, "coef_") and self._serial == ctx.serial and ctx.d == d:
            pass                       # the statistic of this estimator's last fit is still resident
        else:
            ctx.gram_reset(d)          # first tranche of this estimator
        ctx.gram_accumulate(Xh, y)
        self._drop_spectrum()
        singular = False
        try:
            coef, b0 = ctx.solve(alpha=self.alpha, fit_intercept=self.fit_intercept)
            self._set_solution(coef, b0, d)
        except np.linalg.LinAlgError:
            singular = True
        self._S = ctx.gram_export()
        self._serial = ctx.serial
        if with_spectrum or singular:
            self._spectrum(d, need_coef=singular)
        return self

    def solve_resident(self, d: int, S: Optional[np.ndarray] = None) -> "B200LinearRegression":
        """Solve from the statistic currently resident in the context (after gram_import / gram_accumulate calls made
        by the caller, e.g. IncrementalTrainer); ``S``: the caller's host copy of it, kept for deferred attributes."""
        ctx = self.ctx
        self._drop_spectrum()
        self._S = S
        try:
            coef, b0 = ctx.solve(alpha=self.alpha, fit_intercept=self.fit_intercept)
            self._set_solution(coef, b0, d)
        except np.linalg.LinAlgError:
            self._spectrum(d, need_coef=True)
        self._serial = ctx.serial
        return self

    def _ensure_spectrum(self) -> None:
        if hasattr(self, "rank_"):
            return
        ctx = self.ctx
        if self._S is not None:
            ctx.gram_import(self._S)
        elif self._serial != ctx.serial:
            raise RuntimeError("singular_ / rank_ were deferred (with_spectrum=False) and the statistic of this fit is no "
                               "longer resident in the context: refit, or fit with with_spectrum=True")
        self._spectrum(self.n_features_in_, need_coef=False)
        self._serial = ctx.serial

    # -- predict -------------------------------------------------------------------------------------
    def predict(self, X):
        ctx = self.ctx
        if isinstance(X, native.DeviceArray):
            yhat, _ = ctx.score(X, self.coef_, float(self.intercept_))
            return yhat
        Xh = _as_f32_matrix(X)
        if Xh.shape[1] != self.n_features_in_:
            raise ValueError(f"X has {Xh.shape[1]} features, but B200LinearRegression is expecting "
                             f"{self.n_features_in_} features as input.")
        yhat, _ = ctx.score(Xh, self.coef_, float(self.intercept_))
        return yhat.astype(np.float64)

    # -- artefact ----------------------------------------------------------------------------------------
    def to_sklearn(self):
        """A real sklearn LinearRegression with the attributes ``fit`` would have set
        (the joblib layout stage_1_train_model.py:113-114 dumps and stage_2_serve_model.py:65 loads)."""
        from sklearn.linear_model import LinearRegression
        self._ensure_spectrum()
        reg = LinearRegression(fit_intercept=self.fit_intercept)
        reg.coef_ = np.asarray(self.coef_, dtype=np.float64).copy()
        reg.intercept_ = np.float64(self.intercept_)
        reg.rank_ = int(self.rank_)
        reg.singular_ = np.asarray(self.singular_, dtype=np.float64).copy()
        reg.n_features_in_ = int(self.n_features_in_)
        return reg

    def __repr__(self) -> str:
        return "B200LinearRegression()" if self.alpha == 0.0 else f"B200LinearRegression(alpha={self.alpha})"
