"""Host-side model assembly: the reference's ``Dlm`` / ``DlmParameters`` / ``Data`` types.

Mirrors ``core/src/main/scala/dlm/model/Dlm.scala`` (``Dlm`` :14-31, ``DlmParameters``
:36-57, ``Data`` :94, builders :139-243, composition :107-134).  Model assembly stays
on the host (numpy stands in for Breeze); the closures ``f(time)`` (n x p) and
``g(dt)`` (n x n) are evaluated here and handed to the C ABI as flat column-major
arrays, flagged time-invariant when every evaluation is identical.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Callable, Optional, Sequence

import numpy as np


def block_diagonal(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """``Dlm.blockDiagonal`` (Dlm.scala:197-208)."""
    out = np.zeros((a.shape[0] + b.shape[0], a.shape[1] + b.shape[1]))
    out[: a.shape[0], : a.shape[1]] = a
    out[a.shape[0]:, a.shape[1]:] = b
    return out


@dataclass(frozen=True)
class Dlm:
    """``Dlm(f, g)`` (Dlm.scala:14-15): ``f(time)`` is n x p, ``g(dt)`` is n x n."""

    f: Callable[[float], np.ndarray]
    g: Callable[[float], np.ndarray]
    # Host-side hint, not part of the reference's type: the builder KNOWS f ignores its argument
    # (polynomial, autoregressive, seasonal), so flattening a long grid evaluates it once
    # instead of T times.  Hand-written closures leave it False and are probed at every t.
    f_const: bool = False

    def outer_sum(self, y: "Dlm") -> "Dlm":
        """The reference's ``|*|`` (Dlm.scala:22-23, outerSumModel :117-122)."""
        return Dlm(lambda t: block_diagonal(self.f(t), y.f(t)),
                   lambda dt: block_diagonal(self.g(dt), y.g(dt)), self.f_const and y.f_const)

    def compose(self, y: "Dlm") -> "Dlm":
        """The reference's ``|+|`` (Dlm.scala:29-30, composeModels :107-111)."""
        return Dlm(lambda t: np.vstack([self.f(t), y.f(t)]),
                   lambda dt: block_diagonal(self.g(dt), y.g(dt)), self.f_const and y.f_const)

    __mul__ = outer_sum
    __add__ = compose


@dataclass
class DlmParameters:
    """``DlmParameters(v, w, m0, c0)`` (Dlm.scala:36-39)."""

    v: np.ndarray
    w: np.ndarray
    m0: np.ndarray
    c0: np.ndarray

    def __post_init__(self):
        self.v = np.atleast_2d(np.asarray(self.v, dtype=np.float64))
        self.w = np.atleast_2d(np.asarray(self.w, dtype=np.float64))
        self.m0 = np.atleast_1d(np.asarray(self.m0, dtype=np.float64))
        self.c0 = np.atleast_2d(np.asarray(self.c0, dtype=np.float64))

    def outer_sum(self, y: "DlmParameters") -> "DlmParameters":
        """``|*|`` on parameters (outerSumParameters, Dlm.scala:127-134)."""
        return DlmParameters(block_diagonal(self.v, y.v), block_diagonal(self.w, y.w),
                             np.concatenate([self.m0, y.m0]),
                             block_diagonal(self.c0, y.c0))

    __mul__ = outer_sum


@dataclass
class Data:
    """``Data(time, observation)`` (Dlm.scala:94); ``None`` entries are missing."""

    time: float
    observation: Sequence[Optional[float]]


def polynomial(order: int) -> Dlm:
    """``Dlm.polynomial`` (Dlm.scala:139-153): F = e1, G = I + superdiagonal."""
    def f(t):
        e = np.zeros((order, 1))
        e[0, 0] = 1.0
        return e

    def g(dt):
        return np.eye(order) + np.eye(order, k=1)

    return Dlm(f, g, True)


def regression(x: Sequence[np.ndarray]) -> Dlm:
    """``Dlm.regression`` (Dlm.scala:159-169): F_t = (1, x_t), G = I of size 1 + len(x_t)."""
    def f(t):
        idx = int(t) - 1
        return np.concatenate([[1.0], np.asarray(x[idx], dtype=np.float64).ravel()]).reshape(-1, 1)

    n = 1 + np.asarray(x[0], dtype=np.float64).size
    return Dlm(f, lambda dt: np.eye(n))


def autoregressive(*phi: float) -> Dlm:
    """``Dlm.autoregressive`` (Dlm.scala:176-185); G is the k x 1 column of phi."""
    k = len(phi)

    def f(t):
        m = np.zeros((k, 1))
        m[0, 0] = 1.0
        return m

    return Dlm(f, lambda dt: np.asarray(phi, dtype=np.float64).reshape(k, 1), True)


def rotation_matrix(theta: float) -> np.ndarray:
    """``Dlm.rotationMatrix`` (Dlm.scala:190-192)."""
    return np.array([[math.cos(theta), -math.sin(theta)],
                     [math.sin(theta), math.cos(theta)]])


def angle(period: int, dt: float) -> float:
    """``Dlm.angle`` (Dlm.scala:225-227); ``%`` is the JVM's fmod."""
    return 2 * math.pi * math.fmod(dt, period) / period


def seasonal(period: int, harmonics: int) -> Dlm:
    """``Dlm.seasonal`` (Dlm.scala:213-243)."""
    def f(t):
        return np.array([[1.0 if h % 2 == 0 else 0.0] for h in range(2 * harmonics)])

    def g(dt):
        out = rotation_matrix(1 * angle(period, dt))
        for h in range(2, harmonics + 1):
            out = block_diagonal(out, rotation_matrix(h * angle(period, dt)))
        return out

    return Dlm(f, g, True)


# ---------------------------------------------------------------- flattening


def cm(M: np.ndarray) -> np.ndarray:
    """(r, c) numpy matrix -> column-major flat array (Breeze ``DenseMatrix.data``)."""
    return np.ascontiguousarray(np.asarray(M, dtype=np.float64).T).ravel()


def from_cm(flat: np.ndarray, r: int, c: int) -> np.ndarray:
    return np.asarray(flat).reshape(c, r).T


def flatten_data(ys: Sequence[Data]):
    """``Vector[Data]`` -> (times[T], y[T][p]) with NaN for ``None``."""
    T = len(ys)
    if T == 0:
        # initialiseState calls t0.get on an empty collection (KalmanFilter.scala:116-117)
        raise ValueError("empty observation vector (NoSuchElementException in the reference)")
    p = len(ys[0].observation)
    times = np.array([d.time for d in ys], dtype=np.float64)
    y = np.array([[np.nan if o is None else float(o) for o in d.observation] for d in ys],
                 dtype=np.float64).reshape(T, p)
    return times, y


def materialise(mod: Dlm, times: np.ndarray, t_init: Optional[float] = None):
    """Evaluate the closures for a time grid.

    Returns (F, f_tv, G, g_tv, n, p): F is ``[n*p]`` or ``[T][n*p]``, G is ``[n*n]`` or
    ``[T][n*n]`` with ``G[t] = g(times[t] - times[t-1])`` and ``times[-1] := min(times) - 1``
    (KalmanFilter.initialiseState, KalmanFilter.scala:112-118), or ``t_init`` when the filter
    resumes from a saved state at that time.
    """
    times = np.asarray(times, dtype=np.float64)
    t0 = times.min() - 1.0 if t_init is None else float(t_init)
    prev = np.concatenate([[t0], times[:-1]])
    return materialise_dts(mod, times, times - prev)


def materialise_dts(mod: Dlm, times: np.ndarray, dts: np.ndarray):
    """As ``materialise`` with the time increments given explicitly (``G[t] = g(dts[t])``)."""
    # g is a function of dt alone: evaluate it once per distinct increment (a regular grid has
    # one); f is evaluated at every t unless the builder marked it constant
    tsel = times[:1] if getattr(mod, "f_const", False) else times
    Fs = [np.asarray(mod.f(float(t)), dtype=np.float64) for t in tsel]
    udt, inv = np.unique(np.asarray(dts, dtype=np.float64), return_inverse=True)
    Gu = [np.asarray(mod.g(float(dt)), dtype=np.float64) for dt in udt]
    Gs = Gu if len(udt) == 1 else [Gu[i] for i in inv]
    n, p = Fs[0].shape
    if Gs[0].shape != (n, n):
        raise ValueError(f"g(dt) is {Gs[0].shape}, expected {(n, n)}")
    f_tv = any(not np.array_equal(Fs[0], x) for x in Fs[1:])
    g_tv = any(not np.array_equal(Gs[0], x) for x in Gs[1:])
    F = np.stack([cm(x) for x in Fs]) if f_tv else cm(Fs[0])
    G = np.stack([cm(x) for x in Gs]) if g_tv else cm(Gs[0])
    return F, f_tv, G, g_tv, n, p
