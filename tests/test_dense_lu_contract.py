"""Contract tests of the dense LU entry points (scb_getrf_sym_nopiv, scb_getrf_nopiv, scb_getrf_piv,
scb_getrs_nopiv) on synthetic host matrices, element by element against a plain fp64 reference.

The host scheduler of getrf.cu launches different kernels depending on the number of 128-blocks `nb`
(partial / full / several outer panels of q = 8 blocks, empty strip or bulk parts, the clipped band of the
recursive strip schedule), on split panels, look-ahead, the latency kernels, CUDA-graph capture and
replay and on 14 environment switches.  A film solve reaches only a few of these at a time, and a
1e-8 tolerance on the stream function hides a small error.  Here every factor tile and every block
inverse is compared with a reference factorization.

Error measure (`factor_errors`): for every 128 x 64 tile of the packed factors F = L\\U,
    e = max_tile |F - F_ref| / s,   s = max_ij (|L_ref| |U_ref|)_ij,
against the bound 4 n_pad u (u = 2^-53: the rounding-error bound gamma_n of an n-term fp64 inner product,
with a factor 4 for the reordered blocked sums of both sides).  Block inverses X (`dinv_errors`) are
compared element-wise with X_ref = inv(B_ref), B_ref the unit-lower / upper diagonal block of the
reference, weighted by the first-order perturbation of an inverse,
    |X - X_ref| <= 4 n_pad u (s |X_ref| 1 1^T |X_ref| + |X_ref| |B_ref| |X_ref|),
i.e. a block perturbed by as much as the factor bound allows plus the rounding of the inversion itself.
Neither bound is fitted to measured errors.  A failure names the offending tiles.

The switches are read once per process, so every switch setting runs in a worker process
(tools/lu_contract_case.py) that factors the matrices and writes the factors to an .npz.
"""
from __future__ import annotations

import functools
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.linalg as sla

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKER = os.path.join(ROOT, "tools", "lu_contract_case.py")
NB = 128
UNIT = 2.0 ** -53
PADS = (0, 1, 127)


def bound(n_pad: int) -> float:
    return 4 * n_pad * UNIT


# ----------------------------------------------------------------------------------------
# A. reference, generators, checker (numpy / scipy)
# ----------------------------------------------------------------------------------------
def lu_nopiv_ref(A, nb: int = NB) -> np.ndarray:
    """Blocked right-looking LU without pivoting in fp64: returns the packed L\\U (unit lower L)."""
    F = np.array(A, dtype=np.float64, copy=True)
    n = F.shape[0]
    for k0 in range(0, n, nb):
        k1 = min(k0 + nb, n)
        D = F[k0:k1, k0:k1]  # (view) unblocked elimination of the diagonal block
        for j in range(k1 - k0 - 1):
            D[j + 1:, j] /= D[j, j]
            D[j + 1:, j + 1:] -= np.outer(D[j + 1:, j], D[j, j + 1:])
        if k1 == n:
            break
        F[k1:, k0:k1] = sla.solve_triangular(D, F[k1:, k0:k1].T, trans="T", lower=False).T  # L21 = A21 U11^-1
        F[k0:k1, k1:] = sla.solve_triangular(D, F[k0:k1, k1:], lower=True, unit_diagonal=True)  # U12 = L11^-1 A12
        F[k1:, k1:] -= F[k1:, k0:k1] @ F[k0:k1, k1:]
    return F


def split_lu(F):
    n = F.shape[0]
    return np.tril(F, -1) + np.eye(n), np.triu(F)


def lu_scale(F) -> float:
    """s = max (|L| |U|) of packed factors (a magnitude: the product runs in fp32)."""
    L, U = split_lu(F)
    return float((np.abs(L).astype(np.float32) @ np.abs(U).astype(np.float32)).max())


def _pad(A_int, n_pad):
    """Identity padding, as scb_system_assemble writes it for n_int < n_pad."""
    A = np.eye(n_pad)
    n = A_int.shape[0]
    A[:n, :n] = A_int
    return A


def _dominant(R, margin, rng=None):
    """R with its diagonal replaced: |d_i| = (1 + margin) max(row sum, column sum, 1/4) of |R| off the
    diagonal, negative (random signs when rng is given)."""
    np.fill_diagonal(R, 0.0)
    a = np.abs(R)
    d = (1.0 + margin) * np.maximum(np.maximum(a.sum(0), a.sum(1)), 0.25)
    sign = -1.0 if rng is None else rng.choice([-1.0, 1.0], size=len(d))
    np.fill_diagonal(R, sign * d)
    return R


def g1(n_int, n_pad, seed, sym=False):
    """General, row- and column-diagonally dominant with a 5 % margin (the unpivoted general systems);
    sym=True: its symmetric, negative definite variant."""
    rng = np.random.default_rng(seed)
    R = rng.uniform(-1.0, 1.0, (n_int, n_int)) / n_int
    if sym:
        return _pad(_dominant((R + R.T) / 2, 0.05), n_pad)
    return _pad(_dominant(R, 0.05, rng), n_pad)


def g2(n_int, n_pad, seed, m=256, c=0.25):
    """Symmetric negative definite, not diagonally dominant: S = -(B B^T / m + c I), B Gaussian n x m.
    Its Schur complements fall from ~1 + c to ~c on the diagonal within the first m steps."""
    rng = np.random.default_rng(seed)
    B = rng.standard_normal((n_int, m))
    S = -(B @ B.T / m + c * np.eye(n_int))
    return _pad((S + S.T) / 2, n_pad)


def g3(n_int, n_pad, seed):
    """P B with B column-dominant (margin 50 %) and P a random permutation of the real rows: partial
    pivoting undoes P, row r of P A is row argsort(p)[r] of A.  Returns (A, that permutation)."""
    rng = np.random.default_rng(seed)
    B = _dominant(rng.uniform(-1.0, 1.0, (n_int, n_int)) / n_int, 0.5, rng)
    p = rng.permutation(n_int)
    return _pad(B[p], n_pad), np.argsort(p)


def g4(n_int, n_pad, seed):
    """Plain Gaussian: generic partial pivoting."""
    return _pad(np.random.default_rng(seed).standard_normal((n_int, n_int)), n_pad)


GENS = {"g1": lambda n, p, s: g1(n, p, s), "g1s": lambda n, p, s: g1(n, p, s, sym=True), "g2": g2,
        "g3": lambda n, p, s: g3(n, p, s)[0], "g4": g4}
KIND_OF = {"g1": "gen", "g1s": "sym", "g2": "sym", "g3": "piv", "g4": "piv"}


@functools.lru_cache(maxsize=20)
def reference(gen: str, nb: int, pad: int, seed: int = 0):
    """(A, F_ref, s, piv_ref) of a generated matrix; piv kinds: scipy.linalg.lu_factor's factors."""
    n_pad = nb * NB
    A = GENS[gen](n_pad - pad, n_pad, 1000 * nb + 7 * pad + seed)
    if KIND_OF[gen] == "piv":
        F, piv = sla.lu_factor(A, check_finite=False)
    else:
        F, piv = lu_nopiv_ref(A), None
    for a in (A, F):
        a.setflags(write=False)
    return A, F, lu_scale(F), piv


def factor_errors(F, F_ref, s):
    """e[I, J] = max over the 128 x 64 tile (I, J) of |F - F_ref| / s (non-finite entries -> inf)."""
    n = F.shape[0]
    d = np.abs(np.asarray(F, dtype=np.float64) - F_ref)
    d[~np.isfinite(d)] = np.inf
    return d.reshape(n // NB, NB, n // 64, 64).max(axis=(1, 3)) / s


def dinv_errors(dinv, F_ref, s):
    """e[k, w, J]: block k, w = 0 inv(L_kk) / 1 inv(U_kk), 64-column tile J, of
    |X - X_ref| / (s |X_ref| 1 1^T |X_ref| + |X_ref| |B_ref| |X_ref|)."""
    nb = F_ref.shape[0] // NB
    e = np.empty((nb, 2, 2))
    for k in range(nb):
        Dk = F_ref[k * NB:(k + 1) * NB, k * NB:(k + 1) * NB]
        Lk, Uk = split_lu(Dk)
        for w, B in enumerate((Lk, Uk)):
            Xr = sla.solve_triangular(B, np.eye(NB), lower=(w == 0), unit_diagonal=(w == 0))
            aX = np.abs(Xr)
            W = s * np.outer(aX.sum(1), aX.sum(0)) + aX @ np.abs(B) @ aX
            d = np.abs(np.asarray(dinv[k, w], dtype=np.float64) - Xr) / W
            d[~np.isfinite(d)] = np.inf
            e[k, w] = d.reshape(NB, 2, 64).max(axis=(0, 2))
    return e


def check_factors(F, dinv, F_ref, s, what=""):
    """Asserts every factor tile and block-inverse tile is within bound(n_pad); returns the worst
    normalized errors (factor, dinv)."""
    n_pad = F_ref.shape[0]
    b = bound(n_pad)
    ef = factor_errors(F, F_ref, s)
    ed = dinv_errors(dinv, F_ref, s) if dinv is not None else np.zeros(1)
    bad_f = [tuple(int(v) for v in t) for t in np.argwhere(~(ef <= b))]
    bad_d = [tuple(int(v) for v in t) for t in np.argwhere(~(ed <= b))]
    msg = []
    if bad_f:
        msg.append(f"factor tiles (128-row block, 64-column block) over the bound: {bad_f[:12]}"
                   f"{' ...' if len(bad_f) > 12 else ''} (worst {ef.max():.3e})")
    if bad_d:
        msg.append(f"block-inverse tiles (block, 0 = invL / 1 = invU, 64-column half) over the bound: "
                   f"{bad_d[:12]}{' ...' if len(bad_d) > 12 else ''} (worst {ed.max():.3e})")
    assert not msg, f"{what} n_pad={n_pad} bound {b:.3e}: " + "; ".join(msg)
    return float(ef.max()), float(ed.max())


def ref_dinv(F):
    nb = F.shape[0] // NB
    out = np.empty((nb, 2, NB, NB))
    for k in range(nb):
        Lk, Uk = split_lu(F[k * NB:(k + 1) * NB, k * NB:(k + 1) * NB])
        out[k, 0] = sla.solve_triangular(Lk, np.eye(NB), lower=True, unit_diagonal=True)
        out[k, 1] = sla.solve_triangular(Uk, np.eye(NB), lower=False)
    return out


def solve_residual(F, B0, X):
    """Per column ||B0 - L (U X)||_inf / ||L| (|U| |X|)|_inf with the packed factors F."""
    L, U = split_lu(F)
    r = np.abs(B0 - L @ (U @ X)).max(axis=0)
    w = (np.abs(L) @ (np.abs(U) @ np.abs(X))).max(axis=0)
    return r / w


# ---- CPU: the reference and the checker -------------------------------------------------
@pytest.mark.parametrize("n", [1, 127, 128, 300, 513])
def test_reference_matches_lapack_without_interchanges(n):
    """On a column-diagonally-dominant matrix LAPACK dgetrf makes no interchange: then its factors are
    those of the unpivoted elimination."""
    A = _dominant(np.random.default_rng(n).uniform(-1, 1, (n, n)) / n, 0.05, np.random.default_rng(1))
    lu, piv = sla.lu_factor(A)
    assert np.array_equal(piv, np.arange(n))
    F = lu_nopiv_ref(A)
    n_pad = -(-n // NB) * NB
    assert factor_errors(_pad(F, n_pad), _pad(lu, n_pad), lu_scale(lu)).max() <= bound(n_pad)


@pytest.mark.parametrize("n", [5, 128, 257, 400])
def test_reference_matches_cholesky(n):
    """-S = C C^T  =>  S = L U with L = C diag(C)^-1, U = -diag(C) C^T."""
    S = g2(n, n, seed=n, m=max(n // 2, 1))
    C = np.linalg.cholesky(-S)
    dC = np.diag(C)
    F_chol = np.tril(C / dC[None, :], -1) + np.triu(-(dC[:, None] * C.T))
    F = lu_nopiv_ref(S)
    n_pad = -(-n // NB) * NB
    e = factor_errors(_pad(F, n_pad), _pad(F_chol, n_pad), lu_scale(F_chol))
    assert e.max() <= bound(n_pad), e.max()


def test_generators():
    n_int, n_pad = 300, 384
    for gen in GENS:
        A = GENS[gen](n_int, n_pad, 3)
        assert np.array_equal(A[n_int:], np.eye(n_pad)[n_int:]) and not A[:n_int, n_int:].any(), gen
    A = g1(n_int, n_pad, 3)[:n_int, :n_int]
    off = np.abs(A).sum(1) - np.abs(np.diag(A))
    assert (np.abs(np.diag(A)) >= 1.05 * off * (1 - 1e-12)).all()
    offc = np.abs(A).sum(0) - np.abs(np.diag(A))
    assert (np.abs(np.diag(A)) >= 1.05 * offc * (1 - 1e-12)).all()
    S = g2(n_int, n_pad, 3)[:n_int, :n_int]
    assert np.array_equal(S, S.T) and np.linalg.eigvalsh(S).max() < 0
    assert (np.abs(np.diag(S)) < np.abs(S).sum(1) - np.abs(np.diag(S))).any()  # not dominant
    A, perm = g3(n_int, n_pad, 3)
    lu, piv = sla.lu_factor(A)
    assert np.array_equal(perm_from_piv(piv)[:n_int], perm)


def perm_from_piv(piv):
    """Row r of P A is row perm[r] of A, for LAPACK-style interchanges piv."""
    perm = np.arange(len(piv))
    for k, p in enumerate(piv):
        perm[[k, p]] = perm[[p, k]]
    return perm


def test_checker_names_injected_faults():
    """Fault injection: drop one K = 128 contribution from one 64 x 32 tile of the reference factors,
    and perturb one entry of one block inverse; the checker flags exactly those tiles and passes the
    unmodified copies."""
    nb, pad = 5, 37
    A, F_ref, s, _ = reference("g1", nb, pad)
    D_ref = ref_dinv(F_ref)
    assert check_factors(F_ref.copy(), D_ref, F_ref, s) == (0.0, 0.0)
    # a tile of rows 320..383 (block row 2, the first half), columns 416..447 (64-column block 6)
    # misses the contribution of the inner panel k = 1
    F = F_ref.copy()
    r, c, k = slice(320, 384), slice(416, 448), slice(128, 256)
    F[r, c] += F_ref[r, k] @ F_ref[k, c]
    with pytest.raises(AssertionError, match=r"factor tiles .*: \[\(2, 6\)\] "):
        check_factors(F, D_ref, F_ref, s)
    assert np.array_equal(np.argwhere(factor_errors(F, F_ref, s) > bound(nb * NB)), [[2, 6]])
    D = D_ref.copy()
    D[3, 1, 17, 100] += 1e-9 * np.abs(D_ref[3, 1]).max()
    with pytest.raises(AssertionError, match=r"block-inverse tiles .*: \[\(3, 1, 1\)\] "):
        check_factors(F_ref, D, F_ref, s)


def test_pivot_workspace_fits_every_outer_panel_width():
    """scb_getrf_dinv_bytes must leave room for the pivot search of scb_getrf_piv (a 128-column
    panel copied twice + two candidate arrays) behind the first pack set for every SCB_LU_Q."""
    code = ("from superscreen_b200 import _lib\n"
            "L = _lib.load_library()\n"
            "print(*[L.scb_getrf_dinv_bytes(n) for n in (128, 1280, 12416)])\n")
    for q in (1, 2, 8):
        env = dict(os.environ, SCB_LU_Q=str(q), PYTHONPATH=ROOT)
        out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600,
                             cwd=ROOT)
        assert out.returncode == 0, out.stderr
        for n_pad, got in zip((128, 1280, 12416), map(int, out.stdout.split())):
            nb = n_pad // NB
            need = nb * 2 * NB * NB + 2 * n_pad * NB * q + 2 * n_pad * NB + 4 * -(-n_pad // 64) + nb
            assert got >= 8 * need, (q, n_pad, got, 8 * need)


# ----------------------------------------------------------------------------------------
# B. GPU contract tests
# ----------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def L():
    import torch

    assert torch.cuda.is_available()
    from superscreen_b200 import _lib

    return _lib.lib()


class Buffers:
    """(M, dinv, info[, piv, perm]) of one n_pad on the device."""

    def __init__(self, n_pad, piv=False):
        import torch

        from superscreen_b200 import _lib

        self.n_pad = n_pad
        L = _lib.lib()
        self.M = torch.empty(n_pad, n_pad, dtype=torch.float64, device="cuda")
        self.dinv = torch.zeros(int(L.scb_getrf_dinv_bytes(n_pad)) // 8, dtype=torch.float64, device="cuda")
        self.info = torch.zeros(1, dtype=torch.int32, device="cuda")
        self.piv = torch.empty(n_pad, dtype=torch.int32, device="cuda") if piv else None
        self.perm = torch.empty(n_pad, dtype=torch.int32, device="cuda") if piv else None

    def factor(self, A, kind):
        """Copies A into M (same buffer) and factors it on torch's current stream (no sync)."""
        import torch

        from superscreen_b200 import _lib

        L = _lib.lib()
        self.M.copy_(torch.tensor(A) if isinstance(A, np.ndarray) else A)
        sp = _lib.stream_ptr()
        if kind == "piv":
            _lib.check(L.scb_getrf_piv(self.n_pad, _lib.ptr(self.M), _lib.ptr(self.dinv), _lib.ptr(self.piv),
                                       _lib.ptr(self.perm), _lib.ptr(self.info), sp))
        else:
            getrf = L.scb_getrf_sym_nopiv if kind == "sym" else L.scb_getrf_nopiv
            _lib.check(getrf(self.n_pad, _lib.ptr(self.M), _lib.ptr(self.dinv), _lib.ptr(self.info), sp))
        return self

    def host(self):
        import torch

        torch.cuda.synchronize()
        nb = self.n_pad // NB
        return (self.M.cpu().numpy(), self.dinv[: nb * 2 * NB * NB].cpu().numpy().reshape(nb, 2, NB, NB),
                int(self.info.item()))


def _check_piv(piv, perm, F, piv_ref, n_int, what):
    assert np.array_equal(piv, piv_ref), f"{what}: piv differs from LAPACK at rows {np.flatnonzero(piv != piv_ref)[:10]}"
    assert np.array_equal(perm, perm_from_piv(piv)), f"{what}: perm inconsistent with piv"
    n_pad = len(piv)
    assert np.array_equal(perm[n_int:], np.arange(n_int, n_pad)), f"{what}: a padding row was interchanged"
    # multipliers come from products with inv(U_kk), not from divisions: |L| <= 1 up to the factor bound
    assert np.abs(np.tril(F, -1)).max() <= 1.0 + bound(n_pad), f"{what}: |L| > 1"


FACTOR_NBS = (1, 2, 3, 7, 8, 9, 10, 15, 16, 17, 24, 25, 41)
FACTOR_GENS = ("g2", "g1s", "g1", "g3", "g4")


def _pad_of(gen, nb):
    return PADS[(FACTOR_NBS.index(nb) + FACTOR_GENS.index(gen)) % 3] if nb in FACTOR_NBS else PADS[nb % 3]


def _run_case(gen, nb, pad, what):
    A, F_ref, s, piv_ref = reference(gen, nb, pad)
    kind = KIND_OF[gen]
    buf = Buffers(nb * NB, piv=kind == "piv").factor(A, kind)
    F, D, info = buf.host()
    assert info == 0, f"{what}: info = {info}"
    if kind == "piv":
        _check_piv(buf.piv.cpu().numpy(), buf.perm.cpu().numpy(), F, piv_ref, nb * NB - pad, what)
    ef, ed = check_factors(F, D, F_ref, s, what)
    print(f"[lu-contract] {what:<28s} factor {ef:.3e} dinv {ed:.3e} bound {bound(nb * NB):.3e}")
    return buf


@pytest.mark.gpu
@pytest.mark.parametrize("gen", FACTOR_GENS)
@pytest.mark.parametrize("nb", FACTOR_NBS)
def test_factor_sweep(L, gen, nb):
    """Every block-schedule edge: one block, a partial / full / one-block-wide last outer panel, two and
    three or more outer panels (alternating pack sets, bulk update), padding 0 / 1 / 127."""
    pad = _pad_of(gen, nb)
    _run_case(gen, nb, pad, f"{KIND_OF[gen]}/{gen} nb={nb} pad={pad}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["sym", "gen"])
def test_factor_at_graph_limit(L, kind):
    """n_pad = 12416 (97 blocks) and its leading 12288 x 12288 block (96 blocks: the largest size that is
    graph-captured), each factored twice through the same buffers (at 12288 the second call is captured
    and replayed).  Without pivoting the factors of a leading block are the leading block of the factors,
    so one host reference serves both sizes."""
    gen = "g1s" if kind == "sym" else "g1"
    n97, n96 = 97 * NB, 96 * NB
    A = GENS[gen](n97 - 1, n97, 97)
    F_ref = lu_nopiv_ref(A)
    Lr, Ur = split_lu(F_ref)
    P = np.abs(Lr).astype(np.float32) @ np.abs(Ur).astype(np.float32)
    del Lr, Ur
    for n, s in ((n96, float(P[:n96, :n96].max())), (n97, float(P.max()))):
        buf = Buffers(n)
        for rep in range(2):
            F, D, info = buf.factor(A[:n, :n], kind).host()
            assert info == 0
            ef, ed = check_factors(F, D, F_ref[:n, :n], s, f"{kind} nb={n // NB} call {rep}")
            print(f"[lu-contract] {kind}/{gen} nb={n // NB} call {rep}: factor {ef:.3e} dinv {ed:.3e} "
                  f"bound {bound(n):.3e}")
        del buf


SOLVE_NRHS = (1, 2, 7, 8, 9, 15, 16, 17, 31, 64, 127, 128, 129, 200, 256)


@pytest.mark.gpu
@pytest.mark.parametrize("gen", ["g2", "g1", "g4"])
@pytest.mark.parametrize("nb", [1, 9, 17, 41])
def test_triangular_solves(L, gen, nb):
    """scb_getrs_nopiv for 1 .. 256 right-hand sides (one sweep, 8-column chains, 16-column chains and
    the second pass of chains beyond 128 columns), and the pivoted path through solve_film.lu_solve.
    Each column: residual ||b - L U x||_inf <= 4 n_pad u ||L| |U| |x||_inf with the device factors
    (themselves checked against the reference), and the solution against scipy.linalg.lu_solve on the
    reference factors within 2 kappa_1(A) 4 n_pad u ||L||_1 ||U||_1 / ||A||_1."""
    import torch

    from superscreen_b200 import _lib
    from superscreen_b200.solver.solve_film import LinearSystem, lu_solve

    kind = KIND_OF[gen]
    pad = _pad_of(gen, nb)
    n_pad, n_int = nb * NB, nb * NB - pad
    what = f"{kind}/{gen} nb={nb} pad={pad}"
    buf = _run_case(gen, nb, pad, what)
    A, F_ref, s, piv_ref = reference(gen, nb, pad)
    F = buf.M.cpu().numpy()
    b = bound(n_pad)
    anorm = np.abs(A).sum(0).max()
    rcond, _ = sla.lapack.dgecon(F_ref, anorm, norm="1")
    Lr, Ur = split_lu(F_ref)
    fwd_bound = 2.0 / rcond * b * np.abs(Lr).sum(0).max() * np.abs(Ur).sum(0).max() / anorm
    rng = np.random.default_rng(nb)
    worst_r = worst_f = 0.0
    for nrhs in SOLVE_NRHS:
        H = rng.standard_normal((n_int, nrhs))
        if kind == "piv":
            system = LinearSystem(indices=np.arange(n_int), n_pad=n_pad, lu=buf.M, dinv=buf.dinv,
                                  piv=buf.piv, perm=buf.perm[:n_int].to(torch.int64))
            X = lu_solve(system, torch.from_numpy(H).cuda()).cpu().numpy()
            B0 = np.zeros((n_pad, nrhs))
            B0[:n_int] = H[perm_from_piv(piv_ref)[:n_int]]
        else:
            B0 = np.zeros((n_pad, nrhs))
            B0[:n_int] = H
            B = torch.from_numpy(B0).cuda()
            _lib.check(L.scb_getrs_nopiv(n_pad, _lib.ptr(buf.M), _lib.ptr(buf.dinv), nrhs, _lib.ptr(B),
                                         _lib.stream_ptr()))
            X = B.cpu().numpy()[:n_int]
        Xp = np.zeros((n_pad, nrhs))
        Xp[:n_int] = X
        res = solve_residual(F, B0, Xp)
        Xref = sla.lu_solve((F_ref, piv_ref if piv_ref is not None else np.arange(n_pad)), _pad_rhs(H, n_pad))[:n_int]
        fwd = np.abs(X - Xref).sum(0) / np.abs(Xref).sum(0)
        bad = [c for c in range(nrhs) if not (res[c] <= b and fwd[c] <= fwd_bound)]
        assert not bad, (f"{what} nrhs={nrhs}: columns {bad[:10]} residual {res.max():.3e} (bound {b:.3e}) "
                         f"forward {fwd.max():.3e} (bound {fwd_bound:.3e})")
        worst_r, worst_f = max(worst_r, res.max()), max(worst_f, fwd.max())
    print(f"[lu-contract] solve {what}: residual {worst_r:.3e} (bound {b:.3e}) forward {worst_f:.3e} "
          f"(bound {fwd_bound:.3e})")


def _pad_rhs(H, n_pad):
    B = np.zeros((n_pad, H.shape[1]))
    B[: H.shape[0]] = H
    return B


@pytest.mark.gpu
def test_pivot_ties_follow_lapack(L):
    """Exact ties |a_r1| = |a_r2| (one negative) as the column maximum in the first column of panels 0,
    1 and 8, rows untouched by earlier elimination: the lower row wins, as in LAPACK.  The tied rows
    sit in different 64-row CTAs of the pivot search, in the same warp, and in the last CTA that holds
    real rows (partly padding)."""
    nb, n_int = 10, 1243
    n_pad = nb * NB
    rng = np.random.default_rng(11)
    B = _dominant(rng.uniform(-1.0, 1.0, (n_int, n_int)) / n_int, 0.5, rng)
    # (column c, row r1 holding B's row c, row r2 > r1 holding B's row j2 > c)
    ties = [(0, 0, 100), (128, 133, n_int - 1), (1024, 1025, 1026), (1152, 1215, 1216)]
    order = list(rng.permutation(n_int))
    for c, r1, r2 in ties:  # put B's row c at position r1 and some later row of B at r2
        for pos, brow in ((r1, c), (r2, c + 1 + 40 + (r2 % 50))):
            i = order.index(brow)
            order[i], order[pos] = order[pos], order[i]
    Ai = B[order]
    for c, r1, r2 in ties:
        Ai[[r1, r2], :c] = 0.0
        t = 2.0 * np.abs(Ai[:, c]).sum()
        sgn = rng.choice([-1.0, 1.0])
        Ai[r1, c], Ai[r2, c] = sgn * t, -sgn * t
    A = _pad(Ai, n_pad)
    F_ref, piv_ref = sla.lu_factor(A)
    for c, r1, _ in ties:
        assert piv_ref[c] == r1, (c, piv_ref[c], r1)
    buf = Buffers(n_pad, piv=True).factor(A, "piv")
    F, D, info = buf.host()
    assert info == 0
    _check_piv(buf.piv.cpu().numpy(), buf.perm.cpu().numpy(), F, piv_ref, n_int, "ties")
    check_factors(F, D, F_ref, lu_scale(F_ref), "ties")


SINGULAR_AT = (0, 127, 128, 1023, 1024, None)  # None: the last real row


@pytest.mark.gpu
@pytest.mark.parametrize("gen", ["g2", "g1", "g3"])
def test_singular_and_nonfinite_pivots_then_reuse(L, gen):
    """A zero row and column at k gives info = k + 1 (for the pivoted LU: LAPACK dgetrf's info), a NaN
    diagonal entry at k info = k + 1 for the unpivoted LUs; the same buffers then factor a healthy
    matrix with info = 0 and correct factors.  The unpivoted calls after the first one are captured
    and replayed from a CUDA graph, so its info reset must be part of the graph."""
    nb, pad = 10, 37
    kind = KIND_OF[gen]
    A, F_ref, s, piv_ref = reference(gen, nb, pad)
    n_int = nb * NB - pad
    buf = Buffers(nb * NB, piv=kind == "piv")
    faults = [("zero", k) for k in SINGULAR_AT] + ([("nan", k) for k in SINGULAR_AT] if kind != "piv" else [])
    for what, k in faults:
        k = n_int - 1 if k is None else k
        Ab = A.copy()
        if what == "zero":
            Ab[k, :] = 0.0
            Ab[:, k] = 0.0
        else:
            Ab[k, k] = np.nan
        _, _, info = buf.factor(Ab, kind).host()
        expect = k + 1
        if kind == "piv":
            expect = sla.lapack.dgetrf(Ab)[2]
            assert expect == k + 1
        assert info == expect, f"{gen} {what} at {k}: info {info}, expected {expect}"
        F, D, info = buf.factor(A, kind).host()
        assert info == 0, f"{gen}: info {info} after a healthy factorization following a {what} pivot at {k}"
        check_factors(F, D, F_ref, s, f"{gen} after {what} at {k}")
        if kind == "piv":
            _check_piv(buf.piv.cpu().numpy(), buf.perm.cpu().numpy(), F, piv_ref, n_int, gen)


def _write_cases(path, cases):
    np.savez(path, **{f"a{i}": A for i, (A, _) in enumerate(cases)},
             **{f"kind{i}": kind for i, (_, kind) in enumerate(cases)})


def _start_worker(src, dst, env_extra):
    """tools/lu_contract_case.py src dst with only the switches of env_extra set."""
    env = {k: v for k, v in os.environ.items() if not k.startswith(("SCB_LU", "SCB_DIAG"))}
    env.update(env_extra)
    env["PYTHONPATH"] = ROOT + (os.pathsep + env["PYTHONPATH"] if env.get("PYTHONPATH") else "")
    return subprocess.Popen([sys.executable, WORKER, str(src), str(dst)], env=env, stdout=subprocess.PIPE,
                            stderr=subprocess.STDOUT, text=True, cwd=ROOT)


def _finish_worker(proc, dst, env_extra, timeout=900):
    """Waits for the worker (killed on timeout) and returns its outputs; the .npz is removed."""
    try:
        log, _ = proc.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        proc.kill()
        log, _ = proc.communicate()
    assert proc.returncode == 0, f"worker {env_extra} failed (rc {proc.returncode}):\n{log[-4000:]}"
    with np.load(dst) as z:
        res = {k: z[k] for k in z.files}
    dst.unlink()
    return res


def _digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


@pytest.mark.gpu
def test_graph_replay_with_changing_contents(L, tmp_path):
    """Four different matrices through one (M, dinv, info) triple -- direct, capture, replay, replay --
    each equal to its own reference and bit-identical to SCB_LU_GRAPH=0; then more than 96 triples,
    three calls each, so that the LRU table evicts captured graphs, all still correct."""
    nb, pad = 9, 1
    runs = {}
    for kind, gen in (("sym", "g2"), ("gen", "g1")):
        buf = Buffers(nb * NB)
        for seed in range(4):
            A, F_ref, s, _ = reference(gen, nb, pad, seed)
            F, D, info = buf.factor(A, kind).host()
            assert info == 0
            check_factors(F, D, F_ref, s, f"{kind} call {seed}")
            runs[(kind, seed)] = (A, _digest(F, D))
    _write_cases(tmp_path / "in.npz", [(A, kind) for (kind, _), (A, _) in runs.items()])
    proc = _start_worker(tmp_path / "in.npz", tmp_path / "out.npz", {"SCB_LU_GRAPH": "0"})
    ref = _finish_worker(proc, tmp_path / "out.npz", {"SCB_LU_GRAPH": "0"})
    for i, (key, (_, dg)) in enumerate(runs.items()):
        assert _digest(ref[f"lu{i}"], ref[f"dinv{i}"]) == dg, f"{key}: graph replay differs from SCB_LU_GRAPH=0"
    # LRU eviction: 100 triples x 3 calls, then the first 8 triples again (their graphs were evicted)
    nb, n_pad = 2, 256
    pool = [(kind, *reference(gen, nb, p, seed)) for seed in range(3) for kind, gen, p in
            (("sym", "g2", 0), ("gen", "g1", 5))]
    bufs = [Buffers(n_pad) for _ in range(100)]
    order = [(t, c) for t in range(100) for c in range(3)] + [(t, c) for t in range(8) for c in range(3)]
    for t, c in order:
        kind, A, F_ref, s, _ = pool[(t % 2) + 2 * ((t + c) % 3)]
        F, D, info = bufs[t].factor(A, kind).host()
        assert info == 0
        check_factors(F, D, F_ref, s, f"triple {t} call {c}")


@pytest.mark.gpu
def test_concurrent_streams_bit_identical(L):
    """Four factorizations (sym and general, different nb) on four streams at once, as the film streams
    of a multi-film solve run them, equal bit for bit the same factorizations run one after another."""
    import torch

    cases = [("sym", "g2", 9), ("gen", "g1", 17), ("sym", "g1s", 25), ("gen", "g1", 3)]
    mats = [(kind, reference(gen, nb, 1)[0]) for kind, gen, nb in cases]
    seq = []
    for kind, A in mats:
        seq.append(Buffers(A.shape[0]).factor(A, kind).host())
    bufs = [Buffers(A.shape[0]) for _, A in mats]
    inputs = [torch.tensor(A).cuda() for _, A in mats]
    streams = [torch.cuda.Stream() for _ in mats]
    torch.cuda.synchronize()
    for (kind, _), buf, a, st in zip(mats, bufs, inputs, streams):
        with torch.cuda.stream(st):
            buf.factor(a, kind)
    for st in streams:
        torch.cuda.current_stream().wait_stream(st)
    for (F0, D0, i0), buf, (kind, gen, nb) in zip(seq, bufs, cases):
        F, D, info = buf.host()
        assert info == i0 == 0
        assert np.array_equal(F, F0) and np.array_equal(D, D0), f"{kind} nb={nb}: concurrent run differs"
        check_factors(F, D, *reference(gen, nb, 1)[1:3], f"concurrent {kind} nb={nb}")


@pytest.mark.gpu
def test_symmetric_reads_lower_triangle_only(L):
    """scb_getrf_sym_nopiv on a matrix whose strictly upper triangle holds NaN gives the factors of the
    full symmetric matrix, bit for bit."""
    for gen, nb in (("g2", 1), ("g2", 9), ("g1s", 17)):
        A, F_ref, s, _ = reference(gen, nb, 1)
        full = Buffers(nb * NB).factor(A, "sym").host()
        An = A.copy()
        An[np.triu_indices(nb * NB, 1)] = np.nan
        half = Buffers(nb * NB).factor(An, "sym").host()
        bad = np.argwhere(factor_errors(half[0], full[0], 1.0) != 0)
        assert half[2] == 0 and not len(bad), f"{gen} nb={nb}: factors depend on the upper triangle, tiles {bad[:10].tolist()}"
        assert np.array_equal(half[1], full[1])


SWEEP_NBS = (1, 3, 9, 17, 25)
SWEEP = [
    {"SCB_LU_Q": "1"}, {"SCB_LU_Q": "3"}, {"SCB_LU_Q": "4"}, {"SCB_LU_Q": "6"},
    {"SCB_LU_LOOKAHEAD": "0"}, {"SCB_LU_SPLIT": "0"}, {"SCB_LU_RECURSIVE": "0"}, {"SCB_LU_LAZY": "1"},
    {"SCB_DIAG_SMALL": "0"}, {"SCB_DIAG_SYMB": "0"}, {"SCB_LU_BAND": "0"}, {"SCB_LU_INNER_LA": "1"},
    {"SCB_LU_TAIL_Q": "2", "SCB_LU_TAIL_BLOCKS": "5"},
    {"SCB_LU_LAT": "0"}, {"SCB_LU_LAT": "1"}, {"SCB_LU_LAT": "7"}, {"SCB_LU_GRAPH": "0"},
]
BIT_IDENTICAL = ("SCB_LU_LAT", "SCB_LU_BAND", "SCB_LU_GRAPH")  # DESIGN.md section 6


def _sweep_cases():
    return [(gen, nb, _pad_of(gen, nb)) for gen in ("g2", "g1", "g4") for nb in SWEEP_NBS]


def _tag(env):
    return ",".join(f"{k}={v}" for k, v in env.items()) or "default"


def _check_sweep_output(out, tag):
    """(failures, worst (factor, dinv) error per case, digests) of one worker's factors."""
    failures, worst, digests = [], [], []
    for i, (gen, nb, pad) in enumerate(_sweep_cases()):
        kind = KIND_OF[gen]
        A, F_ref, s, piv_ref = reference(gen, nb, pad)
        what = f"[{tag}] {kind}/{gen} nb={nb} pad={pad}"
        digests.append(_digest(out[f"lu{i}"], out[f"dinv{i}"]))
        try:
            assert int(out[f"info{i}"]) == 0, f"{what}: info {int(out[f'info{i}'])}"
            if kind == "piv":
                _check_piv(out[f"piv{i}"], out[f"perm{i}"], out[f"lu{i}"], piv_ref, nb * NB - pad, what)
            worst.append(check_factors(out[f"lu{i}"], out[f"dinv{i}"], F_ref, s, what))
        except AssertionError as exc:
            failures.append(str(exc))
            worst.append((np.inf, np.inf))
    return failures, worst, digests


@pytest.fixture(scope="module")
def sweep_results(L, tmp_path_factory):
    """Runs the default and every SWEEP setting in worker processes, at most four at a time, and checks
    each output as it arrives: {tag: (failures, worst errors, digests)}."""
    work = tmp_path_factory.mktemp("lu_sweep")
    src = work / "in.npz"
    _write_cases(src, [(reference(*c)[0], KIND_OF[c[0]]) for c in _sweep_cases()])
    pending = [{}] + list(SWEEP)
    running, results = [], {}
    try:
        while pending or running:
            while pending and len(running) < 4:
                env = pending.pop(0)
                dst = work / f"out{len(results) + len(running)}.npz"
                running.append((env, dst, _start_worker(src, dst, env)))
            env, dst, proc = running.pop(0)
            try:
                out = _finish_worker(proc, dst, env)
                results[_tag(env)] = _check_sweep_output(out, _tag(env))
            except AssertionError as exc:
                results[_tag(env)] = ([str(exc)], [], [])
    finally:
        for _, _, proc in running:
            proc.kill()
            proc.communicate()
    return results


@pytest.mark.gpu
@pytest.mark.parametrize("env", SWEEP, ids=_tag)
def test_switch_sweep(sweep_results, env):
    """Every LU switch of DESIGN.md section 6, sym / general / pivoted at nb = 1, 3, 9, 17, 25: factors
    within the bound; the settings declared bit-identical also equal the default bit for bit."""
    failures, worst, digests = sweep_results[_tag(env)]
    d_fail, _, d_digests = sweep_results["default"]
    assert not d_fail, "\n".join(d_fail)
    if any(k in BIT_IDENTICAL for k in env) and not failures:
        for (gen, nb, pad), dg, d0 in zip(_sweep_cases(), digests, d_digests):
            if dg != d0:
                failures.append(f"[{_tag(env)}] {KIND_OF[gen]}/{gen} nb={nb}: not bit-identical to the default")
    for (gen, nb, pad), (ef, ed) in zip(_sweep_cases(), worst):
        print(f"[lu-contract] [{_tag(env)}] {KIND_OF[gen]}/{gen} nb={nb} pad={pad} factor {ef:.3e} dinv {ed:.3e} "
              f"bound {bound(nb * NB):.3e}")
    assert not failures, "\n".join(failures)
