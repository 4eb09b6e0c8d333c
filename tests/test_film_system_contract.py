"""Contract tests of the film system pieces that feed the dense LU and check its solutions --
scb_system_assemble (the matrix and its row-dominance margin), scb_kernel_diagonal, scb_apply_operator
(CUDA-core N-body and DMMA GEMM engines), scb_grad_lambda_term and the SCB_BS_VECTOR,
SCB_BS_VECTOR_POTENTIAL and multi-set SCB_BS_FILM_TO_FILM kinds of scb_biot_savart -- element by element
against an extended-precision reference of the same operation.

Reference.  Every pair term (q_ij w_j = w_j / (4 pi r^3), the Biot-Savart terms) is computed from the
fp64 inputs in np.longdouble (x86-64: 64-bit significand, eps = 2^-63) and every sum is accumulated in
np.longdouble, in row chunks so that a 6400^2 matrix or a 1000 x 1e5 pair sum fits in a few GB.  Its
own error is a few 2^-64 relative to the sum of the magnitudes of the terms: negligible next to the
fp64 bounds below.  The assembled matrix restates include/scb.h (scb_system_assemble):
    M[r,c] = q w_c + Lambda_c lap_rc + T_rc        (r != c; q w_c alone off the sparse pattern)
    M[r,r] = -(C_i + sum_{j != i} q_ij w_j) + Lambda_r lap_rr + T_rr
    S[r,c] = q s_r s_c + Lambda_c lap_rc s_r / s_c,   S[r,r] = M[r,r]   (symmetrised, s = sym_scale)
    identity padding, zero off-blocks,
and it is checked against oracle.port.build_system_2d on three goldens.

Bounds (u = 2^-53), derived, not fitted:
  * one pair term q w: dx, dy rounded once each (relative u), r^2 = dx^2 + dy^2 in <= 2 more roundings:
    r^2 within 4u; r^-3 amplifies that by 1.5 (6u); inv_r3 (scb_common.cuh) is within a few ulp
    (rsqrt seed of 2^-22.9 refined to O(e^3) < 2^-64, then ~5 roundings); w / (4 pi) and the products add
    ~3u: < 16u in all.  Dense entries are allowed 32 u |ref|.
  * a sparse entry adds Lambda lap + T (2 roundings, T an input) and, symmetrised, a scale ratio and a
    product (2 more): 32 u (|q w| + |Lambda lap| + |T|), times s_r / s_c when symmetrised.
  * a sum of K terms, each within 32 u of its own magnitude, summed in ANY order (any split, tile or
    pass order) is within (K - 1) u sum|terms| + 32 u sum|terms|: the bound (K + 32) u sum|terms|.  The
    diagonal, every row of scb_kernel_diagonal, scb_apply_operator, scb_grad_lambda_term and every
    Biot-Savart output gets this bound; K counts every term of the row (sources, C, sparse entries,
    an accumulated `out`).
  * the margin: |M_rr| - ((qdw_i - C_i) + sum_sparse (|M_rc| - q w_c)), each of its pieces within the
    bounds above and 4 more roundings: slack_r = (n + 64) u W_r, W_r = 2 (C_i + S_i) + |Lambda lap_rr|
    + |T_rr| + sum_sparse (2 q w + |Lambda lap| + |T|).  The device value must lie within slack_r of
    the documented bound |M_rr| - (S_i + sum_sparse (|M_rc| - q w_c)) (S_i = the sum over ALL j != i), and
    never above the exact margin |M_rr| - sum_{c != r} |M_rc| plus slack_r; when ix covers every vertex
    both coincide.
Errors are reported as err / bound: <= 1 passes.  A failure names its places: (64-row tile, 128-column
tile) of assemble_dense_kernel for matrices, (row) for margins, (target, column / set) for pair sums.
"""
from __future__ import annotations

import functools
import os
from types import SimpleNamespace

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import GOLDEN

UNIT = 2.0 ** -53
LD = np.longdouble
FOUR_PI = 16 * np.arctan(LD(1))
TR, TC = 64, 128          # assemble_dense_kernel tile
NB = 128                  # LU padding block
KTILE, GEMM_SRC = 256, 32  # N-body source tile, DMMA GEMM source tile


def _pad_of(n_int: int) -> int:
    return -(-n_int // NB) * NB


# ----------------------------------------------------------------------------------------
# A. reference, checker, fault injection (numpy / scipy)
# ----------------------------------------------------------------------------------------
def pair_qw(t_xy, s_xy, w):
    """q_ij w_j = w_j / (4 pi r_ij^3) in longdouble [len(t), len(s)], 0 where r = 0 (q_ii = 0)."""
    dx = LD(1) * t_xy[:, None, 0] - s_xy[None, :, 0]
    dy = LD(1) * t_xy[:, None, 1] - s_xy[None, :, 1]
    r2 = dx * dx + dy * dy
    with np.errstate(divide="ignore", invalid="ignore"):
        q = _ld(w)[None, :] / (FOUR_PI * r2 * np.sqrt(r2))
    q[r2 == 0] = 0
    return q


def _ld(a):
    return np.asarray(a, dtype=LD)


def _chunks(m, cols, budget=2 ** 22):
    step = max(1, budget // max(cols, 1))
    for a in range(0, m, step):
        yield a, min(a + step, m)


def row_sums(sites, w, targets):
    """S_i = sum_{j != i} q_ij w_j over every vertex j, for vertex indices `targets` (longdouble)."""
    S = np.zeros(len(targets), dtype=LD)
    for a, b in _chunks(len(targets), len(sites)):
        S[a:b] = pair_qw(sites[targets[a:b]], sites, w).sum(1)
    return S


class Film:
    """Host inputs of the assembly / operator entry points: sites, weights w, C, Lambda and the operator
    pattern (adjacency + identity, sorted rows, int32) with laplacian / gradient values on it."""

    def __init__(self, sites, elements, Lam):
        from oracle import port

        self.sites = np.ascontiguousarray(sites, dtype=np.float64)
        self.elements = np.ascontiguousarray(elements, dtype=np.int64)
        n = self.n = len(self.sites)
        self.w = port.vertex_areas(self.sites, self.elements)
        self.C = port.C_vector(self.sites)
        self.Lam = np.ascontiguousarray(np.broadcast_to(np.asarray(Lam, dtype=np.float64), (n,)))
        P = (port.adjacency_matrix(self.elements) + sp.identity(n, dtype=int, format="csr")).tocsr()
        P.sort_indices()
        self.indptr, self.indices = P.indptr.astype(np.int32), P.indices.astype(np.int32)
        self.rows = np.repeat(np.arange(n), np.diff(self.indptr))
        self.lap = self.on_pattern(port.laplace_operator(self.sites, self.elements, self.w))
        gx, gy = port.gradient_vertices(self.sites, self.elements)
        self.gx, self.gy = self.on_pattern(gx), self.on_pattern(gy)

    def on_pattern(self, X):
        """Values of the sparse matrix X on the operator pattern (absent entries 0)."""
        X = sp.coo_array(X)
        keys = self.rows.astype(np.int64) * self.n + self.indices
        pos = np.searchsorted(keys, X.row.astype(np.int64) * self.n + X.col)
        assert (keys[np.minimum(pos, len(keys) - 1)] == X.row.astype(np.int64) * self.n + X.col).all()
        out = np.zeros(len(keys))
        np.add.at(out, pos, X.data)
        return out

    def csr(self, data):
        return sp.csr_array((data, self.indices, self.indptr), shape=(self.n, self.n))


@functools.lru_cache(maxsize=None)
def golden_film(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    f = Film(g["in_sites"], g["in_elements"], g["in_Lambda"])
    f.name = name
    f.ix = np.asarray(g["out_system_indices"] if "out_system_indices" in g.files else g["in_interior_indices"])
    return f


def grad_lambda_ref(f, Lam):
    """T on the operator pattern and its bound (scb_grad_lambda_term)."""
    Lj = _ld(Lam)[f.indices]
    lx = np.add.reduceat(_ld(f.gx) * Lj, f.indptr[:-1])
    ly = np.add.reduceat(_ld(f.gy) * Lj, f.indptr[:-1])
    ax = np.add.reduceat(np.abs(f.gx * Lam[f.indices]), f.indptr[:-1])
    ay = np.add.reduceat(np.abs(f.gy * Lam[f.indices]), f.indptr[:-1])
    K = np.diff(f.indptr)[f.rows]
    T = lx[f.rows] * _ld(f.gx) + ly[f.rows] * _ld(f.gy)
    bound = (K + 32) * UNIT * (ax[f.rows] * np.abs(f.gx) + ay[f.rows] * np.abs(f.gy))
    return T, bound


class SystemRef:
    """Reference of scb_system_assemble for (film, ix, T, sym): rows on demand, margins for every row."""

    def __init__(self, f, ix, T=None, sym=None, row_tiles=None):
        self.f, self.ix, self.T, self.sym = f, np.asarray(ix, dtype=np.int64), T, sym
        self.n_int = len(self.ix)
        self.n_pad = _pad_of(self.n_int)
        self.pos = np.full(f.n, -1, dtype=np.int64)
        self.pos[self.ix] = np.arange(self.n_int)
        # rows whose diagonal and margin are evaluated (all, or those of the given 64-row tiles)
        self.rsel = np.arange(self.n_int) if row_tiles is None else np.concatenate(
            [np.arange(I * TR, min((I + 1) * TR, self.n_int)) for I in row_tiles])
        self.S = np.zeros(self.n_int, dtype=LD)
        self.S[self.rsel] = row_sums(f.sites, f.w, self.ix[self.rsel])  # sum over ALL j != i
        # sparse entries of the system rows: (row r, column c, vertex i, vertex j, pattern slot q)
        i_of_q = f.rows
        c_of_q = self.pos[f.indices]
        r_of_q = self.pos[i_of_q]
        keep = (r_of_q >= 0) & (c_of_q >= 0)
        self.q_slot = np.flatnonzero(keep)
        self.sr, self.sc = r_of_q[keep], c_of_q[keep]
        self.si, self.sj = i_of_q[keep], f.indices[keep].astype(np.int64)
        q = self.q_slot
        Tq = np.zeros(len(q)) if T is None else np.asarray(T)[q]
        self.s_val = _ld(f.Lam[self.sj]) * _ld(f.lap[q]) + _ld(Tq)  # Lambda_c lap_rc + T_rc
        self.s_abs = np.abs(f.Lam[self.sj] * f.lap[q]) + np.abs(Tq)
        xy_i, xy_j = f.sites[self.si], f.sites[self.sj]
        off = self.sr != self.sc
        self.qw = np.zeros(len(q), dtype=LD)
        self.qw[off] = pair_qw_pairs(xy_i[off], xy_j[off], f.w[self.sj[off]])
        self._margins()

    def _margins(self):
        f, n_int = self.f, self.n_int
        Cx = _ld(f.C[self.ix])
        diag_s = np.zeros(n_int, dtype=LD)
        diag_abs = np.zeros(n_int)
        on = self.sr == self.sc
        np.add.at(diag_s, self.sr[on], self.s_val[on])
        np.add.at(diag_abs, self.sr[on], self.s_abs[on])
        self.diag = -(Cx + self.S) + diag_s
        self.diag_bound = (f.n + 32) * UNIT * (np.asarray(Cx + self.S, dtype=np.float64) + diag_abs)
        off = ~on
        Mrc = self.qw[off] + self.s_val[off]  # the general entry (margins are those of M)
        extra = np.zeros(n_int, dtype=LD)
        np.add.at(extra, self.sr[off], np.abs(Mrc) - self.qw[off])
        wsum = np.zeros(n_int)
        np.add.at(wsum, self.sr[off], 2 * np.asarray(self.qw[off], dtype=np.float64) + self.s_abs[off])
        dense_ix = np.zeros(n_int, dtype=LD)  # sum_{c in ix, c != r} q w_c
        rs = self.rsel
        for a, b in _chunks(len(rs), n_int):
            dense_ix[rs[a:b]] = pair_qw(f.sites[self.ix[rs[a:b]]], f.sites[self.ix], f.w[self.ix]).sum(1)
        self.exact_margin = np.abs(self.diag) - (dense_ix + extra)
        self.doc_margin = np.abs(self.diag) - (self.S + extra)
        W = 2 * np.asarray(Cx + self.S, dtype=np.float64) + diag_abs + wsum
        self.margin_slack = (f.n + 64) * UNIT * W

    def rows(self, r0, r1):
        """(reference longdouble [r1 - r0, n_pad], bound float64 of the same shape) of rows r0..r1."""
        f, n_int, n_pad = self.f, self.n_int, self.n_pad
        ref = np.zeros((r1 - r0, n_pad), dtype=LD)
        bnd = np.zeros((r1 - r0, n_pad))
        for r in range(max(r0, n_int), r1):
            ref[r - r0, r] = 1  # identity padding (exact)
        a, b = min(r0, n_int), min(r1, n_int)
        if a < b:
            xr = f.sites[self.ix[a:b]]
            if self.sym is None:
                D = pair_qw(xr, f.sites[self.ix], f.w[self.ix])
            else:
                s = _ld(self.sym[self.ix])
                D = pair_qw(xr, f.sites[self.ix], np.ones(n_int)) * s[a:b, None] * s[None, :]
            ref[: b - a, :n_int] = D
            bnd[: b - a, :n_int] = 32 * UNIT * np.abs(np.asarray(D, dtype=np.float64))
            sel = (self.sr >= a) & (self.sr < b) & (self.sr != self.sc)
            rr, cc = self.sr[sel] - r0, self.sc[sel]
            qw, sv, sa = self.qw[sel], self.s_val[sel], self.s_abs[sel]
            if self.sym is None:
                ref[rr, cc] = qw + sv
                bnd[rr, cc] = 32 * UNIT * (np.asarray(qw, dtype=np.float64) + sa)
            else:
                s_r, s_c = _ld(self.sym[self.si[sel]]), _ld(self.sym[self.sj[sel]])
                qs = qw / _ld(f.w[self.sj[sel]]) * s_r * s_c  # q s_r s_c
                ratio = s_r / s_c
                ref[rr, cc] = qs + sv * ratio
                bnd[rr, cc] = 32 * UNIT * (np.asarray(qs, dtype=np.float64)
                                           + sa * np.asarray(ratio, dtype=np.float64))
            d = np.arange(a, b)
            ref[d - r0, d] = self.diag[a:b]
            bnd[d - r0, d] = self.diag_bound[a:b]
        return ref, bnd


def pair_qw_pairs(xy_i, xy_j, w_j):
    """q w for matched pairs (longdouble [k])."""
    dx = _ld(xy_i[:, 0]) - xy_j[:, 0]
    dy = _ld(xy_i[:, 1]) - xy_j[:, 1]
    r2 = dx * dx + dy * dy
    return _ld(w_j) / (FOUR_PI * r2 * np.sqrt(r2))


def _ratio(got, ref, bnd):
    """|got - ref| / bnd (0 / 0 -> 0; any error against a zero bound, or a non-finite value -> inf)."""
    err = np.abs(np.asarray(_ld(got) - ref, dtype=np.float64))
    with np.errstate(divide="ignore", invalid="ignore"):
        q = np.where(err == 0, 0.0, err / bnd)
    q[~np.isfinite(q)] = np.inf
    q[~np.isfinite(np.asarray(got, dtype=np.float64))] = np.inf
    return q


def matrix_tile_errors(get_rows, sref: SystemRef, row_tiles=None):
    """e[I, J] = max err / bound over the (64-row tile I, 128-column tile J) of the workspace read by
    get_rows(r0, r1) (NaN for tiles not checked)."""
    n_pad = sref.n_pad
    e = np.full((n_pad // TR, n_pad // TC), np.nan)
    for I in range(n_pad // TR) if row_tiles is None else row_tiles:
        r0, r1 = I * TR, (I + 1) * TR
        ref, bnd = sref.rows(r0, r1)
        e[I] = _ratio(get_rows(r0, r1), ref, bnd).reshape(TR, n_pad // TC, TC).max(axis=(0, 2))
    return e


def check_tiles(e, what, tag="matrix"):
    """Asserts every checked tile <= 1; names offending tiles; returns the worst ratio."""
    bad = [tuple(int(v) for v in t) for t in np.argwhere(~(np.nan_to_num(e, nan=0.0) <= 1.0))]
    worst = float(np.nanmax(e)) if np.isfinite(e).any() or np.isinf(e).any() else 0.0
    assert not bad, (f"{what}: {tag} tiles (64-row tile, 128-column tile) over the bound: {bad[:12]}"
                     f"{' ...' if len(bad) > 12 else ''} (worst err/bound {worst:.3e})")
    return worst


def check_margin(got, sref: SystemRef, what, exact=None):
    """margin[r] <= exact[r] + slack[r] on every row; |margin - documented bound| <= slack (also
    |margin - exact| <= slack when ix covers every vertex).  Returns the worst |dev - doc| / slack."""
    rs = sref.rsel
    got = np.asarray(got, dtype=np.float64)[rs]
    slack = sref.margin_slack[rs]
    above = np.asarray(_ld(got) - sref.exact_margin[rs], dtype=np.float64) / slack
    dev = np.abs(np.asarray(_ld(got) - sref.doc_margin[rs], dtype=np.float64)) / slack
    bad_above = rs[~(above <= 1.0)]
    bad_doc = rs[~(dev <= 1.0)]
    msg = []
    if len(bad_above):
        msg.append(f"margin above the exact margin + slack at rows {bad_above[:12].tolist()} "
                   f"(worst {np.nanmax(above):.3e} slack)")
    if len(bad_doc):
        msg.append(f"margin off the documented bound at rows {bad_doc[:12].tolist()} (worst {np.nanmax(dev):.3e} slack)")
    if len(sref.ix) == sref.f.n:
        ex = np.abs(np.asarray(_ld(got) - sref.exact_margin[rs], dtype=np.float64)) / slack
        bad_ex = rs[~(ex <= 1.0)]
        if len(bad_ex):
            msg.append(f"ix covers every vertex but margin != exact margin at rows {bad_ex[:12].tolist()}")
    assert not msg, f"{what}: " + "; ".join(msg)
    return float(dev.max()) if len(dev) else 0.0


def check_sums(got, ref, bnd, what, cols="column"):
    """Pair sums [targets, columns]: err / bound <= 1 everywhere; names (target, column / set)."""
    q = _ratio(np.asarray(got).reshape(ref.shape), ref, bnd)
    bad = [tuple(int(v) for v in t) for t in np.argwhere(~(q <= 1.0))]
    assert not bad, (f"{what}: (target, {cols}) over the bound: {bad[:12]}{' ...' if len(bad) > 12 else ''} "
                     f"(worst err/bound {q.max():.3e})")
    return float(q.max()) if q.size else 0.0


def _report(what, worst, extra=""):
    print(f"[system-contract] {what:<58s} max err/bound {worst:.3e}{extra}")


# ---- the operator reference ------------------------------------------------------------
def operator_ref(sites, w, qdw, src, v, Lam=None, lap_csr=None, T=None, prefill=None):
    """scb_apply_operator: out = prefill + (-sum_{j in src, j != i} q_ij w_j v_j) + qdw_i v_i
    - sum_pattern (Lambda_j lap_ij + T_ij) v_j (the diagonal and sparse parts act on all of v).
    Returns (ref longdouble [n, k], bound)."""
    n, k = v.shape
    src = np.arange(n) if src is None else np.asarray(src, dtype=np.int64)
    ref = _ld(qdw)[:, None] * _ld(v)
    absum = np.abs(qdw[:, None] * v)
    K = np.full(n, len(src) + 1.0)
    if len(src):
        vs, avs = _ld(v[src]), np.abs(v[src])
        for a, b in _chunks(n, len(src), 2 ** 21):
            Q = pair_qw(sites[a:b], sites[src], w[src])
            ref[a:b] -= Q @ vs
            absum[a:b] += np.asarray(Q, dtype=np.float64) @ avs
    if Lam is not None:
        indptr, indices, lap = lap_csr
        rows = np.repeat(np.arange(n), np.diff(indptr))
        coef = _ld(Lam[indices]) * _ld(lap) + (0 if T is None else _ld(T))
        acoef = np.abs(Lam[indices] * lap) + (0 if T is None else np.abs(T))
        ref -= np.add.reduceat(coef[:, None] * _ld(v[indices]), indptr[:-1])
        absum += np.add.reduceat(acoef[:, None] * np.abs(v[indices]), indptr[:-1])
        K += np.diff(indptr)
    if prefill is not None:
        ref += _ld(prefill)
        absum += np.abs(prefill)
        K += 1
    return ref, (K[:, None] + 32) * UNIT * absum


def diag_ref(sites, w, C, targets=None):
    """scb_kernel_diagonal: qdw_i = C_i + sum_{j != i} q_ij w_j; (ref, bound) for `targets`."""
    t = np.arange(len(sites)) if targets is None else np.asarray(targets)
    S = row_sums(sites, w, t)
    ref = _ld(C[t]) + S
    return ref, (len(sites) + 32) * UNIT * np.abs(np.asarray(ref, dtype=np.float64))


# ---- Biot-Savart references -------------------------------------------------------------
BS_FILM_TO_FILM, BS_VECTOR, BS_VECPOT = 0, 2, 3


def bs_ref(kind, tgt, src, area, J, dz, pf):
    """(ref longdouble, bound) of scb_biot_savart for kind FILM_TO_FILM ([nsets, m]), VECTOR ([m, 3]),
    VECTOR_POTENTIAL ([m, 2]).  J: [nsets, n, 2] for FILM_TO_FILM, [n, 2] otherwise."""
    m, n = len(tgt), len(src)
    pfl = _ld(pf)
    if kind == BS_FILM_TO_FILM:
        ns = J.shape[0]
        ref, ab = np.zeros((ns, m), dtype=LD), np.zeros((ns, m))
        Pa = _ld(area)[None, :, None] * _ld(J)  # [ns, n, 2]
        for a, b in _chunks(m, n, 2 ** 20):
            dx = _ld(tgt[a:b, None, 0]) - src[None, :, 0]
            dy = _ld(tgt[a:b, None, 1]) - src[None, :, 1]
            r2 = dx * dx + dy * dy + _ld(dz) * _ld(dz)
            k3 = 1 / (r2 * np.sqrt(r2))
            Ky, Kx = k3 * dy, k3 * dx
            ref[:, a:b] = pfl * (Ky @ Pa[:, :, 0].T - Kx @ Pa[:, :, 1].T).T
            fKy, fKx = np.abs(np.asarray(Ky, dtype=np.float64)), np.abs(np.asarray(Kx, dtype=np.float64))
            aP = np.abs(np.asarray(Pa, dtype=np.float64))
            ab[:, a:b] = abs(pf) * (fKy @ aP[:, :, 0].T + fKx @ aP[:, :, 1].T).T
        return ref, (2 * n + 32) * UNIT * ab
    ncomp = 3 if kind == BS_VECTOR else 2
    ref, ab = np.zeros((m, ncomp), dtype=LD), np.zeros((m, ncomp))
    Px, Py = _ld(area) * _ld(J[:, 0]), _ld(area) * _ld(J[:, 1])
    aPx, aPy = np.abs(area * J[:, 0]), np.abs(area * J[:, 1])
    for a, b in _chunks(m, n, 2 ** 20):
        d = [_ld(tgt[a:b, None, c]) - src[None, :, c] for c in range(3)]
        r2 = d[0] * d[0] + d[1] * d[1] + d[2] * d[2]
        if kind == BS_VECPOT:
            k1 = 1 / np.sqrt(r2)
            ref[a:b, 0], ref[a:b, 1] = pfl * (k1 @ Px), pfl * (k1 @ Py)
            f1 = np.asarray(k1, dtype=np.float64)
            ab[a:b, 0], ab[a:b, 1] = abs(pf) * (f1 @ aPx), abs(pf) * (f1 @ aPy)
            continue
        k3 = 1 / (r2 * np.sqrt(r2))
        kd = [k3 * d[c] for c in range(3)]
        fkd = [np.abs(np.asarray(x, dtype=np.float64)) for x in kd]
        ref[a:b, 0] = pfl * (kd[2] @ Py)
        ref[a:b, 1] = -pfl * (kd[2] @ Px)
        ref[a:b, 2] = pfl * (kd[1] @ Px - kd[0] @ Py)
        ab[a:b, 0] = abs(pf) * (fkd[2] @ aPy)
        ab[a:b, 1] = abs(pf) * (fkd[2] @ aPx)
        ab[a:b, 2] = abs(pf) * (fkd[1] @ aPx + fkd[0] @ aPy)
    K = 2 * n if kind == BS_VECTOR else n
    return ref, (K + 32) * UNIT * ab


# ---- synthetic inputs --------------------------------------------------------------------
def jittered_points(n, seed, scale=1.0):
    """n distinct points: a shuffled jittered square lattice of spacing `scale` / sqrt(n)."""
    rng = np.random.default_rng(seed)
    k = int(np.ceil(np.sqrt(n)))
    g = np.stack(np.meshgrid(np.arange(k), np.arange(k), indexing="ij"), -1).reshape(-1, 2)[:n].astype(np.float64)
    g += rng.uniform(-0.35, 0.35, g.shape)
    return np.ascontiguousarray(rng.permutation(g) * (scale / k))


def random_pattern(n, seed, per_row=6):
    """CSR pattern with the diagonal and up to per_row other sorted columns per row; int32."""
    rng = np.random.default_rng(seed)
    cols = [np.unique(np.concatenate([[i], rng.integers(0, n, min(per_row, n))])) for i in range(n)]
    indptr = np.concatenate([[0], np.cumsum([len(c) for c in cols])]).astype(np.int32)
    return indptr, np.concatenate(cols).astype(np.int32)


# ---- CPU tests of the reference and the checker -----------------------------------------
@pytest.mark.parametrize("name", ["ring", "square_inhomogeneous", "transport"])
def test_reference_matches_oracle_system(name):
    """The restated assembly reference against oracle.port.build_system_2d (-A, fp64) on a golden mesh,
    within the entry bounds; with T for the inhomogeneous Lambda of square_inhomogeneous."""
    from oracle import port

    f = golden_film(name)
    om = port.build_mesh(f.sites, f.elements)
    inhom = port.lambda_inhomogeneous(f.Lam)
    glt = port.grad_Lambda_term_sparse(om, f.Lam).toarray() if inhom else 0
    T = None
    if inhom:
        T = np.asarray(grad_lambda_ref(f, f.Lam)[0], dtype=np.float64)
    sref = SystemRef(f, f.ix, T=T)
    A = port.build_system_2d(om.Q, om.vertex_areas, f.Lam, om.laplacian.toarray(), glt, f.ix)
    M = np.eye(sref.n_pad)
    M[: sref.n_int, : sref.n_int] = -A
    e = matrix_tile_errors(lambda a, b: M[a:b], sref)
    worst = check_tiles(e, f"{name} oracle build_system_2d")
    if name == "square_inhomogeneous":  # the golden of the live reference, through the oracle
        g = np.load(os.path.join(GOLDEN, name + ".npz"))
        assert np.abs(A - g["out_A"]).max() <= 1e-12 * np.abs(g["out_A"]).max()
    _report(f"oracle {name}", worst)


def test_reference_matches_oracle_grad_lambda():
    """T restated in longdouble against oracle.port.grad_Lambda_term_sparse on the same CSR operators."""
    from oracle import port

    f = golden_film("square_inhomogeneous")
    T, bnd = grad_lambda_ref(f, f.Lam)
    ns = SimpleNamespace(gradient_x=f.csr(f.gx), gradient_y=f.csr(f.gy))
    To = f.on_pattern(port.grad_Lambda_term_sparse(ns, f.Lam))
    check_sums(To[:, None], T[:, None], bnd[:, None], "oracle grad_Lambda_term_sparse", "slot")


def test_operator_and_diagonal_reference_against_fp64():
    """The operator reference against a plain fp64 evaluation of the same formula (dense Q, scipy CSR)."""
    rng = np.random.default_rng(4)
    n = 300
    x = jittered_points(n, 1)
    w = rng.uniform(0.5, 1.5, n) / n
    C = rng.uniform(1.0, 2.0, n)
    qd, qb = diag_ref(x, w, C)
    d = x[:, None, :] - x[None, :, :]
    r2 = (d ** 2).sum(-1)
    np.fill_diagonal(r2, np.inf)
    q = r2 ** -1.5 / (4 * np.pi)
    check_sums((C + q @ w)[:, None], qd[:, None], qb[:, None], "diag vs fp64")
    indptr, indices = random_pattern(n, 2)
    lap, T, Lam = rng.standard_normal(len(indices)), rng.standard_normal(len(indices)), rng.uniform(1, 2, n)
    src = np.sort(rng.choice(n, 100, replace=False))
    v = rng.standard_normal((n, 5))
    ref, bnd = operator_ref(x, w, np.asarray(qd, dtype=np.float64), src, v, Lam, (indptr, indices, lap), T)
    Ls = sp.csr_array((Lam[indices] * lap + T, indices, indptr), shape=(n, n))
    plain = np.asarray(qd, dtype=np.float64)[:, None] * v - (q[:, src] * w[src]) @ v[src] - Ls @ v
    check_sums(plain, ref, bnd, "operator vs fp64")


def _fault_film():
    f = golden_film("square_inhomogeneous")
    T = np.asarray(grad_lambda_ref(f, f.Lam)[0], dtype=np.float64)
    sref = SystemRef(f, f.ix, T=T)
    M = np.asarray(sref.rows(0, sref.n_pad)[0], dtype=np.float64)
    return f, T, sref, M


def _flagged(e):
    return sorted(tuple(int(v) for v in t) for t in np.argwhere(~(np.nan_to_num(e, nan=0.0) <= 1.0)))


def test_checker_names_injected_faults():
    """Fault injection: the checkers pass unmodified reference copies and flag exactly the injected place
    for a dense entry off by 64 u, two columns swapped inside one 128-column tile (in one 64-row tile),
    Lambda_r used for Lambda_c in one row, a row sum missing one 256-source tile / one 32-source GEMM
    tile, and a margin above the exact margin by more than its slack."""
    f, T, sref, M = _fault_film()
    get = lambda M_: (lambda a, b: M_[a:b])
    assert _flagged(matrix_tile_errors(get(M), sref)) == []
    check_margin(np.asarray(sref.doc_margin, dtype=np.float64), sref, "clean margin")
    # one dense entry (not on the sparse pattern) perturbed by 64 u
    r, c = 200, 300
    assert sref.pos[f.indices[f.indptr[sref.ix[r]]:f.indptr[sref.ix[r] + 1]]].tolist().count(c) == 0
    Mb = M.copy()
    Mb[r, c] *= 1 + 64 * UNIT
    assert _flagged(matrix_tile_errors(get(Mb), sref)) == [(r // TR, c // TC)]
    with pytest.raises(AssertionError, match=rf"tiles .*: \[\({r // TR}, {c // TC}\)\] "):
        check_tiles(matrix_tile_errors(get(Mb), sref), "inject")
    # two columns of one 128-column tile swapped in the rows of one 64-row tile
    Mb = M.copy()
    Mb[64:128, [260, 300]] = Mb[64:128, [300, 260]]
    assert _flagged(matrix_tile_errors(get(Mb), sref)) == [(1, 2)]
    # Lambda_r instead of Lambda_c on the sparse off-diagonal entries of one row
    r = 150
    sel = (sref.sr == r) & (sref.sc != r)
    Mb = M.copy()
    lam_r, lam_c = f.Lam[sref.si[sel]], f.Lam[sref.sj[sel]]
    Mb[r, sref.sc[sel]] += (lam_r - lam_c) * f.lap[sref.q_slot[sel]]
    want = sorted({(r // TR, int(c) // TC) for c in sref.sc[sel]})
    assert len(want) and _flagged(matrix_tile_errors(get(Mb), sref)) == want
    # a row sum missing one 256-source tile (scb_kernel_diagonal) / one 32-source tile (the GEMM)
    n = 1200
    x = jittered_points(n, 3)
    w = np.full(n, 1.0 / n)
    C = np.ones(n)
    ref, bnd = diag_ref(x, w, C)
    good = np.asarray(ref, dtype=np.float64)
    check_sums(good[:, None], ref[:, None], bnd[:, None], "clean diag")
    bad = good.copy()
    t0 = 2 * KTILE  # the third 256-source tile
    bad[700] -= float(pair_qw(x[700:701], x[t0:t0 + KTILE], w[t0:t0 + KTILE]).sum())
    with pytest.raises(AssertionError, match=r"\(target, column\) over the bound: \[\(700, 0\)\] "):
        check_sums(bad[:, None], ref[:, None], bnd[:, None], "inject")
    v = np.random.default_rng(5).standard_normal((n, 20))
    ref, bnd = operator_ref(x, w, C, None, v)
    good = np.asarray(ref, dtype=np.float64)
    check_sums(good, ref, bnd, "clean operator")
    bad = good.copy()
    t0 = GEMM_SRC  # the second 32-source tile
    bad[65, 17] += float((pair_qw(x[65:66], x[t0:t0 + GEMM_SRC], w[t0:t0 + GEMM_SRC]) @ _ld(v[t0:t0 + GEMM_SRC, 17:18]))[0, 0])
    with pytest.raises(AssertionError, match=r"\(target, column\) over the bound: \[\(65, 17\)\] "):
        check_sums(bad, ref, bnd, "inject")
    # a margin above the exact margin by more than its slack
    mg = np.asarray(sref.exact_margin, dtype=np.float64)
    mg = np.minimum(mg, np.asarray(sref.doc_margin, dtype=np.float64))
    mg[77] = float(sref.exact_margin[77] + 2 * sref.margin_slack[77])
    with pytest.raises(AssertionError, match=r"above the exact margin \+ slack at rows \[77\] "):
        check_margin(mg, sref, "inject")


def test_square_inhomogeneous_is_not_dominant():
    """The exact margins of the golden inhomogeneous system: not row-dominant with or without its T (the
    B.2 decision case), and the documented bound is never above the exact margin."""
    f = golden_film("square_inhomogeneous")
    T = np.asarray(grad_lambda_ref(f, f.Lam)[0], dtype=np.float64)
    for TT in (None, T):
        sref = SystemRef(f, f.ix, T=TT)
        assert (sref.doc_margin <= sref.exact_margin + sref.margin_slack).all()
        print(f"[system-contract] square_inhomogeneous T={'set' if TT is not None else 'NULL'}: exact min margin "
              f"{float(sref.exact_margin.min()):.4e}, documented bound min {float(sref.doc_margin.min()):.4e}")
    assert float(sref.exact_margin.min()) < 0


# ----------------------------------------------------------------------------------------
# B. GPU contract tests
# ----------------------------------------------------------------------------------------
def _d(a, dtype=None):
    import torch

    a = np.ascontiguousarray(a if dtype is None else np.asarray(a, dtype=dtype))
    return torch.as_tensor(a).cuda()


@pytest.fixture(scope="module")
def L():
    import torch

    assert torch.cuda.is_available()
    from superscreen_b200 import _lib

    return _lib.lib()


class DevFilm:
    """A Film's inputs on the device, qdw from scb_kernel_diagonal."""

    def __init__(self, f):
        import torch

        from superscreen_b200 import _lib

        self.f = f
        self.sites, self.w, self.C = _d(f.sites), _d(f.w), _d(f.C)
        self.indptr, self.indices = _d(f.indptr), _d(f.indices)
        self.lap, self.gx, self.gy = _d(f.lap), _d(f.gx), _d(f.gy)
        self.qdw = torch.empty(f.n, dtype=torch.float64, device="cuda")
        _lib.check(_lib.lib().scb_kernel_diagonal(f.n, _lib.ptr(self.sites), _lib.ptr(self.w), _lib.ptr(self.C),
                                                  _lib.ptr(self.qdw), _lib.stream_ptr()))

    def grad_lambda(self, Lam):
        import torch

        from superscreen_b200 import _lib

        T = torch.full((len(self.f.indices),), np.nan, dtype=torch.float64, device="cuda")
        _lib.check(_lib.lib().scb_grad_lambda_term(self.f.n, _lib.ptr(self.indptr), _lib.ptr(self.indices),
                                                   _lib.ptr(self.gx), _lib.ptr(self.gy), _lib.ptr(_d(Lam)),
                                                   _lib.ptr(T), _lib.stream_ptr()))
        return T

    def assemble(self, ix, Lam, T=None, sym=None, M=None, margin=True):
        """(rc, M, margin) of scb_system_assemble; the workspace starts as NaN."""
        import torch

        from superscreen_b200 import _lib

        n_int = len(ix)
        n_pad = _pad_of(n_int)
        if M is None:
            M = torch.full((n_pad, n_pad), np.nan, dtype=torch.float64, device="cuda")
        mg = torch.full((n_int,), np.nan, dtype=torch.float64, device="cuda") if margin else None
        self._keep = (ix_d := _d(ix, np.int64), Lam_d := _d(Lam), sym_d := None if sym is None else _d(sym))
        pos = torch.empty(self.f.n, dtype=torch.int32, device="cuda")
        rc = _lib.lib().scb_system_assemble(
            self.f.n, _lib.ptr(self.sites), _lib.ptr(self.w), _lib.ptr(self.qdw), _lib.ptr(self.C), _lib.ptr(Lam_d),
            _lib.ptr(self.indptr), _lib.ptr(self.indices), _lib.ptr(self.lap), _lib.ptr(T), n_int, _lib.ptr(ix_d),
            _lib.ptr(pos), n_pad, _lib.ptr(M), _lib.ptr(mg), _lib.ptr(sym_d), _lib.stream_ptr())
        return rc, M, mg


@functools.lru_cache(maxsize=4)
def square_film(n_vertices, seed):
    from superscreen_b200.synthetic import square_mesh

    sites, elements = square_mesh(10.0, n_vertices, seed=seed)
    f = Film(sites, elements, 0.1)
    f.name = f"square{n_vertices}"
    from oracle import port

    f.interior = np.setdiff1d(np.arange(f.n), port.find_boundary_indices(f.elements))
    return f


def _step_lambda(f):
    """A Lambda with a sharp step across the film (inhomogeneous: general system with T)."""
    x = f.sites[:, 0]
    return np.where(x < np.median(x), 0.05, 2.0) + 0.01 * np.cos(f.sites[:, 1])


def _run_assembly(df: DevFilm, ix, mode, what, Lam=None, row_tiles=None):
    """Assembles (ix, mode) on the device and checks every entry (or the given 64-row tiles) and the margin.
    mode: 'gen' (T NULL), 'gen+T' (T from scb_grad_lambda_term), 'sym' (sym_scale = sqrt(w))."""
    import torch

    f = df.f
    Lam = f.Lam if Lam is None else Lam
    T = Td = sym = None
    if mode == "gen+T":
        Td = df.grad_lambda(Lam)
        T = Td.cpu().numpy()
    if mode == "sym":
        sym = np.sqrt(f.w)
    rc, M, mg = df.assemble(ix, Lam, T=Td, sym=sym)
    assert rc == 0
    torch.cuda.synchronize()
    ff = SimpleNamespace(**{**f.__dict__, "Lam": Lam})
    sref = SystemRef(ff, ix, T=T, sym=sym, row_tiles=row_tiles)
    if row_tiles is None:
        Mh = M.cpu().numpy()
        get = lambda a, b: Mh[a:b]
    else:
        get = lambda a, b: M[a:b].cpu().numpy()
    e = matrix_tile_errors(get, sref, row_tiles)
    worst = check_tiles(e, what)
    extra = ""
    if sym is not None and row_tiles is None:  # S = S^T within the entry bounds of both sides
        ref, bnd = sref.rows(0, sref.n_pad)
        d = np.abs(Mh - Mh.T)
        with np.errstate(divide="ignore", invalid="ignore"):
            qs = np.where(d == 0, 0.0, d / (bnd + bnd.T))
        qs[~np.isfinite(qs)] = np.inf
        worst_s = check_tiles(qs.reshape(sref.n_pad // TR, TR, sref.n_pad // TC, TC).max(axis=(1, 3)), what,
                              "S - S^T")
        extra = f"  |S-S^T| {worst_s:.3e}"
    wm = check_margin(mg.cpu().numpy(), sref, what)
    _report(what, worst, f"  margin {wm:.3e} slack{extra}")
    return sref, mg.cpu().numpy()


N_INTS = (1, 63, 64, 65, 127, 128, 129, 255, 256, 257)
MODES = ("gen", "gen+T", "sym")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["ring", "square_inhomogeneous", "transport"])
def test_assemble_goldens(L, name):
    """The golden systems (holes: ix not contiguous) element by element, every mode the API allows
    (square_inhomogeneous: its Lambda is not constant, so general only, with and without T)."""
    f = golden_film(name)
    df = DevFilm(f)
    modes = ("gen", "gen+T") if name == "square_inhomogeneous" else MODES
    for mode in modes:
        _run_assembly(df, f.ix, mode, f"{name} {mode} n_int={len(f.ix)}")


@pytest.mark.gpu
def test_assemble_tile_edges_1500(L):
    """n_int at the 64-row / 128-column tile edges, the full interior, a shuffled ix and ix = every vertex
    (margin exact), on a ~1.5k square mesh, rotating through the modes (each n_int in one mode, the full
    interior and every-vertex sets in all)."""
    f = square_film(1500, 1)
    df = DevFilm(f)
    rng = np.random.default_rng(0)
    step = _step_lambda(f)
    for k, n_int in enumerate(N_INTS):
        ix = np.sort(rng.choice(f.interior, n_int, replace=False))
        mode = MODES[k % 3]
        _run_assembly(df, ix, mode, f"sq1500 {mode} n_int={n_int}", Lam=step if mode == "gen+T" else None)
    for mode in MODES:
        _run_assembly(df, f.interior, mode, f"sq1500 {mode} interior n_int={len(f.interior)}",
                      Lam=step if mode == "gen+T" else None)
        _run_assembly(df, np.arange(f.n), mode, f"sq1500 {mode} all vertices n_int={f.n}",
                      Lam=step if mode == "gen+T" else None)
    shuffled = rng.permutation(f.interior)[:700]
    _run_assembly(df, shuffled, "gen+T", "sq1500 gen+T shuffled n_int=700", Lam=step)
    _run_assembly(df, shuffled, "sym", "sq1500 sym shuffled n_int=700")
    # inhomogeneous Lambda without T is allowed too (general)
    _run_assembly(df, f.interior, "gen", "sq1500 gen step-Lambda T=NULL", Lam=step)


@pytest.mark.gpu
def test_assemble_6400(L):
    """A ~6.4k-vertex square (the C2 mesh at that size), full interior, general and symmetrised."""
    f = square_film(6400, 3)
    df = DevFilm(f)
    for mode in ("gen", "sym"):
        _run_assembly(df, f.interior, mode, f"sq6400 {mode} interior n_int={len(f.interior)}")


@pytest.mark.gpu
def test_assemble_rejects_sym_with_T(L):
    f = golden_film("ring")
    df = DevFilm(f)
    T = df.grad_lambda(f.Lam)
    rc, M, _ = df.assemble(f.ix, f.Lam, T=T, sym=np.sqrt(f.w))
    assert rc == -1  # SCB_ERR_INVALID
    from superscreen_b200 import _lib

    assert b"homogeneous" in _lib.lib().scb_last_error()
    assert bool(M.isnan().all())


@pytest.mark.gpu
def test_assemble_past_32bit_index(L):
    """n_pad = 46464, n_pad^2 > 2^31: every tile of the first and last 64-row block rows and of a few random
    ones, general mode with margins (17.3 GB workspace)."""
    import torch

    n_pad = 46464
    need = 8 * n_pad * n_pad
    free = torch.cuda.mem_get_info()[0]
    if free < 2 * need:
        pytest.skip(f"needs {2 * need / 1e9:.1f} GB free on the device for a {need / 1e9:.1f} GB workspace, "
                    f"{free / 1e9:.1f} GB free")
    f = square_film(47600, 7)
    n_int = n_pad - 127
    assert len(f.interior) >= n_int, len(f.interior)
    ix = f.interior[len(f.interior) - n_int:]
    df = DevFilm(f)
    rng = np.random.default_rng(1)
    tiles = sorted({0, n_pad // TR - 1, (n_int - 1) // TR, *rng.choice(n_pad // TR, 3, replace=False).tolist()})
    _run_assembly(df, ix, "gen", f"sq47600 gen n_int={n_int} rows {tiles}", row_tiles=tiles)
    torch.cuda.empty_cache()


def _perturbed_film():
    """The vertex-perturbed (non-Delaunay) mesh of test_gpu_parity.test_non_delaunay_mesh_uses_refinement."""
    from oracle import port
    from superscreen_b200.synthetic import square_mesh

    sites, elements = square_mesh(10.0, 2500, seed=21)
    rng = np.random.default_rng(5)
    interior = np.setdiff1d(np.arange(len(sites)), port.find_boundary_indices(elements))
    h = np.sqrt(100.0 / len(sites))
    moved = sites.copy()
    moved[interior] += 0.42 * h * (rng.random((len(interior), 2)) * 2 - 1)

    def cross(p):
        return (p[:, 1, 0] - p[:, 0, 0]) * (p[:, 2, 1] - p[:, 0, 1]) - (p[:, 1, 1] - p[:, 0, 1]) * (p[:, 2, 0] - p[:, 0, 0])

    bad = np.unique(elements[cross(moved[elements]) <= 0.05 * h * h])
    moved[bad] = sites[bad]
    assert (cross(moved[elements]) > 0).all()
    f = Film(moved, elements, 2.0)
    f.interior = interior
    return f


@pytest.mark.gpu
def test_pivot_decision_on_non_dominant_systems(L):
    """The decision margin.min() <= 0 (scb_getrf_piv / iterative refinement) against the exact margin on two
    systems that are not provably dominant: the device never reports dominance the exact margin lacks."""
    cases = []
    f = golden_film("square_inhomogeneous")
    cases.append((DevFilm(f), f.ix, "gen+T", "square_inhomogeneous gen+T"))
    pf = _perturbed_film()
    cases.append((DevFilm(pf), pf.interior, "gen", "perturbed non-Delaunay gen"))
    for df, ix, mode, what in cases:
        sref, mg = _run_assembly(df, ix, mode, what)
        ex = float(sref.exact_margin.min())
        print(f"[system-contract] {what}: device min margin {mg.min():.4e}, exact {ex:.4e}, "
              f"documented bound {float(sref.doc_margin.min()):.4e}")
        assert not (mg.min() > 0 and ex <= 0), f"{what}: device reports dominance the exact margin lacks"
        if ex <= 0:
            assert mg.min() <= 0


# ---- scb_kernel_diagonal ------------------------------------------------------------------
DIAG_NS = (1, 2, 255, 256, 257, 511, 512, 513, 4097, 20000)


def _diag_case(L, n, scale, seed):
    import torch

    from superscreen_b200 import _lib

    rng = np.random.default_rng(seed)
    x = jittered_points(n, seed, scale)
    w = rng.uniform(0.5, 1.5, n) * scale ** 2 / n
    C = rng.uniform(0.5, 3.0, n) / scale
    xd, wd, Cd = _d(x), _d(w), _d(C)
    outs = []
    for _ in range(2):
        q = torch.full((n,), np.nan, dtype=torch.float64, device="cuda")
        _lib.check(L.scb_kernel_diagonal(n, _lib.ptr(xd), _lib.ptr(wd), _lib.ptr(Cd), _lib.ptr(q), _lib.stream_ptr()))
        outs.append(q.cpu().numpy())
    assert np.array_equal(outs[0].view(np.int64), outs[1].view(np.int64)), f"n={n}: repeated call differs"
    t = np.arange(n)
    if n > 5000:  # every 256-target and 512-target CTA edge near the ends, and a random sample
        t = np.unique(np.concatenate([t[:1100], t[-1100:], rng.choice(n, 1000, replace=False)]))
    ref, bnd = diag_ref(x, w, C, t)
    return check_sums(outs[0][t, None], ref[:, None], bnd[:, None], f"kernel_diagonal n={n} scale={scale}")


@pytest.mark.gpu
@pytest.mark.parametrize("n", DIAG_NS)
def test_kernel_diagonal(L, n):
    """Unsplit below 512 sources, split and reduced above."""
    _report(f"kernel_diagonal n={n}", _diag_case(L, n, 1.0, n))


@pytest.mark.gpu
def test_kernel_diagonal_si_metres(L):
    """Coordinates in SI metres (1e-6 of the micron scale): no under- or overflow in inv_r3."""
    _report("kernel_diagonal n=4097 scale=1e-6", _diag_case(L, 4097, 1e-6, 11))


# ---- scb_apply_operator --------------------------------------------------------------------
APPLY_NRHS = (1, 2, 3, 4, 7, 8, 9, 15, 16, 17, 31, 32, 33, 48, 63, 64, 65, 80, 128, 130)
# (targets n, sources): an int = that many sources through src_idx, "all" = every vertex through src_idx
# (shuffled), None = src_idx NULL.  Below 512 sources the N-body sum runs unsplit, from 512 on it splits.
UNSPLIT = [(63, 0), (64, 1), (65, 31), (63, 32), (64, 33), (65, "all"), (63, None), (511, 255), (512, 256),
           (513, 257), (64, None), (511, "all"), (511, None)]
SPLIT = [(512, None), (513, "all"), (513, None), (512, "all")]
SPLIT_6K = {1: (6000, None), 3: (6000, "all"), 9: (6000, None), 17: (6000, "all")}  # (the reference costs n^2 nrhs)
FLAGS = [  # (Lambda, T, accumulate)
    (False, False, 0), (True, False, 1), (True, True, 0), (False, False, 1), (True, True, 1), (True, False, 0)]


def _apply_cases():
    cases = []
    for k, nrhs in enumerate(APPLY_NRHS):
        cases.append((*UNSPLIT[k % len(UNSPLIT)], nrhs, *FLAGS[k % len(FLAGS)]))
        cases.append((*SPLIT_6K.get(nrhs, SPLIT[k % len(SPLIT)]), nrhs, *FLAGS[(k + 3) % len(FLAGS)]))
    # the GEMM's 64-target CTA and 32-source tile edges with the GEMM passes 16 / 32 / 64
    for nrhs, (n, s) in zip((16, 32, 64, 65, 80), [(63, 31), (64, 32), (65, 33), (63, 33), (65, 32)]):
        cases.append((n, s, nrhs, True, True, 1))
    return cases


def _n_src(n, s):
    return n if s in ("all", None) else s


def test_apply_case_list_covers_every_edge():
    """Every column count with both the unsplit and the split N-body path; every target and source edge;
    the GEMM passes at the 64-target and 32-source edges; every flag combination."""
    cases = _apply_cases()
    for nrhs in APPLY_NRHS:
        kinds = {_n_src(n, s) >= 512 for n, s, r, *_ in cases if r == nrhs}
        assert kinds == {False, True}, nrhs
    assert {n for n, *_ in cases} == {63, 64, 65, 511, 512, 513, 6000}
    assert {s for _, s, *_ in cases} >= {0, 1, 31, 32, 33, 255, 256, 257, "all", None}
    gemm = {(n, s) for n, s, r, *_ in cases if r >= 16}
    assert {n for n, _ in gemm} >= {63, 64, 65} and {s for _, s in gemm} >= {31, 32, 33, None, "all"}
    assert {tuple(c[3:]) for c in cases} == set(FLAGS)


@functools.lru_cache(maxsize=None)
def _apply_inputs(n):
    rng = np.random.default_rng(n)
    x = jittered_points(n, n + 1, 10.0)
    w = rng.uniform(0.5, 1.5, n) * 100.0 / n
    qdw = rng.uniform(1.0, 3.0, n) * np.sqrt(n)
    indptr, indices = random_pattern(n, n + 2)
    lap = rng.standard_normal(len(indices)) * n / 100.0
    T = rng.standard_normal(len(indices))
    Lam = rng.uniform(0.05, 2.0, n)
    return x, w, qdw, indptr, indices, lap, T, Lam


def _apply_case(L, n, s, nrhs, use_lam, use_T, acc):
    import torch

    from superscreen_b200 import _lib

    x, w, qdw, indptr, indices, lap, T, Lam = _apply_inputs(n)
    rng = np.random.default_rng([n, nrhs, 0 if s is None else (n if s == "all" else s) + 1])
    if s is None:
        src, n_src, src_d = None, 0, None
    else:
        src = rng.permutation(n) if s == "all" else np.sort(rng.choice(n, s, replace=False))
        n_src = len(src)
        # n_src = 0 with a real (non-NULL) buffer: NULL would mean "every vertex"
        src_d = _d(src if len(src) else np.array([n // 2]), np.int64)
    v = rng.standard_normal((n, nrhs))
    pre = rng.standard_normal((n, nrhs)) if acc else None
    args = [_d(a) for a in (x, w, qdw)]
    lam_d = _d(Lam) if use_lam else None
    T_d = _d(T) if use_T else None
    ip, ii, lp, vd = _d(indptr), _d(indices), _d(lap), _d(v)
    outs = []
    for _ in range(2):
        out = _d(pre) if acc else torch.full((n, nrhs), np.nan, dtype=torch.float64, device="cuda")
        _lib.check(L.scb_apply_operator(n, *(_lib.ptr(a) for a in args), _lib.ptr(lam_d), _lib.ptr(ip), _lib.ptr(ii),
                                        _lib.ptr(lp), _lib.ptr(T_d), n_src, _lib.ptr(src_d), nrhs, _lib.ptr(vd),
                                        _lib.ptr(out), acc, _lib.stream_ptr()))
        outs.append(out.cpu().numpy())
    what = (f"apply n={n} src={s} nrhs={nrhs} Lambda={'set' if use_lam else 'NULL'} "
            f"T={'set' if use_T and use_lam else 'NULL'} acc={acc}")
    assert np.array_equal(outs[0].view(np.int64), outs[1].view(np.int64)), f"{what}: repeated call differs"
    ref, bnd = operator_ref(x, w, qdw, src, v, Lam if use_lam else None, (indptr, indices, lap),
                            T if (use_T and use_lam) else None, pre)
    return what, check_sums(outs[0], ref, bnd, what)


@pytest.mark.gpu
@pytest.mark.parametrize("case", _apply_cases(), ids=lambda c: f"n{c[0]}-s{c[1]}-r{c[2]}-f{int(c[3])}{int(c[4])}{c[5]}")
def test_apply_operator(L, case):
    """Both engines (GEMM passes of 64 / 32 / 16 columns, CUDA-core passes of 8 / 4 / 2 / 1) at the CTA
    and tile edges, split and unsplit, src_idx / NULL / empty, accumulate into random values / overwrite
    NaN, the sparse part with Lambda and T NULL or set; bit-identical on repetition."""
    what, worst = _apply_case(L, *case)
    _report(what, worst)


# ---- scb_grad_lambda_term ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("which", ["golden", "step"])
def test_grad_lambda_term(L, which):
    """T on the operator pattern against the longdouble restatement and oracle.port.grad_Lambda_term_sparse
    (absent entries 0): the golden inhomogeneous Lambda, and a sharp step on a 1.5k square."""
    from oracle import port

    f = golden_film("square_inhomogeneous") if which == "golden" else square_film(1500, 1)
    Lam = f.Lam if which == "golden" else _step_lambda(f)
    df = DevFilm(f)
    T1, T2 = df.grad_lambda(Lam).cpu().numpy(), df.grad_lambda(Lam).cpu().numpy()
    assert np.array_equal(T1.view(np.int64), T2.view(np.int64))
    ref, bnd = grad_lambda_ref(f, Lam)
    worst = check_sums(T1[:, None], ref[:, None], bnd[:, None], f"grad_lambda {which}", "slot")
    To = f.on_pattern(port.grad_Lambda_term_sparse(SimpleNamespace(gradient_x=f.csr(f.gx),
                                                                   gradient_y=f.csr(f.gy)), Lam))
    check_sums(To[:, None], ref[:, None], bnd[:, None], f"oracle grad_lambda {which}", "slot")
    _report(f"grad_lambda {which} nnz={len(T1)}", worst)


# ---- the remaining N-body kinds ------------------------------------------------------------
BS_SIZES = [(1, 1), (511, 255), (512, 256), (513, 257), (1000, 3000), (1, 3000), (1000, 1), (512, 257),
            (300, 100000)]
F2F_NSETS = (1, 2, 3, 7, 8, 9, 17, 130)


def _bs_run(L, kind, tgt, src, area, J, dz, pf, nsets, out_shape):
    import torch

    from superscreen_b200 import _lib

    outs = []
    t_d, s_d, a_d, J_d = _d(tgt), _d(src), _d(area), _d(J)
    for _ in range(2):
        out = torch.full(out_shape, np.nan, dtype=torch.float64, device="cuda")
        _lib.check(L.scb_biot_savart(kind, len(tgt), _lib.ptr(t_d), len(src), _lib.ptr(s_d), _lib.ptr(a_d),
                                     _lib.ptr(J_d), dz, pf, nsets, _lib.ptr(out), _lib.stream_ptr()))
        outs.append(out.cpu().numpy())
    assert np.array_equal(outs[0].view(np.int64), outs[1].view(np.int64)), "repeated call differs"
    return outs[0]


def _pts3(rng, m, z, scale=3.0):
    p = np.empty((m, 3))
    p[:, :2] = rng.uniform(-scale, scale, (m, 2))
    p[:, 2] = z
    return p


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [BS_VECTOR, BS_VECPOT], ids=["vector", "vector_potential"])
@pytest.mark.parametrize("size", BS_SIZES, ids=lambda s: f"m{s[0]}-n{s[1]}")
def test_biot_savart_vector_kinds(L, kind, size):
    """SCB_BS_VECTOR (out [m, 3], 4 split accumulators) and SCB_BS_VECTOR_POTENTIAL (out [m, 2], 2)."""
    m, n = size
    rng = np.random.default_rng(m * 7 + n + kind)
    tgt, src = _pts3(rng, m, 0.7), _pts3(rng, n, 0.0)
    src[:, 2] = rng.uniform(-0.2, 0.2, n)
    area, J = rng.uniform(0.5, 1.5, n) / max(n, 1), rng.standard_normal((n, 2))
    pf = 1e-7
    ncomp = 3 if kind == BS_VECTOR else 2
    got = _bs_run(L, kind, tgt, src, area, J, 0.0, pf, 1, (m, ncomp))
    ref, bnd = bs_ref(kind, tgt, src, area, J, 0.0, pf)
    what = f"{'vector' if kind == BS_VECTOR else 'vector_potential'} m={m} n={n}"
    _report(what, check_sums(got, ref, bnd, what, "component"))


def _f2f_cases():
    sizes = [(513, 257), (511, 255), (1000, 3000), (1, 1), (512, 256), (300, 100000), (1000, 1), (513, 257)]
    return [(ns, *sizes[k]) for k, ns in enumerate(F2F_NSETS)] + [(9, 1, 3000), (8, 513, 257)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", _f2f_cases(), ids=lambda c: f"sets{c[0]}-m{c[1]}-n{c[2]}")
def test_biot_savart_film_to_film_sets(L, case):
    """SCB_BS_FILM_TO_FILM with 1 .. 130 current-density sets (passes of 8 / 4 / 2 / 1 sharing r^-3), dz != 0."""
    nsets, m, n = case
    rng = np.random.default_rng(nsets * 100003 + m + n)
    tgt, src = rng.uniform(-3, 3, (m, 2)), rng.uniform(-3, 3, (n, 2))
    area, J = rng.uniform(0.5, 1.5, n) / n, rng.standard_normal((nsets, n, 2))
    dz, pf = 0.35, 1.0 / (4 * np.pi)
    got = _bs_run(L, BS_FILM_TO_FILM, tgt, src, area, J, dz, pf, nsets, (nsets, m))
    ref, bnd = bs_ref(BS_FILM_TO_FILM, tgt, src, area, J, dz, pf)
    what = f"film_to_film nsets={nsets} m={m} n={n}"
    _report(what, check_sums(got.T, ref.T, bnd.T, what, "set"))
