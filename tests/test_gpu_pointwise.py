"""Per-atom, per-component force and energy bounds for every evaluation path (-m gpu), with CPU self-tests of the checker.

The other GPU parity tests check forces in max-norm over a batch, |F - F_ref|.max() <= tol * |F_ref|.max(). Their recipes
put a few atoms outside the grid, where the restraint force sets max|F|, so the interpolated forces of most atoms are
checked against a number they never come close to: a wrong corner that spoils a few small-force atoms passes there. Here
every atom and every component is held to a bound built from the terms the kernels sum for THAT atom:

  |f - f_ref| <= tol_f * max(|f_ref|, R) + tol_d * D + tol_v * V + fixed_adds * 2^-32

  D  (differenced) sum over grids g of |s_g| * c_g * sum_k |dw_k/da| * |v_k - v_k0| / h_a over the points k the method
     reads (trilinear: the 2x2x2 cell; B-spline: the 4x4x4 block with clamped indices; tricubic: the 32 flat-indexed points
     of tricubic_interpolate, wrapped reads in the last y/z cell and zeros past the array included), k0 the stencil's first
     point. It is the size of what an FP32 gradient formed from corner differences can lose. c = 1, or |n| * max|v|^(n-1)
     on an inv-power grid.
  V  (value-sized) the same sum with |v_k|: FP64 arithmetic on values of size |V| (DOUBLE keeps the reference's vp - vm)
     and, on grids that are not FP32-representable, storage rounding.
  R  the restraint forces' magnitude |k * dev| summed over the grids an atom is outside of.

Energies are held per replica (and per atom where per-atom energies are requested) to tol * sum |s| * sum_k |w_k| |v_k|
plus the restraint energies. Grids are FP32-representable unless a case says otherwise, so on the MIXED value paths
(all FP64) the honest error is FP64 rounding.

Each bound constant below carries the worst ratio err / bound measured on a B200 across this file's cases; none allows
more than 8x headroom over it. Every GPU case asserts gfb_kernel_eval_path.
"""
import itertools
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import test_gpu_coverage as cov  # noqa: E402

U = 2.0 ** -24                      # FP32 unit roundoff
FIXED_QUANTUM = 2.0 ** -32          # OpenMM's fixed-point force unit; truncation loses less than one per add
CELLS, ROWS, PAIRS, BSPLINE, POINTS, HERMITE, BSPLINE_POINTS = 1, 2, 3, 4, 5, 6, 7
METHOD = cov.METHOD
N_THREADS = cov.N_THREADS

# ---------------------------------------------------------------------------------------------------------------------
# Bounds. Measured worst ratio err / bound over this file's GPU cases on a B200 in the comment of each.
# ---------------------------------------------------------------------------------------------------------------------
# MIXED, one grid's gradient in FP32 from corner differences (one-grid lines kernel, general kernel, resident evaluator):
# trilinear<float> with FP32 fractions, scaling cast to float, the FP32 product with 1/spacing. Worst 0.68 (one-grid
# lines kernel, FIXED_ADD); the general kernel 0.33, the resident evaluator 0.34.
TOL_TRILINEAR_F32 = dict(tol_f=2 * U, tol_d=8 * U, tol_v=0.0)
# MIXED B-spline (records and points): FP32 sums of weight * (point - first point) over 64 points. Worst 0.29.
TOL_BSPLINE_F32 = dict(tol_f=2 * U, tol_d=8 * U, tol_v=0.0)
# MIXED 2-4 grid lines kernel: scaled corners summed in FP64, value and gradient in FP64, the force rounded to FP32 once.
# Worst 0.50 with FP64 stores (the FP32 rounding); 0.98 for FIXED_ADD, where small forces sit at the 2^-32 quantum.
TOL_LINES_MULTI = dict(tol_f=2 * U, tol_d=0.0, tol_v=1e-14)
# FP64 arithmetic: every DOUBLE trilinear and B-spline path. Worst 0.32 (the general kernel, grids of mixed geometry).
TOL_F64 = dict(tol_f=2e-16, tol_d=2e-15, tol_v=2e-15)
# Tricubic (MIXED and DOUBLE: FP64 arithmetic). Its weights are not rounded in proportion to their size: near a fraction
# of 1 the derivative weight 6t^2 - 6t is a small difference of terms of size 6, and the staged arithmetic (x edges, then
# y and z differences of partly interpolated values) differences intermediates of size |V|. The kernel forms the basis as
# 6 * (t * t) where the reference has (6 * t) * t, and 0.5 * (v1 - v0) where it has (v1 - v0) / (2s) * s; the two
# roundings differ by up to 7.1e-14 of D + V (cell (11, 3, 14), fractions (0.010, 0.379, 0.013)). Worst 0.37.
TOL_TRICUBIC = dict(tol_f=1e-15, tol_d=2e-13, tol_v=2e-13)
# Energies of either precision on FP32-representable grids: FP64 rounding only. Worst 0.16 (per-atom energies of the
# 3-grid lines kernel); per replica 0.011.
TOL_E = 1e-13
# Energies on grids that are not FP32-representable (MIXED): the storage rounding 2^-24 |v| per point. Worst 0.13 (the
# C5 sample, whose forces reach 0.68 of TOL_LINES_MULTI plus 2^-24 V).
TOL_E_STORAGE = 6e-8


def _tol(precision, method, n_grids=1, path=None):
    if method == 2:
        return dict(TOL_TRICUBIC)
    if precision == 1:
        return dict(TOL_F64)
    if method == 1:
        return dict(TOL_BSPLINE_F32)
    if path == 1 and n_grids > 1:
        return dict(TOL_LINES_MULTI)
    return dict(TOL_TRILINEAR_F32)


def _f32_output(tol):
    """Forces returned as float: one more rounding of |F|."""
    return dict(tol, tol_f=tol["tol_f"] + U)


# ---------------------------------------------------------------------------------------------------------------------
# Scales (numpy only)
# ---------------------------------------------------------------------------------------------------------------------
def _geom(case, g):
    if "geoms" in case:
        return case["geoms"][g]
    return case["counts"], case["spacing"], case["origin"]


def _classify(pos, counts, sp, og):
    """The kernels' cell: inside by <= on both faces, ix = min(floor(q), n-2), fraction q - ix (1 on the upper face).
    Also the neighbouring cell on each axis where the fraction is within 1e-12 of 0 or 1."""
    n, sp, og = np.array(counts), np.array(sp, dtype=np.float64), np.array(og, dtype=np.float64)
    rel = pos - og
    inside = ((rel >= 0.0) & (rel <= sp * (n - 1))).all(axis=-1)
    q = rel / sp
    idx = np.clip(np.floor(q), 0, n - 2).astype(np.int64)
    f = np.clip(q - idx, 0.0, 1.0)
    idx[~inside] = 0
    f[~inside] = 0.0
    alt_idx, alt_f = idx.copy(), f.copy()
    lo = (f < 1e-12) & (idx > 0) & inside[:, None]
    hi = (f > 1.0 - 1e-12) & (idx < n - 2) & inside[:, None]
    alt_idx[lo] -= 1
    alt_f[lo] = np.minimum(f[lo] + 1.0, 1.0)
    alt_idx[hi] += 1
    alt_f[hi] = np.maximum(f[hi] - 1.0, 0.0)
    return inside, idx, f, alt_idx, alt_f


def _bspline_basis(t):
    u = 1.0 - t
    b = np.stack([u * u * u / 6.0, (3 * t ** 3 - 6 * t ** 2 + 4) / 6.0, (-3 * t ** 3 + 3 * t ** 2 + 3 * t + 1) / 6.0, t ** 3 / 6.0], -1)
    d = np.stack([-u * u / 2.0, (3 * t * t - 4 * t) / 2.0, (-3 * t * t + 2 * t + 1) / 2.0, t * t / 2.0], -1)
    return b, d


def _hermite_basis(t):
    """order h00, h01, h10, h11 (gf_kernels.cuh hermite_basis)"""
    u = 1.0 - t
    h = np.stack([(1 + 2 * t) * u * u, t * t * (3 - 2 * t), t * u * u, t * t * (t - 1)], -1)
    d0 = 6 * t * t - 6 * t
    d = np.stack([d0, -d0, 3 * t * t - 4 * t + 1, 3 * t * t - 2 * t], -1)
    return h, d


def _tricubic_eval(V, xin, yin, zin, hx, dhx, hy, dhy, hz, dhz):
    """gf_kernels.cuh tricubic_eval over V[..., i, r, k] (the point at offsets (i-1, r-1, k-1) from the cell)."""
    xin, yin, zin = (x.astype(np.float64) for x in (xin, yin, zin))
    vv, dv = {}, {}
    for j in range(2):
        for k in range(2):
            f0, f1 = V[..., 1, 1 + j, 1 + k], V[..., 2, 1 + j, 1 + k]
            d0 = xin * 0.5 * (f1 - V[..., 0, 1 + j, 1 + k])
            d1 = xin * 0.5 * (V[..., 3, 1 + j, 1 + k] - f0)
            vv[j, k] = hx[:, 0] * f0 + hx[:, 1] * f1 + hx[:, 2] * d0 + hx[:, 3] * d1
            dv[j, k] = dhx[:, 0] * f0 + dhx[:, 1] * f1 + dhx[:, 2] * d0 + dhx[:, 3] * d1
    vk, dxk = {}, {}
    dvdy = 0.0
    for k in range(2):
        rm = hx[:, 0] * V[..., 1, 0, 1 + k] + hx[:, 1] * V[..., 2, 0, 1 + k]
        rp = hx[:, 0] * V[..., 1, 3, 1 + k] + hx[:, 1] * V[..., 2, 3, 1 + k]
        dy0, dy1 = yin * (vv[1, k] - rm), yin * (rp - vv[0, k])
        vk[k] = hy[:, 0] * vv[0, k] + hy[:, 1] * vv[1, k] + hy[:, 2] * dy0 + hy[:, 3] * dy1
        dxk[k] = hy[:, 0] * dv[0, k] + hy[:, 1] * dv[1, k]
        if k == 0:
            dvdy = dhy[:, 0] * vv[0, 0] + dhy[:, 1] * vv[1, 0] + dhy[:, 2] * dy0 + dhy[:, 3] * dy1
    zm = hy[:, 0] * (hx[:, 0] * V[..., 1, 1, 0] + hx[:, 1] * V[..., 2, 1, 0]) + hy[:, 1] * (hx[:, 0] * V[..., 1, 2, 0] + hx[:, 1] * V[..., 2, 2, 0])
    zp = hy[:, 0] * (hx[:, 0] * V[..., 1, 1, 3] + hx[:, 1] * V[..., 2, 1, 3]) + hy[:, 1] * (hx[:, 0] * V[..., 1, 2, 3] + hx[:, 1] * V[..., 2, 2, 3])
    dz0, dz1 = zin * (vk[1] - zm), zin * (zp - vk[0])
    val = hz[:, 0] * vk[0] + hz[:, 1] * vk[1] + hz[:, 2] * dz0 + hz[:, 3] * dz1
    gx = hz[:, 0] * dxk[0] + hz[:, 1] * dxk[1]
    gz = dhz[:, 0] * vk[0] + dhz[:, 1] * vk[1] + dhz[:, 2] * dz0 + dhz[:, 3] * dz1
    return val, gx, dvdy, gz


def _stencil(method, vals, counts, idx, f):
    """(v [N, K], w [N, K], dw [N, K, 3] per unit fraction, k0) of the points method `method` reads for cells idx [N, 3]
    at fractions f [N, 3]. Weights of a point read twice (clamped indices) are kept apart, as the kernels sum them."""
    n = np.array(counts)
    if method == 0:
        corners = list(itertools.product((0, 1), repeat=3))             # v000, v001, v010, ... (z fastest)
        v = np.stack([vals[idx[:, 0] + a, idx[:, 1] + b, idx[:, 2] + c] for a, b, c in corners], 1)
        wa = [np.stack([1.0 - f[:, a], f[:, a]], -1) for a in range(3)]
        da = np.array([-1.0, 1.0])
        w = np.stack([wa[0][:, a] * wa[1][:, b] * wa[2][:, c] for a, b, c in corners], 1)
        dw = np.stack([np.stack([da[a] * wa[1][:, b] * wa[2][:, c], wa[0][:, a] * da[b] * wa[2][:, c],
                                 wa[0][:, a] * wa[1][:, b] * da[c]], -1) for a, b, c in corners], 1)
        return v, w, dw, 0
    if method == 1:
        bd = [_bspline_basis(f[:, a]) for a in range(3)]
        pts = list(itertools.product(range(4), repeat=3))
        ix = [np.clip(idx[:, a, None] - 1 + np.arange(4), 0, n[a] - 1) for a in range(3)]
        v = np.stack([vals[ix[0][:, i], ix[1][:, j], ix[2][:, k]] for i, j, k in pts], 1)
        (bx, dx), (by, dy), (bz, dz) = bd
        w = np.stack([bx[:, i] * by[:, j] * bz[:, k] for i, j, k in pts], 1)
        dw = np.stack([np.stack([dx[:, i] * by[:, j] * bz[:, k], bx[:, i] * dy[:, j] * bz[:, k], bx[:, i] * by[:, j] * dz[:, k]], -1)
                       for i, j, k in pts], 1)
        return v, w, dw, 0
    # method 2: weights by linearity (tricubic_eval of each unit point), values by flat index as the reference reads them
    nz, nyz, total = n[2], n[1] * n[2], int(np.prod(n))
    flat = vals.ravel()
    im = idx[:, 0] * nyz + idx[:, 1] * nz + idx[:, 2]
    pts = list(itertools.product(range(4), repeat=3))
    fi = np.stack([im + (i - 1) * nyz + (r - 1) * nz + (k - 1) for i, r, k in pts], 1)
    v = np.where((fi >= 0) & (fi < total), flat[np.clip(fi, 0, total - 1)], 0.0)
    hx, dhx = _hermite_basis(f[:, 0])
    hy, dhy = _hermite_basis(f[:, 1])
    hz, dhz = _hermite_basis(f[:, 2])
    xin, yin, zin = ((idx[:, a] > 0) & (idx[:, a] < n[a] - 1) for a in range(3))
    unit = np.eye(64).reshape(64, 1, 4, 4, 4)
    val, gx, gy, gz = _tricubic_eval(unit, xin, yin, zin, hx, dhx, hy, dhy, hz, dhz)
    w = np.broadcast_to(val, (64, idx.shape[0])).T
    dw = np.stack([np.broadcast_to(g, (64, idx.shape[0])).T for g in (gx, gy, gz)], -1)
    return v, w, dw, pts.index((1, 1, 1))


def _grid_scales(case, g, pos, s):
    """Per atom of the flat positions pos [N, 3]: (D [N,3], V [N,3], E [N], R [N,3], Er [N], inside, idx, f) of grid g."""
    counts, sp, og = _geom(case, g)
    vals = np.asarray(case["grids"][g], dtype=np.float64)
    method = case.get("method", 0)
    n_pow = case["inv_power"][g] if case.get("inv_power") else 0.0
    h = np.array(sp, dtype=np.float64)
    inside, idx, f, alt_idx, alt_f = _classify(pos, counts, sp, og)
    N = pos.shape[0]
    D, V, E = np.zeros((N, 3)), np.zeros((N, 3)), np.zeros(N)
    has_alt = (alt_idx != idx).any(axis=1)
    for combo in range(8):
        if combo and not has_alt.any():
            break
        use = np.array([(combo >> a) & 1 for a in range(3)], dtype=bool)
        ci = np.where(use, alt_idx, idx)
        cf = np.where(use, alt_f, f)
        v, w, dw, k0 = _stencil(method, vals, counts, ci, cf)
        c = np.ones(N)
        if n_pow > 0.0:
            c = abs(n_pow) * np.abs(v).max(axis=1) ** (n_pow - 1.0)
        d = (np.abs(dw) * np.abs(v - v[:, k0:k0 + 1])[..., None]).sum(axis=1) / h
        vv = (np.abs(dw) * np.abs(v)[..., None]).sum(axis=1) / h
        e = (np.abs(w) * np.abs(v)).sum(axis=1)
        if n_pow > 0.0:
            e = np.abs(v).max(axis=1) ** n_pow
        D = np.maximum(D, (c * np.abs(s))[:, None] * d)
        V = np.maximum(V, (c * np.abs(s))[:, None] * vv)
        E = np.maximum(E, np.abs(s) * e)
    live = inside & (s != 0.0)
    D[~live], V[~live], E[~live] = 0.0, 0.0, 0.0
    rel = pos - np.array(og)
    hc = np.array(sp) * (np.array(counts) - 1)
    dev = np.where(rel < 0.0, rel, np.where(rel > hc, rel - hc, 0.0))
    k = case["oob_k"][g]
    R = np.abs(k * dev) * (~live)[:, None]
    Er = (0.5 * k * dev * dev).sum(axis=1) * (~live)
    return D, V, E, R, Er, inside, idx, f


def force_scale(case, pos):
    """Per-atom, per-axis scales of the terms the kernels sum to form each force: dict of D, V, R [R, A, 3] (see the module
    docstring) and, for reports, grid 0's inside flag [R, A], cell [R, A, 3] and fractions [R, A, 3]."""
    pos = np.asarray(pos, dtype=np.float64)
    r, a, _ = pos.shape
    flat = pos.reshape(-1, 3)
    out = dict(D=np.zeros((r * a, 3)), V=np.zeros((r * a, 3)), R=np.zeros((r * a, 3)))
    for g in range(len(case["grids"])):
        s = np.tile(np.asarray(case["scaling"][g], dtype=np.float64), r)
        D, V, _, R, _, inside, idx, f = _grid_scales(case, g, flat, s)
        out["D"] += D
        out["V"] += V
        out["R"] += R
        if g == 0:
            out.update(inside=inside.reshape(r, a), cell=idx.reshape(r, a, 3), frac=f.reshape(r, a, 3))
    for key in ("D", "V", "R"):
        out[key] = out[key].reshape(r, a, 3)
    return out


def energy_scale(case, pos):
    """(per replica [R], per atom [R, A]) sum over grids of |s| * sum_k |w_k| |v_k| over the points the method reads
    (|s| * max|v|^n on inv-power grids), plus the restraint energies."""
    pos = np.asarray(pos, dtype=np.float64)
    r, a, _ = pos.shape
    flat = pos.reshape(-1, 3)
    per_atom = np.zeros(r * a)
    for g in range(len(case["grids"])):
        s = np.tile(np.asarray(case["scaling"][g], dtype=np.float64), r)
        _, _, E, _, Er, _, _, _ = _grid_scales(case, g, flat, s)
        per_atom += E + Er
    per_atom = per_atom.reshape(r, a)
    return per_atom.sum(axis=1), per_atom


# ---------------------------------------------------------------------------------------------------------------------
# Checks
# ---------------------------------------------------------------------------------------------------------------------
def force_bound(f_ref, scale, tol_f, tol_d, tol_v, fixed_adds=0):
    return (tol_f * np.maximum(np.abs(f_ref), scale["R"]) + tol_d * scale["D"] + tol_v * scale["V"]
            + fixed_adds * FIXED_QUANTUM)


def check_forces(f, f_ref, scale, tol_f, tol_d, tol_v, fixed_adds=0, what=""):
    """Asserts |f - f_ref| <= bound per atom and component; returns the worst ratio err / bound. On failure the message
    names the worst atom: replica, atom, grid 0's cell and fractions, inside or outside."""
    f = np.asarray(f, dtype=np.float64).reshape(f_ref.shape)
    err = np.abs(f - f_ref)
    bound = force_bound(f_ref, scale, tol_f, tol_d, tol_v, fixed_adds)
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(bound > 0.0, err / np.where(bound > 0.0, bound, 1.0), np.where(err > 0.0, np.inf, 0.0))
    worst = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
    r, a, ax = worst
    worst_ratio = float(ratio[worst])
    assert worst_ratio <= 1.0, (
        f"{what}: force error {err[worst]:.3e} on replica {r} atom {a} axis {'xyz'[ax]} is {worst_ratio:.3g}x its bound "
        f"{bound[worst]:.3e} (f_ref {f_ref[worst]:.6e}, f {f[worst]:.6e}; D {scale['D'][worst]:.3e}, V {scale['V'][worst]:.3e}, "
        f"R {scale['R'][worst]:.3e}; {'inside' if scale['inside'][r, a] else 'outside'} cell {tuple(scale['cell'][r, a])} "
        f"fractions {tuple(float(x) for x in scale['frac'][r, a])}); {int((ratio > 1.0).sum())} components over")
    return worst_ratio


def check_energies(e, e_ref, escale, tol, what=""):
    """|e - e_ref| <= tol * escale, elementwise: per replica ([R]) or per atom ([R, A]). Returns the worst ratio."""
    e = np.asarray(e, dtype=np.float64).reshape(np.shape(e_ref))
    err = np.abs(e - e_ref)
    bound = tol * np.asarray(escale)
    ratio = np.where(bound > 0.0, err / np.where(bound > 0.0, bound, 1.0), np.where(err > 0.0, np.inf, 0.0))
    worst = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
    assert ratio[worst] <= 1.0, (f"{what}: energy error {err[worst]:.3e} at {worst} is {ratio[worst]:.3g}x its bound "
                                 f"{bound[worst]:.3e} (ref {np.asarray(e_ref)[worst]:.9e}, got {e[worst]:.9e})")
    return float(ratio[worst])


def _report(what, **ratios):
    print(f"POINTWISE {what}: " + " ".join(f"{k}={v:.3g}" for k, v in ratios.items()))


# ---------------------------------------------------------------------------------------------------------------------
# Inputs: forces of inside atoms spanning about four decades
# ---------------------------------------------------------------------------------------------------------------------
def _field(counts, rng, amp=4.0):
    """A smooth field of amplitude amp plus noise of amplitude 0.1 * amp, the noise 1e-3 of that in the octant at the
    origin; FP32-representable."""
    nx, ny, nz = counts
    x = np.sin(2 * np.pi * np.arange(nx) / max(nx - 1, 1))[:, None, None]
    y = np.cos(2 * np.pi * np.arange(ny) / max(ny - 1, 1) + 0.3)[None, :, None]
    z = np.sin(np.pi * np.arange(nz) / max(nz - 1, 1) + 0.7)[None, None, :]
    noise = rng.normal(size=counts) * 0.1 * amp
    noise[:(nx + 1) // 2, :(ny + 1) // 2, :(nz + 1) // 2] *= 1e-3
    return (amp * x * y * z + noise).astype(np.float32).astype(np.float64)


def _case(n_grids, r, a, seed, method=0, counts=cov.COUNTS, sp=cov.SPACING, og=cov.ORIGIN, edges=True):
    """test_gpu_coverage._case's atoms (8 % outside up to 0.3 box lengths deep, edge cells and upper faces, zero scaling
    factors) on _field grids."""
    c = cov._case(n_grids, r, a, seed, method=method, counts=counts, sp=sp, og=og, edges=edges)
    rng = np.random.default_rng(seed + 7)
    c["grids"] = [_field(counts, rng) for _ in range(n_grids)]
    return c


def _oracle_atoms(oracle, c, pos):
    """Per-atom energies [R, A] from one-atom oracle runs (summed over grids)."""
    want = np.zeros(pos.shape[:2])
    for ia in range(pos.shape[1]):
        g1, _ = cov._oracle(oracle, c, pos=np.ascontiguousarray(pos[:, ia:ia + 1]), scaling=np.asarray(c["scaling"])[:, ia:ia + 1])
        want[:, ia] = g1.sum(axis=1)
    return want


def _emulate_mixed_one_grid(c, pos):
    """numpy emulation of the one-grid MIXED lines kernel's force: trilinear<float> on FP32 fractions (corner differences
    first), fmaf with the float scaling factor, the FP32 product with (float) 1/spacing; restraint in FP64 rounded to
    float. Returns forces [R, A, 3] as float64."""
    r, a, _ = pos.shape
    flat = pos.reshape(-1, 3)
    inside, idx, f, _, _ = _classify(flat, c["counts"], c["spacing"], c["origin"])
    s = np.tile(np.asarray(c["scaling"][0]), r)
    vals = np.asarray(c["grids"][0], dtype=np.float32)
    v = [vals[idx[:, 0] + i, idx[:, 1] + j, idx[:, 2] + k] for i, j, k in itertools.product((0, 1), repeat=3)]
    f32 = np.float32
    fx, fy, fz = (f[:, k].astype(f32) for k in range(3))
    one = f32(1.0)
    ax, ay, az = one - fx, one - fy, one - fz
    dx = ((v[4] - v[0]) * az + (v[5] - v[1]) * fz) * ay + ((v[6] - v[2]) * az + (v[7] - v[3]) * fz) * fy
    dy = ((v[2] - v[0]) * az + (v[3] - v[1]) * fz) * ax + ((v[6] - v[4]) * az + (v[7] - v[5]) * fz) * fx
    dz = ((v[1] - v[0]) * ay + (v[3] - v[2]) * fy) * ax + ((v[5] - v[4]) * ay + (v[7] - v[6]) * fy) * fx
    sf = s.astype(f32)
    inv = (1.0 / np.asarray(c["spacing"])).astype(f32)
    live = inside & (s != 0.0)
    F = np.zeros((r * a, 3))
    for ax_, d in enumerate((dx, dy, dz)):
        F[:, ax_] = np.where(live, -(sf * d) * inv[ax_], 0.0).astype(f32)
    rel = flat - np.array(c["origin"])
    hc = np.array(c["spacing"]) * (np.array(c["counts"]) - 1)
    dev = np.where(rel < 0.0, rel, np.where(rel > hc, rel - hc, 0.0))
    F -= np.where(live[:, None], 0.0, (c["oob_k"][0] * dev).astype(f32))
    return F.reshape(r, a, 3)


# ---------------------------------------------------------------------------------------------------------------------
# CPU self-tests of the checker
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("method", [0, 1, 2], ids=["trilinear", "bspline", "tricubic"])
def test_checker_passes_the_oracle_against_itself(oracle_built, method):
    c = _case(3, 5, 47, seed=1 + method, method=method)
    ge_ref, f_ref = cov._oracle(oracle_built, c)
    scale = force_scale(c, c["pos"])
    inner = scale["inside"] & (np.abs(f_ref).max(axis=-1) > 0)
    assert (scale["D"][inner].max(axis=-1) > 0).all()
    assert check_forces(f_ref, f_ref, scale, **_tol(0, method)) == 0.0
    e_scale, _ = energy_scale(c, c["pos"])
    assert (e_scale > 0).all()
    assert check_energies(ge_ref.sum(axis=1), ge_ref.sum(axis=1), e_scale, TOL_E) == 0.0
    # the scales bound what they claim to: |F| <= D (a difference of corners against the first corner) plus R
    assert (np.abs(f_ref) <= (1.0 + 1e-9) * scale["D"] + scale["R"]).all()


def _emulation_case(oracle):
    c = _case(1, 256, 47, seed=2024, edges=True)
    ge_ref, f_ref = cov._oracle(oracle, c)
    return c, f_ref, force_scale(c, c["pos"])


def test_checker_passes_the_fp32_emulation(oracle_built):
    """The one-grid MIXED gradient emulated in FP32 passes at TOL_TRILINEAR_F32."""
    c, f_ref, scale = _emulation_case(oracle_built)
    f = _emulate_mixed_one_grid(c, c["pos"])
    assert np.abs(f - f_ref).max() > 0.0
    check_forces(f, f_ref, scale, **TOL_TRILINEAR_F32, what="emulation")


def test_planted_error_fails_pointwise_passes_max_norm(oracle_built):
    """Forces of the inside atoms with below-median |F| scaled by (1 + 3e-4): the max-norm criterion of the other GPU tests
    (1e-5 of max|F|) passes it, the per-atom check does not."""
    c, f_ref, scale = _emulation_case(oracle_built)
    f = _emulate_mixed_one_grid(c, c["pos"])
    mag = np.abs(f_ref).max(axis=-1)
    inside = scale["inside"] & (mag > 0)
    small = inside & (mag < np.median(mag[inside]))
    f[small] *= 1.0 + 3e-4
    assert cov._err_f(f, f_ref) <= 1e-5
    with pytest.raises(AssertionError, match="its bound"):
        check_forces(f, f_ref, scale, **TOL_TRILINEAR_F32, what="planted")


def test_wrong_corner_in_one_edge_cell_fails(oracle_built):
    """One atom in the last cell of an axis evaluated with two corners of its cell swapped (what a wrong slot or granule
    mapping does to one stencil): the per-atom check fails on that atom."""
    c, f_ref, scale = _emulation_case(oracle_built)
    f = _emulate_mixed_one_grid(c, c["pos"])
    n = np.array(c["counts"])
    cell, inside = scale["cell"], scale["inside"]
    edge = inside & (cell == n - 2).any(axis=-1) & (c["scaling"][0][None, :] != 0)
    mag = np.where(edge, np.abs(f_ref).max(axis=-1), np.inf)
    r, a = np.unravel_index(int(np.argmin(mag)), mag.shape)        # the edge atom with the smallest force
    grid = c["grids"][0].copy()
    ix, iy, iz = cell[r, a]
    grid[ix + 1, iy, iz + 1], grid[ix + 1, iy + 1, iz] = grid[ix + 1, iy + 1, iz], grid[ix + 1, iy, iz + 1]
    wrong = dict(c, grids=[grid])
    _, f_wrong = cov._oracle(oracle_built, wrong, pos=np.ascontiguousarray(c["pos"][r:r + 1]))
    f[r, a] = f_wrong[0, a]
    with pytest.raises(AssertionError, match=f"replica {r} atom {a} "):
        check_forces(f, f_ref, scale, **TOL_TRILINEAR_F32, what="wrong corner")


# ---------------------------------------------------------------------------------------------------------------------
# GPU cases
# ---------------------------------------------------------------------------------------------------------------------
def _make(gf, dev, c, precision, layout, particles=None):
    return cov._make(gf, dev, c, precision, layout, particles=particles)


def _check_host(k, c, ge_ref, f_ref, tol, what, force_mode=None, want_forces=True):
    """execute_host (F64_STORE unless force_mode says otherwise) against the oracle, per atom and per replica."""
    import openmmgridforce_b200 as gf
    scale = force_scale(c, c["pos"])
    e_scale, _ = energy_scale(c, c["pos"])
    if not want_forces:
        en, none, _ = k.execute_host(c["pos"], want_forces=False)
        assert none is None
        re = check_energies(en, ge_ref.sum(axis=1), e_scale, TOL_E, what + " energy-only")
        _report(what + " energy-only", energy=re)
        return
    mode = gf.FORCE_F64_STORE if force_mode is None else force_mode
    en, forces, _ = k.execute_host(c["pos"], force_mode=mode)
    t = _f32_output(tol) if mode == gf.FORCE_F32_STORE else tol
    rf = check_forces(forces, f_ref, scale, **t, what=what)
    re = check_energies(en, ge_ref.sum(axis=1), e_scale, TOL_E, what)
    _report(what, force=rf, energy=re)


# Path 1: the lines kernel ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_grids", [1, 2, 3, 4])
def test_lines_host_modes(gpu_device, oracle_built, n_grids):
    """F64_STORE (pageable), F32_STORE into pinned memory (host zero-copy) and energy-only through execute_host."""
    import torch
    import openmmgridforce_b200 as gf
    c = _case(n_grids, 200, 47, seed=10 + n_grids)
    ge_ref, f_ref = cov._oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, 0, CELLS)
    assert k.eval_path() == 1
    tol = _tol(0, 0, n_grids, path=1)
    _check_host(k, c, ge_ref, f_ref, tol, f"lines{n_grids} f64_store")
    pos_pin = torch.from_numpy(c["pos"].copy()).pin_memory()
    f_pin = torch.full(c["pos"].shape, 7.0, dtype=torch.float32).pin_memory()
    en, _, _ = k.execute_host(pos_pin.numpy(), forces=f_pin.numpy(), force_mode=gf.FORCE_F32_STORE)
    scale = force_scale(c, c["pos"])
    rf = check_forces(f_pin.numpy(), f_ref, scale, **_f32_output(tol), what=f"lines{n_grids} f32_store pinned")
    _report(f"lines{n_grids} f32_store pinned", force=rf)
    _check_host(k, c, ge_ref, f_ref, tol, f"lines{n_grids}", want_forces=False)
    cov._close(grids, k)


def _device_fixed(gf, k, c, launches, stream):
    """`launches` FIXED_ADD launches into one buffer; returns (energies of the last launch, summed forces [R, A, 3])."""
    import torch
    dev = torch.device("cuda:0")
    r, a, _ = c["pos"].shape
    n = r * a
    stride = ((n + 31) // 32) * 32
    d_pos = torch.from_numpy(c["pos"]).to(dev)
    d_f = torch.zeros(3 * stride, dtype=torch.int64, device=dev)
    d_e = [torch.zeros(r, dtype=torch.float64, device=dev) for _ in range(2)]
    d_out = torch.empty(n, 3, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    for i in range(launches):
        k.execute_device(r, a, d_pos.data_ptr(), d_e[i % 2].data_ptr(), None, d_f.data_ptr(), gf.FORCE_FIXED_ADD, stride, None,
                         stream.cuda_stream, d_energies_clear=d_e[(i + 1) % 2].data_ptr())
    k.device.fixed_to_f64(d_f.data_ptr(), stride, n, d_out.data_ptr(), stream.cuda_stream)
    stream.synchronize()
    return d_e[(launches - 1) % 2].cpu().numpy(), d_out.cpu().numpy().reshape(r, a, 3)


@pytest.mark.gpu
@pytest.mark.parametrize("n_grids", [1, 2, 3, 4])
def test_lines_device_fixed_point(gpu_device, oracle_built, n_grids):
    """FIXED_ADD on the device path, one block per tile (launch overlap off) and the tile-striding instantiation (launch
    overlap on; 9000 replicas of 47 atoms are 6 610 tiles, 2-6 per block): two launches into one buffer."""
    import torch
    import openmmgridforce_b200 as gf
    c = _case(n_grids, 9000, 47, seed=20 + n_grids)
    ge_ref, f_ref = cov._oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, 0, CELLS)
    assert k.eval_path() == 1
    tol = _tol(0, 0, n_grids, path=1)
    scale = force_scale(c, c["pos"])
    e_scale, _ = energy_scale(c, c["pos"])
    stream = torch.cuda.Stream()
    for overlap in (False, True):
        k.set_launch_overlap(overlap)
        en, fsum = _device_fixed(gf, k, c, 2, stream)
        what = f"lines{n_grids} fixed {'tile-striding' if overlap else 'one block per tile'}"
        rf = check_forces(fsum / 2, f_ref, scale, **tol, fixed_adds=1, what=what)
        re = check_energies(en, ge_ref.sum(axis=1), e_scale, TOL_E, what)
        _report(what, force=rf, energy=re)
    k.set_launch_overlap(False)
    cov._close(grids, k)


# Paths 2-6: the record kernels ----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_grids", [2, 3, 4])
def test_double_records(gpu_device, oracle_built, n_grids):
    import openmmgridforce_b200 as gf
    c = _case(n_grids, 200, 47, seed=30 + n_grids)
    ge_ref, f_ref = cov._oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, 1, CELLS)
    assert k.eval_path() == 2
    _check_host(k, c, ge_ref, f_ref, _tol(1, 0), f"double-records{n_grids}")
    cov._close(grids, k)


@pytest.mark.gpu
@pytest.mark.parametrize("n_grids", [1, 2, 3, 4])
@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
@pytest.mark.parametrize("method", [1, 2], ids=["bspline", "tricubic"])
def test_record_kernels(gpu_device, oracle_built, method, precision, n_grids):
    """Paths 3-6 with edge cells and upper faces."""
    import openmmgridforce_b200 as gf
    layout = cov.RECORD_LAYOUT[method]
    c = _case(n_grids, 37, 47, seed=100 * method + 10 * precision + n_grids, method=method)
    ge_ref, f_ref = cov._oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, precision, layout)
    assert k.eval_path() == cov._path(precision, layout, n_grids)
    _check_host(k, c, ge_ref, f_ref, _tol(precision, method), f"records m{method} p{precision} g{n_grids}")
    cov._close(grids, k)


# Path 0: the general kernel -------------------------------------------------------------------------------------------
GENERAL = [(1, CELLS, 1), (0, ROWS, 1), (1, ROWS, 1), (0, PAIRS, 1), (0, BSPLINE_POINTS, 1), (1, BSPLINE_POINTS, 2),
           (0, POINTS, 1), (1, POINTS, 2), (0, CELLS, 5), (1, CELLS, 5), (0, CELLS, 8), (0, ROWS, 8)]


@pytest.mark.gpu
@pytest.mark.parametrize("spec", GENERAL, ids=[f"{'mixed' if p == 0 else 'double'}-{cov.LAYOUT_IDS[l]}{g}" for p, l, g in GENERAL])
def test_general_kernel(gpu_device, oracle_built, spec):
    import openmmgridforce_b200 as gf
    precision, layout, n_grids = spec
    method = METHOD[layout]
    c = _case(n_grids, 23, 47, seed=200 + 10 * layout + n_grids + precision, method=method)
    ge_ref, f_ref = cov._oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, precision, layout)
    assert k.eval_path() == 0
    _check_host(k, c, ge_ref, f_ref, _tol(precision, method), f"general {spec}")
    cov._close(grids, k)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
def test_general_kernel_mixed_geometry(gpu_device, oracle_built, precision):
    """Three grids of different geometry, overlapping in part: atoms inside one grid and outside another."""
    import openmmgridforce_b200 as gf
    rng = np.random.default_rng(300 + precision)
    geoms = [((23, 19, 31), (0.05, 0.07, 0.04), (0.3, -0.2, 1.0)), ((17, 21, 15), (0.06, 0.05, 0.07), (0.6, 0.1, 1.3)),
             ((29, 13, 19), (0.04, 0.09, 0.05), (0.1, 0.3, 0.9))]
    r, a = 23, 47
    pos = rng.uniform(0.0, 1.0, size=(r, a, 3)) * np.array([1.3, 1.3, 1.4]) + np.array([0.1, -0.2, 0.85])
    sc = rng.normal(size=(3, a))
    sc[:, ::7] = 0.0
    c = dict(geoms=geoms, grids=[_field(g[0], rng) for g in geoms], scaling=sc, pos=pos, oob_k=cov.OOB_K[:3],
             inv_power=[0.0] * 3, method=0)
    ge_ref = np.zeros((r, 3))
    f_ref = np.zeros_like(pos)
    for g, (cnt, sp, og) in enumerate(geoms):
        port = oracle_built.PortOracle(cnt, sp, og, [c["grids"][g]], sc[g:g + 1], oob_k=[c["oob_k"][g]])
        e, f = port.execute_batched(pos, n_threads=N_THREADS)
        ge_ref[:, g] = e[:, 0]
        f_ref += f
    grids = [gf.Grid(gpu_device, cnt, sp, og, v, precision, layout=CELLS) for (cnt, sp, og), v in zip(geoms, c["grids"])]
    k = gf.Kernel(gpu_device, grids, sc, oob_k=c["oob_k"])
    assert k.eval_path() == 0
    scale = force_scale(c, pos)
    ins = [_classify(pos.reshape(-1, 3), *g)[0] for g in geoms]
    assert (ins[0] & ~ins[1]).any() and (ins[1] & ~ins[0]).any()
    _check_host(k, c, ge_ref, f_ref, _tol(precision, 0), f"mixed geometry p{precision}")
    assert scale["D"].any()
    cov._close(grids, k)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
def test_general_kernel_inv_power_one_of_three(gpu_device, oracle_built, precision):
    import openmmgridforce_b200 as gf
    c = _case(3, 23, 47, seed=404 + precision)
    c["grids"][1] = np.random.default_rng(5).uniform(0.5, 3.0, size=cov.COUNTS).astype(np.float32).astype(np.float64)
    c["inv_power"] = [0.0, 4.0, 0.0]
    ge_ref, f_ref = cov._oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, precision, CELLS)
    assert k.eval_path() == 0
    _check_host(k, c, ge_ref, f_ref, _tol(precision, 0), f"inv-power p{precision}")
    cov._close(grids, k)


@pytest.mark.gpu
def test_general_kernel_sorted_order(gpu_device, oracle_built):
    """ROWS (the general kernel) on the device path in the evaluation order of sort_atoms, F64_STORE."""
    import torch
    import openmmgridforce_b200 as gf
    c = _case(1, 300, 47, seed=505)
    ge_ref, f_ref = cov._oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, 0, ROWS)
    assert k.eval_path() == 0
    dev = torch.device("cuda:0")
    r, a, _ = c["pos"].shape
    n = r * a
    d_pos = torch.from_numpy(c["pos"]).to(dev)
    d_order = torch.full((n,), -1, dtype=torch.int32, device=dev)
    d_e = torch.zeros(r, dtype=torch.float64, device=dev)
    d_f = torch.zeros(n * 3, dtype=torch.float64, device=dev)
    stream = torch.cuda.Stream()
    torch.cuda.synchronize()
    k.sort_atoms(r, a, d_pos.data_ptr(), d_order.data_ptr(), stream.cuda_stream)
    k.execute_device(r, a, d_pos.data_ptr(), d_e.data_ptr(), None, d_f.data_ptr(), gf.FORCE_F64_STORE, 0, d_order.data_ptr(),
                     stream.cuda_stream)
    stream.synchronize()
    order = d_order.cpu().numpy()
    assert np.array_equal(np.sort(order), np.arange(n)) and not np.array_equal(order, np.arange(n))
    scale = force_scale(c, c["pos"])
    e_scale, _ = energy_scale(c, c["pos"])
    rf = check_forces(d_f.cpu().numpy().reshape(r, a, 3), f_ref, scale, **_tol(0, 0), what="sorted order")
    re = check_energies(d_e.cpu().numpy(), ge_ref.sum(axis=1), e_scale, TOL_E, "sorted order")
    _report("sorted order", force=rf, energy=re)
    cov._close(grids, k)


# Entry points ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("buffers", ["pinned", "pageable"])
def test_chunked_host_pipeline(gpu_device, oracle_built, buffers):
    """4 000 replicas x 47 atoms: 4.5 MB of positions, so execute_host copies and evaluates in 2 chunks."""
    import torch
    import openmmgridforce_b200 as gf
    c = _case(3, 4000, 47, seed=600)
    assert c["pos"].nbytes >= 4 << 20
    ge_ref, f_ref = cov._oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, 0, CELLS)
    assert k.eval_path() == 1
    keep = []
    if buffers == "pinned":
        tp, tf = torch.from_numpy(c["pos"].copy()).pin_memory(), torch.zeros(c["pos"].shape, dtype=torch.float64).pin_memory()
        te = torch.zeros(c["pos"].shape[0], dtype=torch.float64).pin_memory()
        keep = [tp, tf, te]
        pos, forces, en_out = tp.numpy(), tf.numpy(), te.numpy()
    else:
        pos, forces, en_out = c["pos"].copy(), np.zeros_like(c["pos"]), np.zeros(c["pos"].shape[0])
    en, forces, _ = k.execute_host(pos, forces=forces, energies_out=en_out)
    scale = force_scale(c, c["pos"])
    e_scale, _ = energy_scale(c, c["pos"])
    what = f"chunked {buffers}"
    rf = check_forces(forces, f_ref, scale, **_tol(0, 0, 3, path=1), what=what)
    re = check_energies(en, ge_ref.sum(axis=1), e_scale, TOL_E, what)
    _report(what, force=rf, energy=re)
    del keep
    cov._close(grids, k)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
@pytest.mark.parametrize("n_replicas", [2, 21])
def test_small_host_mapped(gpu_device, oracle_built, n_replicas, precision):
    """At most 4 096 particles in all: one launch on host-mapped staging."""
    import openmmgridforce_b200 as gf
    c = _case(3, n_replicas, 47, seed=700 + n_replicas)
    assert n_replicas * 47 <= 4096
    ge_ref, f_ref = cov._oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, precision, CELLS)
    assert k.eval_path() == (1 if precision == 0 else 2)
    tol = _tol(precision, 0, 3, path=k.eval_path())
    _check_host(k, c, ge_ref, f_ref, tol, f"mapped r{n_replicas} p{precision}")
    _check_host(k, c, ge_ref, f_ref, tol, f"mapped r{n_replicas} p{precision}", want_forces=False)
    cov._close(grids, k)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
def test_resident_moving_ligand(gpu_device, oracle_built, precision):
    """The resident evaluator: 20 steps of one 47-atom ligand moving through the grid."""
    import openmmgridforce_b200 as gf
    c = _case(1, 1, 47, seed=800 + precision)
    rng = np.random.default_rng(801)
    steps = np.cumsum(rng.normal(scale=0.02, size=(20, 1, 3)), axis=0)
    c["pos"] = np.ascontiguousarray(c["pos"][0][None] + steps)
    ge_ref, f_ref = cov._oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, precision, CELLS)
    grids2, k2 = _make(gf, gpu_device, c, precision, CELLS)
    assert k.eval_path() == cov._path(precision, CELLS, 1)
    k2.execute_host(c["pos"][0])     # the launch path's module is loaded before the block resides
    k.set_resident(True)
    scale = force_scale(c, c["pos"])
    e_scale, _ = energy_scale(c, c["pos"])
    tol = _tol(precision, 0)
    worst_f = worst_e = 0.0
    for step in range(20):
        en, forces, _ = k.execute_host(c["pos"][step])
        sl = slice(step, step + 1)
        sc = dict(scale, D=scale["D"][sl], V=scale["V"][sl], R=scale["R"][sl], inside=scale["inside"][sl], cell=scale["cell"][sl],
                  frac=scale["frac"][sl])
        worst_f = max(worst_f, check_forces(forces, f_ref[sl], sc, **tol, what=f"resident step {step}"))
        worst_e = max(worst_e, check_energies(en, ge_ref[sl].sum(axis=1), e_scale[sl], TOL_E, f"resident step {step}"))
    assert 1 <= k.resident_launches() <= 2
    _report(f"resident p{precision}", force=worst_f, energy=worst_e)
    k.set_resident(False)
    cov._close(grids, k)
    cov._close(grids2, k2)


ATOM_ENERGY = [(0, CELLS, 3), (1, CELLS, 3), (0, BSPLINE, 2), (1, HERMITE, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("spec", ATOM_ENERGY, ids=[f"{'mixed' if p == 0 else 'double'}-{cov.LAYOUT_IDS[l]}{g}" for p, l, g in ATOM_ENERGY])
def test_per_atom_energies(gpu_device, oracle_built, spec):
    """request_atom_energies against the oracle run on one-atom replicas, per atom."""
    import openmmgridforce_b200 as gf
    precision, layout, n_grids = spec
    method = METHOD[layout]
    c = _case(n_grids, 9, 47, seed=900 + layout + precision, method=method)
    grids, k = _make(gf, gpu_device, c, precision, layout)
    assert k.eval_path() == cov._path(precision, layout, n_grids)
    k.request_atom_energies(True)
    en, _, _ = k.execute_host(c["pos"])
    ae = k.atom_energies(c["pos"].shape[0])
    want = _oracle_atoms(oracle_built, c, c["pos"])
    e_rep, e_atom = energy_scale(c, c["pos"])
    ra = check_energies(ae, want, e_atom, TOL_E, f"atom energies {spec}")
    re = check_energies(en, want.sum(axis=1), e_rep, TOL_E, f"replica energies {spec}")
    _report(f"atom energies {spec}", atom=ra, energy=re)
    k.request_atom_energies(False)
    cov._close(grids, k)


@pytest.mark.gpu
def test_c5_workload_sample(gpu_device, oracle_built):
    """8 192 replicas of the benchmark's C5 workload (3 grids of 192^3, not FP32-representable): the storage rounding of
    each point enters V (force) and the energy scale."""
    import openmmgridforce_b200 as gf
    from openmmgridforce_b200 import workloads as W
    w = W.c5_sharded_replicas(n_local=8192)
    c = dict(counts=w.counts, spacing=w.spacing, origin=w.origin, grids=w.grids, scaling=w.scaling, pos=w.pos, oob_k=w.oob_k,
             inv_power=w.inv_power, method=0)
    ge_ref, f_ref = cov._oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, 0, CELLS)
    assert k.eval_path() == 1
    en, forces, _ = k.execute_host(w.pos)
    scale = force_scale(c, w.pos)
    e_scale, _ = energy_scale(c, w.pos)
    tol = dict(_tol(0, 0, 3, path=1))
    tol["tol_v"] += U          # storage: each point within 2^-24 of its FP64 value
    rf = check_forces(forces, f_ref, scale, **tol, what="C5 sample")
    re = check_energies(en, ge_ref.sum(axis=1), e_scale, TOL_E_STORAGE, "C5 sample")
    _report("C5 sample", force=rf, energy=re)
    cov._close(grids, k)
