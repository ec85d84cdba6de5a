"""Parity on every cell of production-size grids (-m gpu), for every layout and every grid-construction route, with CPU
self-tests of the position generator and of the checker.

The other value-checked tests use grids of at most ~80 K points, or put their atoms where ligand poses land (within ~0.9 nm
of the centre of a full-size grid). Here one atom sits in EVERY cell of two production-size worlds, plus a shell of atoms
on, just inside and just outside every face, edge and corner, all shuffled over 47-atom replicas so that each warp reads
records from all over the grid:

  world T  C4's geometry, 208 x 278 x 231 points at 0.0125 nm from TEST_GRID_ORIGIN (13 187 970 cells; the DOUBLE 3-grid
           record table is 3.14 GiB, so every record past ~8.39 M cells sits above the 2 GiB byte offset), 4 grids;
  world S  181 x 211 x 187 points, anisotropic (7 030 800 cells; the B-spline / tricubic records take 47 grid-stride
           passes of the repack kernel on a B200, the point layouts 6), 2 grids, interpolation methods 1 and 2.

Grids are FP32-representable, scaling factors non-zero (|s| in [0.5, 1.5], random signs, different per grid), so every
cell is checked for every grid. Two tiers:

  exhaustive  every atom, against a bound that needs no per-atom weights: for each cell and grid Rng = max - min and
              Mx = max |v| of the values the method reads (the 2x2x2 cell, the clamped 4x4x4 block, the tricubic flat-index
              neighbourhood with its wrapped reads and zeros), and
                |f - f_ref| <= tol_f * max(|f_ref|, R) + sum_g |s_g| * (tol_d * C_dw * Rng + tol_v * C_dw * Mx) / h_a + n 2^-32
                |e - e_ref| <= TOL_E * (sum_g |s_g| * C_w * Mx + restraint energies)
                               + FRAC_ROUNDING * sum_a q_a * sum_g |s_g| * C_dw * Rng         (per atom; per replica summed)
              with test_gpu_pointwise's constants. C_dw bounds sum_k |dw_k/da| and C_w sum_k |w_k| over the points; both
              are measured on a fraction grid in every xin/yin/zin case (weight_bounds). This is test_gpu_pointwise's
              bound with D <= C_dw * Rng and V <= C_dw * Mx, so it is never tighter than that one.
  exact       ~110 K atoms (every replica that holds a shell atom plus a stride through the rest) with test_gpu_pointwise's
              own per-atom scales and bounds (energies: plus FRAC_ROUNDING * sum_a q_a * h_a * D_a).

Every GPU case asserts gfb_kernel_eval_path. The grid-construction routes (V3 files streamed in 32 MB pieces, device
pointers) must give bit-identical per-atom forces and energies to a Grid built from host memory, and the inv-power
transform is held to 2 ulp of the C oracle on 13.4 M values.
"""
import functools
import itertools
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_gpu_pointwise as pw  # noqa: E402
from openmmgridforce_b200 import workloads as W  # noqa: E402

cov = pw.cov
U = pw.U
CELLS, ROWS, PAIRS, BSPLINE, POINTS, HERMITE, BSPLINE_POINTS = 1, 2, 3, 4, 5, 6, 7
METHOD = pw.METHOD
N_ATOMS = 47

T_COUNTS, T_SPACING, T_ORIGIN = W.TEST_GRID_COUNTS, (W.TEST_GRID_SPACING,) * 3, W.TEST_GRID_ORIGIN
S_COUNTS, S_SPACING, S_ORIGIN = (181, 211, 187), (0.0125, 0.011, 0.0135), (-0.61234567, 0.9876543, 0.3141592653)
EXACT_ATOMS = 100_000          # the exact tier's stride sample (the replicas holding shell atoms come on top)
# The MIXED kernels form a fraction from pi * fl(1/h), within 3.3e-16 * q of the oracle's pi / h (gf_eval_lines.cuh,
# classify_fast), so an energy may move by |dE/df_a| * 3.3e-16 * q_a <= 3.3e-16 * q_a * h_a * D_a. At q of 30 (the other
# tests' grids) that is far below TOL_E; at q of 277 it is not: measured on a B200 (1000 W) without this term, per-atom
# energies reached 1.47x TOL_E's bound (3-grid lines kernel, q_y = 263) and 2.34x (MIXED tricubic records).
FRAC_ROUNDING = 3.3e-16


# ---------------------------------------------------------------------------------------------------------------------
# Positions: one atom in every cell, a shell on and around the faces, shuffled into 47-atom replicas
# ---------------------------------------------------------------------------------------------------------------------
def exact_upper_face(og, hc):
    """A coordinate p with p - og == hc in FP64 (the kernels' and the oracle's upper-face test), searched within 8 ulp of
    og + hc. Not every origin admits one (p - og may round past hc from both neighbours): the worlds' origins do."""
    p0 = og + hc
    for step in sorted(range(-8, 9), key=abs):
        p = p0
        for _ in range(abs(step)):
            p = np.nextafter(p, np.inf if step > 0 else -np.inf)
        if p - og == hc:
            return float(p)
    raise AssertionError(f"no coordinate within 8 ulp of {p0!r} lies exactly on the upper face (origin {og!r})")


def every_cell_positions(counts, sp, og, rng):
    """[n_cells, 3]: one atom in each cell, in memory order, at fractions U(1e-6, 1 - 1e-6) (far enough from 0 and 1 that
    FP64 rounding of origin + (cell + fraction) * spacing cannot move it to a neighbouring cell)."""
    ncell = tuple(int(n) - 1 for n in counts)
    idx = np.stack(np.unravel_index(np.arange(int(np.prod(ncell))), ncell), 1)
    return np.asarray(og, dtype=np.float64) + (idx + rng.uniform(1e-6, 1.0 - 1e-6, size=idx.shape)) * np.asarray(sp)


OUT_DEPTHS = np.array([1e-9, 1e-4, 0.02, 0.3, 1.5])       # nm beyond a face


def shell_positions(counts, sp, og, rng):
    """Atoms exactly on each of the 6 faces (16 each), 12 edges (4 each) and 8 corners, 1 ulp inside and 1 ulp outside each
    face (4 each), outside each face at OUT_DEPTHS and outside each corner along its diagonal. Free coordinates are inside,
    away from the faces. Upper-face coordinates satisfy pos - origin == spacing * (counts - 1) in FP64."""
    sp, og = np.asarray(sp, dtype=np.float64), np.asarray(og, dtype=np.float64)
    hc = sp * (np.array(counts) - 1)
    face = [og.copy(), np.array([exact_upper_face(og[a], hc[a]) for a in range(3)])]

    def inner(m):
        return og + rng.uniform(0.02, 0.98, size=(m, 3)) * hc

    out = []
    for a in range(3):
        for side in (0, 1):
            inward = np.inf if side == 0 else -np.inf
            for m, coord in ((16, face[side][a]), (4, np.nextafter(face[side][a], inward)), (4, np.nextafter(face[side][a], -inward)),
                             (len(OUT_DEPTHS), face[side][a] + (OUT_DEPTHS if side else -OUT_DEPTHS))):
                p = inner(m)
                p[:, a] = coord
                out.append(p)
    for a, b in ((0, 1), (0, 2), (1, 2)):
        for sa, sb in itertools.product((0, 1), repeat=2):
            p = inner(4)
            p[:, a], p[:, b] = face[sa][a], face[sb][b]
            out.append(p)
    for s in itertools.product((0, 1), repeat=3):
        corner = np.array([face[s[a]][a] for a in range(3)])
        out.append(corner[None])
        out.append(corner + np.array([0.05, 0.7])[:, None] * np.where(np.array(s) == 1, 1.0, -1.0))
    return np.concatenate(out)


def pack_atoms(cell_pos, shell_pos, rng):
    """Every-cell and shell atoms, the last replica padded with shell atoms, under one seeded global permutation.
    Returns (pos [R, 47, 3], shell flag [R * 47])."""
    n = len(cell_pos) + len(shell_pos)
    extra = shell_pos[np.arange((-n) % N_ATOMS) % len(shell_pos)]
    pos = np.concatenate([cell_pos, shell_pos, extra])
    shell = np.zeros(len(pos), dtype=bool)
    shell[len(cell_pos):] = True
    perm = rng.permutation(len(pos))
    return np.ascontiguousarray(pos[perm].reshape(-1, N_ATOMS, 3)), shell[perm]


def world_atoms(counts, sp, og, seed):
    rng = np.random.default_rng(seed)
    return pack_atoms(every_cell_positions(counts, sp, og, rng), shell_positions(counts, sp, og, rng), rng)


# ---------------------------------------------------------------------------------------------------------------------
# Fraction-free per-cell scales
# ---------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def weight_bounds(method):
    """(C_w, C_dw): the largest sum_k |w_k| and sum_k |dw_k/da| (per unit fraction, any axis a) over the points method reads,
    taken over a 1/32 fraction grid on [0, 1]^3 in every xin/yin/zin case (tricubic: first cell layer or not), times 1.02
    for what lies between the samples. Weights of a point read twice are kept apart, as the kernels sum them."""
    t = np.linspace(0.0, 1.0, 33)
    f = np.stack(np.meshgrid(t, t, t, indexing="ij"), -1).reshape(-1, 3)
    counts = (4, 4, 4)
    cells = itertools.product((0, 1), repeat=3) if method == 2 else [(1, 1, 1)]
    cw = cdw = 0.0
    for cell in cells:
        idx = np.broadcast_to(np.array(cell), f.shape).copy()
        _, w, dw, _ = pw._stencil(method, np.zeros(counts), counts, idx, f)
        cw = max(cw, float(np.abs(w).sum(axis=1).max()))
        cdw = max(cdw, float(np.abs(dw).sum(axis=1).max()))
    return 1.02 * cw, 1.02 * cdw


def _window(a, step, fn):
    """fn over a[i - step], a[i], a[i + step], a[i + 2 step] (wrapping: callers pad so that the wrap is never read)."""
    return fn.reduce([np.roll(a, -o * step) for o in (-1, 0, 1, 2)])


def cell_ranges(method, vals):
    """(Rng, Mx) [nx-1, ny-1, nz-1]: max - min and max |v| of the values `method` reads for each cell."""
    from scipy import ndimage
    v = np.asarray(vals, dtype=np.float64)
    if method == 0:
        hi, lo = v, v
        for ax in range(3):
            a, b = [slice(None)] * 3, [slice(None)] * 3
            a[ax], b[ax] = slice(None, -1), slice(1, None)
            hi = np.maximum(hi[tuple(a)], hi[tuple(b)])
            lo = np.minimum(lo[tuple(a)], lo[tuple(b)])
    elif method == 1:       # points clamp(i-1) .. clamp(i+2) on each axis
        hi = ndimage.maximum_filter(v, size=4, mode="nearest", origin=-1)[:-1, :-1, :-1]
        lo = ndimage.minimum_filter(v, size=4, mode="nearest", origin=-1)[:-1, :-1, :-1]
    else:                   # flat indices im + (i-1) nyz + (r-1) nz + (k-1), 0 outside the array
        nx, ny, nz = v.shape
        nyz = ny * nz
        pad_lo, pad_hi = nyz + nz + 1, 2 * (nyz + nz + 1)
        flat = np.concatenate([np.zeros(pad_lo), v.ravel(), np.zeros(pad_hi)])
        hi, lo = flat, flat
        for step in (1, nz, nyz):
            hi, lo = _window(hi, step, np.maximum), _window(lo, step, np.minimum)
        hi = hi[pad_lo:pad_lo + v.size].reshape(v.shape)[:-1, :-1, :-1]
        lo = lo[pad_lo:pad_lo + v.size].reshape(v.shape)[:-1, :-1, :-1]
    return hi - lo, np.maximum(np.abs(hi), np.abs(lo))


# ---------------------------------------------------------------------------------------------------------------------
# A world: geometry, grids, atoms, scaling factors; oracle results, both tiers' scales
# ---------------------------------------------------------------------------------------------------------------------
class World:
    def __init__(self, counts, spacing, origin, grids, seed):
        self.counts, self.spacing, self.origin = tuple(counts), tuple(spacing), tuple(origin)
        self.grids = grids
        self.pos, self.shell = world_atoms(counts, spacing, origin, seed)
        self.n_replicas = self.pos.shape[0]
        rng = np.random.default_rng(seed + 1)
        g = len(grids)
        self.scaling = rng.uniform(0.5, 1.5, size=(g, N_ATOMS)) * rng.choice([-1.0, 1.0], size=(g, N_ATOMS))
        self.oob_k = cov.OOB_K[:g]
        flat = self.pos.reshape(-1, 3)
        inside, idx, _, alt_idx, _ = pw._classify(flat, counts, spacing, origin)
        ncell = tuple(int(n) - 1 for n in counts)
        self.inside = inside
        self.cell = np.ravel_multi_index(tuple(idx.T), ncell)
        self.alt_rows = np.nonzero((alt_idx != idx).any(axis=1))[0]
        self.alt_cells = []
        for combo in range(1, 8):
            use = np.array([(combo >> a) & 1 for a in range(3)], dtype=bool)
            ci = np.where(use, alt_idx[self.alt_rows], idx[self.alt_rows])
            self.alt_cells.append(np.ravel_multi_index(tuple(ci.T), ncell))
        del idx, alt_idx
        rel = flat - np.asarray(origin)
        hc = np.asarray(spacing) * (np.array(counts) - 1)
        self.dev = np.where(rel < 0.0, rel, np.where(rel > hc, rel - hc, 0.0))
        self.qsum = np.where(inside, (rel / np.asarray(spacing)).sum(axis=1), 0.0)
        del rel
        self.atom = np.tile(np.arange(N_ATOMS), self.n_replicas)
        shell_reps = np.unique(np.nonzero(self.shell)[0] // N_ATOMS)
        stride = max(1, self.n_replicas * N_ATOMS // EXACT_ATOMS)
        self.sub = np.union1d(shell_reps, np.arange(0, self.n_replicas, stride))
        self.sub_pos = np.ascontiguousarray(self.pos[self.sub])
        self._ref, self._ranges, self._exact = {}, {}, {}

    def case(self, method, ids, grids=None):
        ids = list(ids)
        return dict(counts=self.counts, spacing=self.spacing, origin=self.origin,
                    grids=[self.grids[g] for g in ids] if grids is None else grids, scaling=self.scaling[ids], pos=self.pos,
                    oob_k=[self.oob_k[g] for g in ids], inv_power=[0.0] * len(ids), method=method)

    def make(self, gf, dev, precision, layout, ids):
        grids = [gf.Grid(dev, self.counts, self.spacing, self.origin, self.grids[g], precision, layout=layout) for g in ids]
        assert all(g.layout == layout for g in grids)
        return grids, self.kernel(gf, dev, grids, ids)

    def kernel(self, gf, dev, grids, ids):
        return gf.Kernel(dev, grids, self.scaling[list(ids)], oob_k=[self.oob_k[g] for g in ids])

    # oracle -----------------------------------------------------------------------------------------------------------
    def _ref_grid(self, oracle, method, g):
        if (method, g) not in self._ref:
            c = self.case(method, (g,))
            ge, f = cov._oracle(oracle, c)
            self._ref[method, g] = (ge[:, 0], f, pw._oracle_atoms(oracle, c, self.pos))
        return self._ref[method, g]

    def reference(self, oracle, method, ids):
        """(per-replica energies [R], forces [R, A, 3], per-atom energies [R, A]): the oracle run per grid, summed."""
        parts = [self._ref_grid(oracle, method, g) for g in ids]
        return tuple(sum(p[i] for p in parts) for i in range(3))

    # exhaustive tier ----------------------------------------------------------------------------------------------------
    def _atom_ranges(self, method, g):
        """Per atom: (Rng, Mx) of its cell in grid g (the larger over the neighbouring cells a fraction within 1e-12 of 0 or 1
        may be evaluated in), 0 outside."""
        if (method, g) not in self._ranges:
            rng_c, mx_c = (a.ravel() for a in cell_ranges(method, self.grids[g]))
            out = []
            for per_cell in (rng_c, mx_c):
                a = per_cell[self.cell]
                for cells in self.alt_cells:
                    a[self.alt_rows] = np.maximum(a[self.alt_rows], per_cell[cells])
                a[~self.inside] = 0.0
                out.append(a)
            self._ranges[method, g] = tuple(out)
        return self._ranges[method, g]

    def exhaustive_scales(self, method, ids):
        """D, V [N] (to be divided by h_a), R [N, 3], E [N] (in units of TOL_E) of the exhaustive bound, N = R * 47 atoms."""
        cw, cdw = weight_bounds(method)
        n = self.atom.size
        s_rng, s_mx, R, Er = np.zeros(n), np.zeros(n), np.zeros((n, 3)), np.zeros(n)
        dev2 = (self.dev * self.dev).sum(axis=1)
        for g in ids:
            s = np.abs(self.scaling[g])[self.atom]
            rg, mx = self._atom_ranges(method, g)
            s_rng += s * rg
            s_mx += s * mx
            R += self.oob_k[g] * np.abs(self.dev)
            Er += 0.5 * self.oob_k[g] * dev2
        return dict(D=cdw * s_rng, V=cdw * s_mx, R=R, E=cw * s_mx + Er + FRAC_ROUNDING / pw.TOL_E * self.qsum * cdw * s_rng)

    # exact tier ---------------------------------------------------------------------------------------------------------
    def exact_scales(self, method, ids):
        """test_gpu_pointwise's force and energy scales on the sampled replicas, summed over the grids; the energy scales (per
        replica, per atom) with the fraction-rounding term in units of TOL_E."""
        for g in ids:
            if (method, g) not in self._exact:
                c = self.case(method, (g,))
                self._exact[method, g] = (pw.force_scale(c, self.sub_pos), pw.energy_scale(c, self.sub_pos))
        parts = [self._exact[method, g] for g in ids]
        fs = dict(parts[0][0])
        for key in ("D", "V", "R"):
            fs[key] = sum(p[0][key] for p in parts)
        frac = FRAC_ROUNDING / pw.TOL_E * ((fs["cell"] + fs["frac"]) * np.asarray(self.spacing) * fs["D"]).sum(axis=-1)
        return fs, sum(p[1][0] for p in parts) + frac.sum(axis=1), sum(p[1][1] for p in parts) + frac

    def describe(self, i):
        r, a = divmod(int(i), N_ATOMS)
        ncell = tuple(int(n) - 1 for n in self.counts)
        where = f"cell {np.unravel_index(self.cell[i], ncell)}" if self.inside[i] else "outside"
        return f"replica {r} atom {a} ({'shell' if self.shell[i] else 'every-cell'} atom, {where}, pos {tuple(self.pos[r, a])})"


# ---------------------------------------------------------------------------------------------------------------------
# Exhaustive-tier checks
# ---------------------------------------------------------------------------------------------------------------------
def _ratio(err, bound):
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(bound > 0.0, err / np.where(bound > 0.0, bound, 1.0), np.where(err > 0.0, np.inf, 0.0))
    return np.where(np.isnan(err), np.inf, r)


def exhaustive_force_ratio(f, f_ref, sc, spacing, tol_f, tol_d, tol_v, fixed_adds=0):
    """Per atom [N]: the largest err / bound over its three components (inf for a NaN)."""
    f = np.asarray(f, dtype=np.float64).reshape(-1, 3)
    f_ref = f_ref.reshape(-1, 3)
    bound = (tol_f * np.maximum(np.abs(f_ref), sc["R"]) + (tol_d * sc["D"] + tol_v * sc["V"])[:, None] / np.asarray(spacing)
             + fixed_adds * pw.FIXED_QUANTUM)
    return _ratio(np.abs(f - f_ref), bound).max(axis=1)


def exhaustive_energy_ratio(e, e_ref, sc, per_atom):
    """Per atom [N] or per replica [R]: err / (TOL_E * scale)."""
    scale = sc["E"] if per_atom else sc["E"].reshape(-1, N_ATOMS).sum(axis=1)
    e = np.asarray(e, dtype=np.float64).ravel()
    return _ratio(np.abs(e - e_ref.ravel()), pw.TOL_E * scale)


def _assert_ratio(w, ratio, what, per_replica=False):
    i = int(np.argmax(ratio))
    worst = float(ratio[i])
    where = f"replica {i}" if per_replica else w.describe(i)
    assert worst <= 1.0, f"{what}: {worst:.3g}x the exhaustive bound at {where}; {int((ratio > 1.0).sum())} over"
    return worst


def _report(what, **ratios):
    print(f"PRODUCTION {what}: " + " ".join(f"{k}={v:.3g}" for k, v in ratios.items()))


def check_both_tiers(w, oracle, method, ids, tol, what, en, forces=None, atom_e=None, fixed_adds=0):
    """en [R], forces [R, A, 3], atom_e [R, A] against the oracle: every atom (exhaustive tier) and the sampled replicas
    (exact tier). Prints and returns the worst ratio of each check."""
    e_ref, f_ref, ae_ref = w.reference(oracle, method, ids)
    sc = w.exhaustive_scales(method, ids)
    out = {}
    if forces is not None:
        assert np.isfinite(forces).all(), f"{what}: non-finite forces"
        out["force"] = _assert_ratio(w, exhaustive_force_ratio(forces, f_ref, sc, w.spacing, **tol, fixed_adds=fixed_adds), what)
    out["energy"] = _assert_ratio(w, exhaustive_energy_ratio(en, e_ref, sc, False), what + " energy", per_replica=True)
    if atom_e is not None:
        out["atom"] = _assert_ratio(w, exhaustive_energy_ratio(atom_e, ae_ref, sc, True), what + " atom energy")
    fs, e_rep, e_atom = w.exact_scales(method, ids)
    sub = w.sub
    if forces is not None:
        out["exact_force"] = pw.check_forces(np.asarray(forces)[sub], f_ref[sub], fs, **tol, fixed_adds=fixed_adds,
                                             what=what + " (exact tier)")
    out["exact_energy"] = pw.check_energies(np.asarray(en)[sub], e_ref[sub], e_rep, pw.TOL_E, what + " (exact tier)")
    if atom_e is not None:
        out["exact_atom"] = pw.check_energies(np.asarray(atom_e)[sub], ae_ref[sub], e_atom, pw.TOL_E, what + " atom (exact tier)")
    _report(what, **out)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# CPU self-tests
# ---------------------------------------------------------------------------------------------------------------------
SMALL = [((9, 8, 11), (0.05, 0.07, 0.04), (0.0, 0.0, 0.0)), ((21, 18, 25), T_SPACING, T_ORIGIN)]


def _faces_hit(pos, counts, sp, og):
    """Per atom and axis: -1 on the lower face, +1 on the upper face, 0 strictly inside, 9 outside."""
    rel = pos - np.asarray(og)
    hc = np.asarray(sp) * (np.array(counts) - 1)
    state = np.where(rel == 0.0, -1, np.where(rel == hc, 1, 0))
    return np.where((rel < 0.0) | (rel > hc), 9, state)


@pytest.mark.parametrize("geom", SMALL, ids=["small", "t-spacing"])
def test_positions_visit_every_cell_once(geom):
    counts, sp, og = geom
    pos, shell = world_atoms(counts, sp, og, seed=5)
    assert pos.shape[1] == N_ATOMS and shell.size == pos.shape[0] * N_ATOMS
    flat = pos.reshape(-1, 3)
    ncell = tuple(n - 1 for n in counts)
    inside, idx, _, _, _ = pw._classify(flat[~shell], counts, sp, og)
    assert inside.all()
    assert np.array_equal(np.sort(np.ravel_multi_index(tuple(idx.T), ncell)), np.arange(int(np.prod(ncell))))
    # the permutation spreads both kinds of atoms over the replicas
    assert not np.array_equal(np.nonzero(shell)[0], np.arange(shell.sum()) + (~shell).sum())
    state = _faces_hit(flat[shell], counts, sp, og)
    on = (state == -1) | (state == 1)
    inner = state == 0
    for n_on in (1, 2, 3):                 # faces, edges, corners
        for axes in itertools.combinations(range(3), n_on):
            free = [a for a in range(3) if a not in axes]
            for sides in itertools.product((-1, 1), repeat=n_on):
                hit = inner[:, free].all(axis=1) & on[:, list(axes)].all(axis=1) & (state[:, list(axes)] == np.array(sides)).all(axis=1)
                assert hit.any(), (axes, sides)
    # 1 ulp outside and deeper outside every face
    out = state == 9
    for a in range(3):
        rel = flat[shell][:, a] - og[a]
        hc = sp[a] * (counts[a] - 1)
        assert (out[:, a] & (rel < 0.0) & (rel > -1e-12)).any() and (out[:, a] & (rel > hc) & (rel < hc + 1e-12)).any()
        assert (rel < -1.0).any() and (rel > hc + 1.0).any()


@pytest.mark.parametrize("method", [0, 1, 2], ids=["trilinear", "bspline", "tricubic"])
def test_weight_bounds_hold(method):
    """No sampled fraction in any xin/yin/zin case exceeds C_w or C_dw."""
    cw, cdw = weight_bounds(method)
    rng = np.random.default_rng(11 + method)
    counts = (4, 4, 4)
    for cell in itertools.product((0, 1), repeat=3):
        f = rng.uniform(0.0, 1.0, size=(20_000, 3))
        f[:8] = np.array(list(itertools.product((0.0, 1.0), repeat=3)))
        idx = np.broadcast_to(np.array(cell), f.shape).copy()
        _, w, dw, _ = pw._stencil(method, np.zeros(counts), counts, idx, f)
        assert np.abs(w).sum(axis=1).max() <= cw and np.abs(dw).sum(axis=1).max() <= cdw
    if method == 0:
        assert 2.0 <= cdw <= 2.1 and 1.0 <= cw <= 1.03


def _stencil_points(method, counts, idx):
    """Flat point index [N, K] of each stencil position of pw._stencil (same order), -1 for a zero read past the array."""
    n = np.array(counts)
    ny, nz = n[1], n[2]
    if method == 0:
        pts = list(itertools.product((0, 1), repeat=3))
        return np.stack([((idx[:, 0] + a) * ny + idx[:, 1] + b) * nz + idx[:, 2] + c for a, b, c in pts], 1)
    pts = list(itertools.product(range(4), repeat=3))
    if method == 1:
        ix = [np.clip(idx[:, a, None] - 1 + np.arange(4), 0, n[a] - 1) for a in range(3)]
        return np.stack([(ix[0][:, i] * ny + ix[1][:, j]) * nz + ix[2][:, k] for i, j, k in pts], 1)
    im = (idx[:, 0] * ny + idx[:, 1]) * nz + idx[:, 2]
    fi = np.stack([im + (i - 1) * ny * nz + (r - 1) * nz + (k - 1) for i, r, k in pts], 1)
    return np.where((fi >= 0) & (fi < int(np.prod(n))), fi, -1)


@pytest.mark.parametrize("method", [0, 1, 2], ids=["trilinear", "bspline", "tricubic"])
def test_exhaustive_bound_holds_for_the_oracle_and_catches_a_swap(oracle_built, method):
    """The oracle passes against itself with ratio 0; the oracle on a copy of the grid with two corners of the last cell in
    memory order swapped fails on exactly the atoms whose energy or force depends on the swap."""
    counts, sp, og = SMALL[0]
    rng = np.random.default_rng(20 + method)
    vals = (rng.normal(size=counts) * 4).astype(np.float32).astype(np.float64)
    p1, p2 = tuple(n - 2 for n in counts), tuple(n - 1 for n in counts)      # corners 000 and 111 of the last cell
    vals[p1], vals[p2] = 10.0, -10.0
    w = World(counts, sp, og, [vals], seed=30 + method)
    tol = pw._tol(0, method, 1, path=0)
    e_ref, f_ref, ae_ref = w.reference(oracle_built, method, (0,))
    sc = w.exhaustive_scales(method, (0,))
    assert exhaustive_force_ratio(f_ref, f_ref, sc, sp, **tol).max() == 0.0
    assert exhaustive_energy_ratio(ae_ref, ae_ref, sc, True).max() == 0.0
    assert exhaustive_energy_ratio(e_ref, e_ref, sc, False).max() == 0.0
    assert (sc["D"][w.inside] > 0).all()

    swapped = vals.copy()
    swapped[p1], swapped[p2] = vals[p2], vals[p1]
    c = w.case(method, (0,), grids=[swapped])
    _, f_bad = cov._oracle(oracle_built, c)
    ae_bad = pw._oracle_atoms(oracle_built, c, w.pos)
    fails = (exhaustive_force_ratio(f_bad, f_ref, sc, sp, **tol) > 1.0) | (exhaustive_energy_ratio(ae_bad, ae_ref, sc, True) > 1.0)

    # what the swap changes for each atom: (W(p1) - W(p2)) * (v1 - v2), W the summed weights of a point's stencil positions
    flat = w.pos.reshape(-1, 3)
    inside, idx, f, _, _ = pw._classify(flat, counts, sp, og)
    _, wt, dwt, _ = pw._stencil(method, vals, counts, idx, f)
    pts = _stencil_points(method, counts, idx)
    i1, i2 = np.ravel_multi_index(p1, counts), np.ravel_multi_index(p2, counts)
    dw_e = ((pts == i1) * wt).sum(axis=1) - ((pts == i2) * wt).sum(axis=1)
    dw_f = ((pts == i1)[..., None] * dwt).sum(axis=1) - ((pts == i2)[..., None] * dwt).sum(axis=1)
    depends = inside & ((np.abs(dw_e) > 1e-12) | (np.abs(dw_f) > 1e-12).any(axis=1))
    assert depends.sum() >= 3 and (~depends).sum() > 0
    assert np.array_equal(fails, depends), (np.nonzero(fails & ~depends)[0], np.nonzero(depends & ~fails)[0])


# ---------------------------------------------------------------------------------------------------------------------
# GPU: world T (trilinear)
# ---------------------------------------------------------------------------------------------------------------------
def _fp32(v):
    return v.astype(np.float32).astype(np.float64)


@pytest.fixture(scope="module")
def world_t():
    return World(T_COUNTS, T_SPACING, T_ORIGIN, [_fp32(W.synthetic_grid(T_COUNTS, T_SPACING, seed=W.SEED + 20 + g)) for g in range(4)],
                 seed=2026)


@pytest.fixture(scope="module")
def world_s():
    rng = np.random.default_rng(77)
    return World(S_COUNTS, S_SPACING, S_ORIGIN, [_fp32(W.synthetic_grid(S_COUNTS, S_SPACING, seed=W.SEED + 30 + g, wavelength=0.3 + 0.1 * g)
                                                       + 0.5 * rng.normal(size=S_COUNTS)) for g in range(2)], seed=2027)


@pytest.fixture(scope="module")
def t_mixed_cells(gpu_device, world_t):
    """World T's four MIXED CELLS grids, built once: the 1-, 3- and 4-grid kernels share them, so that no grid is rebuilt
    from the same values into memory its previous copy just freed."""
    import openmmgridforce_b200 as gf
    grids = [gf.Grid(gpu_device, world_t.counts, world_t.spacing, world_t.origin, v, gf.PRECISION_MIXED, layout=CELLS) for v in world_t.grids]
    yield grids
    for g in grids:
        g.close()


def _host_run(gf, k, w, want_forces=True):
    """execute_host (F64_STORE) of every replica with per-atom energies: (energies, forces or None, atom energies)."""
    k.request_atom_energies(True)
    en, forces, _ = k.execute_host(w.pos, want_forces=want_forces)
    ae = k.atom_energies(w.n_replicas)
    k.request_atom_energies(False)
    return en, forces, ae


@pytest.mark.gpu
@pytest.mark.parametrize("n_grids", [1, 3, 4])
def test_world_t_mixed_cells(gpu_device, oracle_built, world_t, t_mixed_cells, n_grids):
    """The lines kernel (path 1) on every cell: one grid (also one device FIXED_ADD launch), 3 and 4 grids through the
    interleaved 128-byte records (3 grids: also energy only, compared with the forces run)."""
    import torch
    import openmmgridforce_b200 as gf
    w, ids = world_t, tuple(range(n_grids))
    k = w.kernel(gf, gpu_device, t_mixed_cells[:n_grids], ids)
    try:
        assert k.eval_path() == 1
        tol = pw._tol(0, 0, n_grids, path=1)
        what = f"T mixed-cells{n_grids}"
        en, forces, ae = _host_run(gf, k, w)
        check_both_tiers(w, oracle_built, 0, ids, tol, what, en, forces, ae)
        del forces
        if n_grids == 1:
            e_dev, f_dev = pw._device_fixed(gf, k, dict(pos=w.pos), 1, torch.cuda.Stream())
            check_both_tiers(w, oracle_built, 0, ids, tol, what + " device fixed", e_dev, f_dev, fixed_adds=1)
        if n_grids == 3:
            e0, none, ae0 = _host_run(gf, k, w, want_forces=False)
            assert none is None
            check_both_tiers(w, oracle_built, 0, ids, tol, what + " energy-only", e0, atom_e=ae0)
            ratio = exhaustive_energy_ratio(e0, en, w.exhaustive_scales(0, ids), False)
            _report(what + " energy-only vs forces run", energy=_assert_ratio(w, ratio, "energy-only vs forces run", per_replica=True))
    finally:
        k.close()


T_CASES = [("double-cells3", 1, CELLS, (0, 1, 2), 2), ("double-cells1", 1, CELLS, (3,), 0), ("mixed-rows3", 0, ROWS, (0, 1, 2), 0),
           ("mixed-pairs3", 0, PAIRS, (0, 1, 2), 0), ("double-rows3", 1, ROWS, (0, 1, 2), 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("spec", T_CASES, ids=[s[0] for s in T_CASES])
def test_world_t_layouts(gpu_device, oracle_built, world_t, spec):
    """DOUBLE 256-byte records (path 2; 3.14 GiB, records above the 2 GiB offset; also energy only), DOUBLE CELLS on one
    grid and the ROWS / PAIRS layouts (general kernel), every cell of world T. The one-grid DOUBLE case uses grid 3, so
    that no layout is rebuilt from the values it held just before."""
    import openmmgridforce_b200 as gf
    name, precision, layout, ids, path = spec
    w = world_t
    grids, k = w.make(gf, gpu_device, precision, layout, ids)
    try:
        assert k.eval_path() == path
        tol = pw._tol(precision, 0, len(ids), path=path)
        en, forces, ae = _host_run(gf, k, w)
        check_both_tiers(w, oracle_built, 0, ids, tol, f"T {name}", en, forces, ae)
        del forces
        if path == 2:
            e0, none, ae0 = _host_run(gf, k, w, want_forces=False)
            assert none is None
            check_both_tiers(w, oracle_built, 0, ids, tol, f"T {name} energy-only", e0, atom_e=ae0)
            ratio = exhaustive_energy_ratio(e0, en, w.exhaustive_scales(0, ids), False)
            _report(f"T {name} energy-only vs forces run", energy=_assert_ratio(w, ratio, "energy-only vs forces run", per_replica=True))
    finally:
        cov._close(grids, k)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: world S (B-spline and tricubic)
# ---------------------------------------------------------------------------------------------------------------------
S_CASES = [("mixed-bspline", 0, BSPLINE, 3), ("double-bspline", 1, BSPLINE, 4), ("mixed-hermite", 0, HERMITE, 5),
           ("double-hermite", 1, HERMITE, 6), ("mixed-bspline_points", 0, BSPLINE_POINTS, 0),
           ("double-bspline_points", 1, BSPLINE_POINTS, 0), ("mixed-points", 0, POINTS, 0), ("double-points", 1, POINTS, 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("spec", S_CASES, ids=[s[0] for s in S_CASES])
def test_world_s_layouts(gpu_device, oracle_built, world_s, spec):
    """The B-spline and tricubic record kernels (paths 3-6; 47 repack passes) and the point layouts through the general
    kernel (6 repack passes), two grids, every cell of world S."""
    import openmmgridforce_b200 as gf
    name, precision, layout, path = spec
    w, ids, method = world_s, (0, 1), METHOD[layout]
    grids, k = w.make(gf, gpu_device, precision, layout, ids)
    try:
        assert k.eval_path() == path
        en, forces, ae = _host_run(gf, k, w)
        check_both_tiers(w, oracle_built, method, ids, pw._tol(precision, method, 2, path=path), f"S {name}", en, forces, ae)
    finally:
        cov._close(grids, k)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the benchmark's method-1/2 configurations
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("layout", [BSPLINE, HERMITE], ids=["C5_bspline", "C5_tricubic"])
def test_bench_c5_records(gpu_device, oracle_built, layout):
    """bench.py's C5_bspline / C5_tricubic state (3 grids of 192^3, not FP32-representable, MIXED records) on 2 048
    replicas of the C5 poses, exact tier, with the storage rounding 2^-24 |v| per point in tol_v and TOL_E_STORAGE."""
    import openmmgridforce_b200 as gf
    w = W.c5_sharded_replicas(n_local=2048)
    method = METHOD[layout]
    c = dict(counts=w.counts, spacing=w.spacing, origin=w.origin, grids=w.grids, scaling=w.scaling, pos=w.pos, oob_k=w.oob_k,
             inv_power=w.inv_power, method=method)
    grids, k = cov._make(gf, gpu_device, c, gf.PRECISION_MIXED, layout)
    try:
        assert k.eval_path() == (3 if layout == BSPLINE else 5)
        k.request_atom_energies(True)
        en, forces, _ = k.execute_host(w.pos)
        ae = k.atom_energies(w.n_replicas)
    finally:
        cov._close(grids, k)
    ge_ref, f_ref = cov._oracle(oracle_built, c)
    ae_ref = pw._oracle_atoms(oracle_built, c, w.pos)
    tol = pw._tol(0, method, 3, path=3)
    tol["tol_v"] += U
    e_rep, e_atom = pw.energy_scale(c, w.pos)
    what = f"C5 {'bspline' if layout == BSPLINE else 'tricubic'}"
    _report(what, force=pw.check_forces(forces, f_ref, pw.force_scale(c, w.pos), **tol, what=what),
            energy=pw.check_energies(en, ge_ref.sum(axis=1), e_rep, pw.TOL_E_STORAGE, what),
            atom=pw.check_energies(ae, ae_ref, e_atom, pw.TOL_E_STORAGE, what + " atom"))


# ---------------------------------------------------------------------------------------------------------------------
# GPU: grid-construction routes, against a Grid built from host memory
# ---------------------------------------------------------------------------------------------------------------------
ROUTE_LAYOUTS = [(0, CELLS, 1), (1, CELLS, 0), (0, BSPLINE, 3)]
ROUTE_IDS = ["mixed-cells", "double-cells", "mixed-bspline"]


def _assert_identical(gf, dev, pos, scaling, g_route, g_host, path, what):
    """Per-atom forces and per-atom energies bit-identical, per-replica energies within 1e-13 (FP64 atomics of two warps
    may land in either order)."""
    out = []
    for g in (g_route, g_host):
        k = gf.Kernel(dev, [g], scaling, oob_k=[10000.0])
        try:
            assert k.eval_path() == path
            k.request_atom_energies(True)
            en, f, _ = k.execute_host(pos)
            out.append((en, f, k.atom_energies(pos.shape[0])))
        finally:
            k.close()
    (en_a, f_a, ae_a), (en_b, f_b, ae_b) = out
    assert np.isfinite(f_b).all() and np.abs(f_b).max() > 0.0
    diff = (f_a != f_b).any(axis=-1)
    assert not diff.any(), f"{what}: forces of {int(diff.sum())} atoms differ, first at {np.argwhere(diff)[0]}"
    diff = ae_a != ae_b
    assert not diff.any(), f"{what}: energies of {int(diff.sum())} atoms differ, first at {np.argwhere(diff)[0]}"
    assert (np.abs(en_a - en_b) <= 1e-13 * np.abs(ae_b).sum(axis=1)).all(), what


@pytest.fixture(scope="module")
def t_grid_file(tmp_path_factory, world_t):
    """World T's grid 0 as a V3 file: 13 357 344 doubles, 3.18 pieces of 4 194 304."""
    import openmmgridforce_b200 as gf
    path = str(tmp_path_factory.mktemp("grids") / "world_t_grid0.grid")
    gf.write_grid_file(path, world_t.counts, world_t.spacing, world_t.origin, world_t.grids[0])
    return path


def _check_header(g, counts, sp, og):
    assert g.header["counts"] == tuple(counts)
    assert g.header["spacing"] == tuple(sp) and g.header["origin"] == tuple(og)
    assert g.counts == tuple(counts) and g.spacing == tuple(sp) and g.origin == tuple(og)


@pytest.mark.gpu
@pytest.mark.parametrize("spec", ROUTE_LAYOUTS, ids=ROUTE_IDS)
def test_route_file(gpu_device, world_t, t_grid_file, spec):
    """Grid.from_file (two alternating pinned 32 MB buffers, four pieces, the last partial) against Grid from host values,
    every cell of world T. The file grid is built first, so that its staging buffer cannot inherit the host build's."""
    import openmmgridforce_b200 as gf
    precision, layout, path = spec
    w = world_t
    g_file = gf.Grid.from_file(gpu_device, t_grid_file, precision, layout)
    try:
        _check_header(g_file, w.counts, w.spacing, w.origin)
        assert g_file.layout == layout
        g_host = gf.Grid(gpu_device, w.counts, w.spacing, w.origin, w.grids[0], precision, layout=layout)
        try:
            _assert_identical(gf, gpu_device, w.pos, w.scaling[:1], g_file, g_host, path, f"file {spec}")
        finally:
            g_host.close()
    finally:
        g_file.close()
    if spec == ROUTE_LAYOUTS[0]:
        header, vals = gf.read_grid_file(t_grid_file)
        assert header["counts"] == w.counts and np.array_equal(vals, w.grids[0])


PIECE_FILES = [("two-pieces", (128, 128, 512)), ("one-piece-plus-4", (2, 2, 1_048_577))]


@pytest.mark.gpu
@pytest.mark.parametrize("name,counts", PIECE_FILES, ids=[p[0] for p in PIECE_FILES])
def test_route_file_piece_boundaries(gpu_device, tmp_path, name, counts):
    """Files of exactly 2 pieces (8 388 608 doubles) and of one piece + 4 values, MIXED CELLS, one atom in every cell."""
    import openmmgridforce_b200 as gf
    assert int(np.prod(counts)) in (2 << 22, (4 << 20) + 4)
    rng = np.random.default_rng(int(np.prod(counts)) % 1000)
    sp, og = (0.011, 0.013, 0.0007), (0.0, 0.0, 0.0)
    vals = _fp32(rng.normal(size=counts) * 4)
    path = str(tmp_path / f"{name}.grid")
    gf.write_grid_file(path, counts, sp, og, vals)
    pos, _ = world_atoms(counts, sp, og, seed=9)
    scaling = rng.uniform(0.5, 1.5, size=(1, N_ATOMS))
    g_file = gf.Grid.from_file(gpu_device, path, gf.PRECISION_MIXED, CELLS)
    try:
        _check_header(g_file, counts, sp, og)
        g_host = gf.Grid(gpu_device, counts, sp, og, vals, gf.PRECISION_MIXED, layout=CELLS)
        try:
            _assert_identical(gf, gpu_device, pos, scaling, g_file, g_host, 1, f"file {name}")
        finally:
            g_host.close()
    finally:
        g_file.close()


@pytest.mark.gpu
@pytest.mark.parametrize("spec", ROUTE_LAYOUTS, ids=ROUTE_IDS)
def test_route_device_pointer(gpu_device, world_t, spec):
    """Grid(..., device_ptr=...) (gfb_grid_create_from_device) from a torch tensor; the tensor is left unchanged."""
    import torch
    import openmmgridforce_b200 as gf
    precision, layout, path = spec
    w = world_t
    t = torch.from_numpy(w.grids[0].ravel()).to("cuda:0")
    torch.cuda.synchronize()
    g_dev = gf.Grid(gpu_device, w.counts, w.spacing, w.origin, None, precision, layout=layout, device_ptr=t.data_ptr())
    try:
        assert np.array_equal(t.cpu().numpy(), w.grids[0].ravel())
        g_host = gf.Grid(gpu_device, w.counts, w.spacing, w.origin, w.grids[0], precision, layout=layout)
        try:
            _assert_identical(gf, gpu_device, w.pos, w.scaling[:1], g_dev, g_host, path, f"device pointer {spec}")
        finally:
            g_host.close()
    finally:
        g_dev.close()
    del t


def _ulps(a, b):
    """|a - b| in units in the last place of same-signed doubles."""
    ia, ib = a.view(np.int64), b.view(np.int64)
    return np.abs(ia - ib)


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["host", "device"])
def test_inv_power_transform_production_size(gpu_device, oracle_built, form):
    """Device.inv_power_transform on 13 357 344 values (11 grid-stride passes on a B200): mixed signs, zeros (both signs)
    and magnitudes over 10 decades, within 2 ulp of the C oracle; zeros and signs preserved."""
    import torch
    rng = np.random.default_rng(404)
    n = int(np.prod(T_COUNTS))
    v = rng.choice([-1.0, 1.0], size=n) * 10.0 ** rng.uniform(-5.0, 5.0, size=n)
    zero = rng.uniform(size=n) < 0.05
    v[zero] = 0.0
    v[np.nonzero(zero)[0][::2]] = -0.0
    inv_power = 4.0 if form == "host" else 3.0
    want = oracle_built.port_inv_power_transform(v, inv_power)
    if form == "host":
        got = gpu_device.inv_power_transform(v, inv_power)
    else:
        t = torch.from_numpy(v).to("cuda:0")
        torch.cuda.synchronize()
        gpu_device.inv_power_transform(None, inv_power, device_ptr=t.data_ptr(), n=t.numel())
        got = t.cpu().numpy()
        del t
    assert np.array_equal(got[zero].view(np.int64), v[zero].view(np.int64))
    assert np.array_equal(np.signbit(got), np.signbit(v)) and (got[~zero] != 0.0).all()
    ulps = _ulps(got, want)
    worst = int(ulps.max())
    assert worst <= 2, f"{int((ulps > 2).sum())} values more than 2 ulp from the oracle, first at {int(np.argmax(ulps > 2))}"
    _report(f"inv-power {form}", max_ulp=worst)
