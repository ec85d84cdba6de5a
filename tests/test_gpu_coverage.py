"""GPU parity tests (-m gpu) of the dispatch paths and modes the other GPU test files reach in one or two of their
instantiations, each against the C oracle (oracle/gridforce_oracle.c, bit-exact with the reference's
ReferenceCalcGridForceKernel) on the same inputs:

  A. offset fields V = C + noise (|C| up to 1e4, noise amplitude 1): the FP32 gradient arithmetic of the MIXED kernels must
     lose precision in proportion to |grad V|, not to |V|, in every path that evaluates one grid's gradient in FP32;
  B. the record kernels (eval paths 3-6: B-spline and tricubic, MIXED and DOUBLE) in every force mode, 1-4 grids, ragged
     totals, edge cells and upper faces, and thin grids;
  C. the device path, particle subsets, interleaved energy slots, per-atom energies and inv-power on the record kernels;
  D. 5 and 8 grids, grids of mixed geometry, inv-power on one grid of several, update_parameters moving a state between
     paths, and energy slots that own no atoms (read 0; the launch clears every entry of the next accumulator).

Every grid is FP32-representable, so a MIXED failure is arithmetic and not storage rounding. Tolerances (BASELINE.json
north_star): MIXED energies 1e-6 per replica, forces 1e-5 relative (max-norm); DOUBLE 1e-12; MIXED tricubic (FP64
arithmetic on FP32-stored points) 1e-10. Every case asserts gfb_kernel_eval_path, so that a dispatch change cannot move a
test onto another kernel unnoticed.
"""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import cases  # noqa: E402

pytestmark = pytest.mark.gpu

CELLS, ROWS, PAIRS, BSPLINE, POINTS, HERMITE, BSPLINE_POINTS = 1, 2, 3, 4, 5, 6, 7
METHOD = {CELLS: 0, ROWS: 0, PAIRS: 0, BSPLINE: 1, BSPLINE_POINTS: 1, HERMITE: 2, POINTS: 2}
COUNTS, SPACING, ORIGIN = (23, 19, 31), (0.05, 0.07, 0.04), (0.3, -0.2, 1.0)
OOB_K = [10000.0, 1234.0, 777.0, 5000.0, 300.0, 2000.0, 4321.0, 9000.0]
N_THREADS = min(8, os.cpu_count() or 1)


def _tol(precision, method):
    if precision == 1:
        return 1e-12, 1e-12
    return (1e-10, 1e-10) if method == 2 else (1e-6, 1e-5)


def _path(precision, layout, n_grids, lines_ok=True):
    """gfb_kernel_eval_path of a one-geometry state (lines_ok=False: inv-power on some grid)."""
    if layout == CELLS and lines_ok:
        if precision == 0 and n_grids <= 4:
            return 1
        if precision == 1 and 2 <= n_grids <= 4:
            return 2
    if layout == BSPLINE:
        return 3 if precision == 0 else 4
    if layout == HERMITE:
        return 5 if precision == 0 else 6
    return 0


def _edges(pos, counts, sp, og, method, rng):
    """Moves about a third of the atoms into the first and last cells of every axis and onto the upper faces (the corner
    included). Method 2 then gets the reference's undefined places moved inside (cases._tricubic_safe)."""
    flat = pos.reshape(-1, 3)
    n = flat.shape[0]
    sp, og = np.array(sp), np.array(og)
    length = sp * (np.array(counts) - 1)
    idx = rng.permutation(n)
    k = max(1, n // 10)
    first, last, face = idx[:k], idx[k:2 * k], idx[2 * k:3 * k]
    flat[first] = og + rng.uniform(0.0, 1.0, size=(len(first), 3)) * sp
    flat[last] = og + length - rng.uniform(1e-6, 1.0, size=(len(last), 3)) * sp
    for j, i in enumerate(face):
        flat[i, j % 3] = og[j % 3] + length[j % 3]
    flat[idx[0]] = og + length
    if method == 2:
        cases._tricubic_safe(dict(counts=counts, spacing=tuple(sp), origin=tuple(og), pos=flat), rng)
    return pos


def _case(n_grids, n_replicas, n_atoms, seed, method=0, counts=COUNTS, sp=SPACING, og=ORIGIN, offset=0.0, amp=4.0,
          frac_outside=0.08, out_depth=0.3, edges=False):
    """test_gpu_lines._case's recipe: random anisotropic FP32-representable grids (offset + amp * noise), replicas scattered
    over the box with a few atoms outside, scaling factors zero on every 7th atom and on one grid only for atom 3."""
    rng = np.random.default_rng(seed)
    grids = [(offset + rng.normal(size=counts) * amp).astype(np.float32).astype(np.float64) for _ in range(n_grids)]
    length = np.array(sp) * (np.array(counts) - 1)
    pos = np.array(og) + rng.uniform(0.0, 1.0, size=(n_replicas, n_atoms, 3)) * length
    if edges:
        _edges(pos, counts, sp, og, method, rng)
    out = rng.uniform(size=(n_replicas, n_atoms)) < frac_outside
    pos[out] += rng.choice([-1.0, 1.0], size=(int(out.sum()), 3)) * rng.uniform(0.0, out_depth, size=(int(out.sum()), 3)) * length
    sc = rng.normal(size=(n_grids, n_atoms))
    sc[:, ::7] = 0.0
    if n_grids > 1 and n_atoms > 3:
        sc[1, 3] = 0.0
    return dict(counts=counts, spacing=sp, origin=og, grids=grids, scaling=sc, pos=pos, oob_k=OOB_K[:n_grids],
                inv_power=[0.0] * n_grids, method=method)


def _port(oracle, c, scaling=None, method=None):
    return oracle.PortOracle(c["counts"], c["spacing"], c["origin"], c["grids"], c["scaling"] if scaling is None else scaling,
                             oob_k=c["oob_k"], inv_power=c["inv_power"],
                             interpolation_method=c["method"] if method is None else method)


def _oracle(oracle, c, pos=None, scaling=None):
    return _port(oracle, c, scaling).execute_batched(c["pos"] if pos is None else pos, n_threads=N_THREADS)


def _make(gf, dev, c, precision, layout, particles=None):
    grids = [gf.Grid(dev, c["counts"], c["spacing"], c["origin"], g, precision, layout=layout) for g in c["grids"]]
    assert all(g.layout == layout for g in grids)
    k = gf.Kernel(dev, grids, c["scaling"], particles=particles, inv_power=c["inv_power"], oob_k=c["oob_k"])
    return grids, k


def _close(grids, k):
    k.close()
    for g in grids:
        g.close()


def _err_f(f, ref):
    return np.abs(f - ref).max() / max(np.abs(ref).max(), 1e-300)


def _check(en, ge, forces, ge_ref, f_ref, te, tf, what=""):
    """Per replica: |E - E_ref| <= te * max(|E_ref|, largest per-grid term of that replica); forces max-norm relative."""
    term = np.abs(ge_ref).max(axis=1)
    if ge is not None:
        assert (np.abs(ge - ge_ref) <= te * np.maximum(np.abs(ge_ref), term[:, None])).all(), what
    e_ref = ge_ref.sum(axis=1)
    assert (np.abs(en - e_ref) <= te * np.maximum(np.abs(e_ref), term)).all(), what
    if forces is not None:
        err = _err_f(forces, f_ref)
        assert err <= tf, f"{what}: force error {err:.3e} of max|F| (bound {tf:g})"


# ---------------------------------------------------------------------------------------------------------------------
# A. Offset fields
# ---------------------------------------------------------------------------------------------------------------------
# (name, precision, layout, n_grids)
OFFSET_PATHS = [
    ("mixed-lines1", 0, CELLS, 1), ("mixed-lines3", 0, CELLS, 3), ("mixed-cells5", 0, CELLS, 5), ("mixed-rows", 0, ROWS, 1),
    ("mixed-pairs", 0, PAIRS, 1), ("mixed-bspline", 0, BSPLINE, 1), ("mixed-bspline-points", 0, BSPLINE_POINTS, 1),
    ("mixed-hermite", 0, HERMITE, 1),
    ("double-cells1", 1, CELLS, 1), ("double-cells3", 1, CELLS, 3), ("double-rows", 1, ROWS, 1), ("double-bspline", 1, BSPLINE, 1),
    ("double-bspline-points", 1, BSPLINE_POINTS, 1), ("double-hermite", 1, HERMITE, 1),
]
OFFSETS = [0.0, 1e2, -1e2, 1e3, -1e3, 1e4, -1e4]
# DOUBLE stops at |C| = 1e3: the reference's own FP64 gradient (vp - vm, and the B-spline derivative sums over values of
# size |V|) rounds at 1.1e-16 |V|, which at |C| = 1e4 is ~1e-12 of max|F| on this field, so the oracle itself is no
# longer good to the 1e-12 bound there (measured on a B200: kernel against oracle 1.1e-12 to 2.5e-12 at |C| = 1e4).
OFFSET_CASES = [(spec, o) for spec in OFFSET_PATHS for o in OFFSETS if spec[1] == 0 or abs(o) <= 1e3]


def _offset_case(n_grids, r, a, offset, method, seed):
    """V = C + noise of amplitude 1, isotropic spacing 0.05; atoms inside, in edge cells, on the upper faces and just
    outside (a shallow wall, so that restraint forces do not dwarf the interpolated ones in max|F|)."""
    return _case(n_grids, r, a, seed, method=method, sp=(0.05, 0.05, 0.05), offset=offset, amp=1.0, out_depth=0.01, edges=True)


@pytest.mark.parametrize("spec,offset", OFFSET_CASES, ids=[f"{s[0]}-{o:g}" for s, o in OFFSET_CASES])
def test_offset_field(gpu_device, oracle_built, spec, offset):
    import openmmgridforce_b200 as gf
    name, precision, layout, n_grids = spec
    method = METHOD[layout]
    c = _offset_case(n_grids, 7, 300, offset, method, seed=len(name) * 31 + int(abs(offset)) % 97 + (offset < 0))
    ge_ref, f_ref = _oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, precision, layout)
    assert k.eval_path() == _path(precision, layout, n_grids)
    te, tf = _tol(precision, method)
    en, forces, ge = k.execute_host(c["pos"], want_grid_energies=True)
    _check(en, ge, forces, ge_ref, f_ref, te, tf, f"{name} C={offset:g}")
    _close(grids, k)


RESIDENT_CASES = [(p, o) for p in (0, 1) for o in OFFSETS if p == 0 or abs(o) <= 1e3]


@pytest.mark.parametrize("precision,offset", RESIDENT_CASES, ids=[f"{'mixed' if p == 0 else 'double'}-{o:g}" for p, o in RESIDENT_CASES])
def test_offset_field_resident(gpu_device, oracle_built, precision, offset):
    """The resident evaluator (one ligand of up to 224 atoms per step, csrc/gf_resident.cu) runs the general kernel's
    device functions."""
    import openmmgridforce_b200 as gf
    c = _offset_case(1, 6, 200, offset, 0, seed=500 + int(abs(offset)) % 89 + (offset < 0))
    ge_ref, f_ref = _oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, precision, CELLS)
    grids2, k2 = _make(gf, gpu_device, c, precision, CELLS)
    assert k.eval_path() == _path(precision, CELLS, 1)
    k2.execute_host(c["pos"][0], want_grid_energies=True)     # the launch path's module is loaded before the block resides
    k.set_resident(True)
    te, tf = _tol(precision, 0)
    for step in range(c["pos"].shape[0]):
        en, forces, ge = k.execute_host(c["pos"][step], want_grid_energies=True)
        _check(en, ge, forces, ge_ref[step:step + 1], f_ref[step:step + 1], te, tf, f"resident C={offset:g} step {step}")
    assert 1 <= k.resident_launches() <= 2
    k.set_resident(False)
    _close(grids, k)
    _close(grids2, k2)


# ---------------------------------------------------------------------------------------------------------------------
# B. Record-kernel mode matrix
# ---------------------------------------------------------------------------------------------------------------------
SHAPES = [(1, 1), (1, 5), (1, 300), (3, 47), (37, 47), (130, 9), (1, 4099)]
RECORD_LAYOUT = {1: BSPLINE, 2: HERMITE}


@pytest.mark.parametrize("shape", SHAPES, ids=[f"{r}x{a}" for r, a in SHAPES])
@pytest.mark.parametrize("n_grids", [1, 2, 3, 4])
@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
@pytest.mark.parametrize("method", [1, 2], ids=["bspline", "tricubic"])
def test_record_kernel_modes(gpu_device, oracle_built, method, precision, n_grids, shape):
    import openmmgridforce_b200 as gf
    r, a = shape
    layout = RECORD_LAYOUT[method]
    c = _case(n_grids, r, a, seed=1000 * method + 100 * precision + 10 * n_grids + r + a, method=method, edges=True)
    ge_ref, f_ref = _oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, precision, layout)
    assert k.eval_path() == _path(precision, layout, n_grids)
    te, tf = _tol(precision, method)
    # F64_STORE with per-grid energies
    en, f64, ge = k.execute_host(c["pos"], want_grid_energies=True)
    _check(en, ge, f64, ge_ref, f_ref, te, tf, "F64_STORE")
    # F64_ADD onto a random base
    base = np.random.default_rng(r + a).normal(size=c["pos"].shape)
    acc = base.copy()
    en2, _, _ = k.execute_host(c["pos"], forces=acc, force_mode=gf.FORCE_F64_ADD)
    _check(en2, None, None, ge_ref, f_ref, te, tf, "F64_ADD")
    assert np.abs(acc - base - f_ref).max() <= tf * np.abs(f_ref).max() + 1e-15 * np.abs(base).max()
    # energy only: the same FP64 value path
    e0, none, _ = k.execute_host(c["pos"], want_forces=False)
    assert none is None
    assert np.abs(e0 - en).max() <= 1e-13 * max(np.abs(en).max(), np.abs(ge_ref).max(), 1.0)
    # F32_STORE: the F64 forces rounded to float
    f32 = np.full(c["pos"].shape, 7.0, dtype=np.float32)
    k.execute_host(c["pos"], forces=f32, force_mode=gf.FORCE_F32_STORE)
    assert np.array_equal(f32, f64.astype(np.float32)), int((f32 != f64.astype(np.float32)).sum())
    # classification, bit-exact (the trilinear oracle's cell: upper faces are the last cell at fraction 1)
    port0 = _port(oracle_built, c, method=0)
    got = k.classify_host(c["pos"], 0)
    for rep in range(min(r, 3)):
        _, _, want = port0.execute(c["pos"][rep], 0, classify=True)
        sl = slice(rep * a, (rep + 1) * a)
        assert np.array_equal(got["inside"][sl], want["inside"]) and np.array_equal(got["cell"][sl], want["cell"])
    _close(grids, k)


@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
@pytest.mark.parametrize("counts", [(2, 2, 2), (2, 3, 7), (9, 5, 6)])
def test_bspline_records_edges_and_thin_grids(gpu_device, oracle_built, counts, precision):
    """Every cell of small grids through the B-spline record kernels: clamped neighbours on every side, atoms on the faces,
    the corners and outside (mirrors test_gpu_tricubic.test_tricubic_edges_and_thin_grids)."""
    import openmmgridforce_b200 as gf
    rng = np.random.default_rng(sum(counts) + 7 * precision)
    sp = (0.2, 0.15, 0.1)
    length = np.array(sp) * (np.array(counts) - 1)
    n = 600
    pos = rng.uniform(-0.05, 1.05, size=(n, 3)) * length
    pos[0] = length
    pos[1] = 0.0
    pos[2:12, 0] = length[0]
    pos[12:22, 1] = length[1]
    pos[22:32, 2] = length[2]
    pos[32:42] = length - rng.uniform(0.0, 1.0, size=(10, 3)) * np.array(sp)
    grid = (rng.normal(size=counts) * 4).astype(np.float32).astype(np.float64)
    c = dict(counts=counts, spacing=sp, origin=(0.0, 0.0, 0.0), grids=[grid], scaling=rng.uniform(0.5, 1.5, size=(1, n)),
             pos=pos[None], oob_k=[10000.0], inv_power=[0.0], method=1)
    ge_ref, f_ref = _oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, precision, BSPLINE)
    assert k.eval_path() == _path(precision, BSPLINE, 1)
    en, forces, ge = k.execute_host(pos, want_grid_energies=True)
    te, tf = _tol(precision, 1)
    _check(en, ge, forces, ge_ref, f_ref, te, tf)
    _close(grids, k)


# ---------------------------------------------------------------------------------------------------------------------
# C. Device path, particle subsets, energy slots, per-atom energies and inv-power on the record kernels
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("method", [1, 2], ids=["bspline", "tricubic"])
def test_record_kernel_device_fixed_point_mixed(gpu_device, oracle_built, method):
    """OpenMM's fixed-point force buffer accumulated over two launches, energies accumulated, the next step's
    accumulator cleared by the launch."""
    import torch
    import openmmgridforce_b200 as gf
    r, a = 41, 47
    c = _case(3, r, a, seed=70 + method, method=method, edges=True)
    ge_ref, f_ref = _oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, 0, RECORD_LAYOUT[method])
    assert k.eval_path() == _path(0, RECORD_LAYOUT[method], 3)
    te, tf = _tol(0, method)
    dev = torch.device("cuda:0")
    n = r * a
    stride = ((n + 31) // 32) * 32
    d_pos = torch.from_numpy(c["pos"]).to(dev)
    d_f = torch.zeros(3 * stride, dtype=torch.int64, device=dev)
    d_e = torch.zeros(r, dtype=torch.float64, device=dev)
    d_next = torch.full((r,), 123.0, dtype=torch.float64, device=dev)
    d_out = torch.empty(n, 3, dtype=torch.float64, device=dev)
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    for _ in range(2):
        k.execute_device(r, a, d_pos.data_ptr(), d_e.data_ptr(), None, d_f.data_ptr(), gf.FORCE_FIXED_ADD, stride, None,
                         side.cuda_stream, d_energies_clear=d_next.data_ptr())
    gpu_device.fixed_to_f64(d_f.data_ptr(), stride, n, d_out.data_ptr(), side.cuda_stream)
    torch.cuda.synchronize()
    _check(d_e.cpu().numpy() / 2, None, None, ge_ref, f_ref, te, tf)
    # each launch truncates to the 2^-32 quantum once per component
    assert np.abs(d_out.cpu().numpy().reshape(r, a, 3) - 2 * f_ref).max() <= 2 * 2.0 ** -32 + tf * 2 * np.abs(f_ref).max()
    assert not d_next.cpu().numpy().any()
    _close(grids, k)


@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
@pytest.mark.parametrize("method", [1, 2], ids=["bspline", "tricubic"])
def test_record_kernel_subset_slots_and_atom_energies(gpu_device, oracle_built, method, precision):
    """A particle subset (forces land at the particle index, untouched entries stay, STORE and ADD), energy slots that
    interleave (0,1,2,0,1,2,...: every run of equal keys in a warp has length 1), and per-atom energies."""
    import openmmgridforce_b200 as gf
    layout = RECORD_LAYOUT[method]
    rng = np.random.default_rng(10 * method + precision)
    r, n_particles, a = 5, 90, 60
    c = _case(3, r, n_particles, seed=11 + method, method=method, edges=True)
    particles = np.sort(rng.choice(n_particles, size=a, replace=False)).astype(np.int32)
    sub = dict(c, scaling=rng.normal(size=(3, a)))
    sub["scaling"][:, ::7] = 0.0
    te, tf = _tol(precision, method)
    grids, k = _make(gf, gpu_device, sub, precision, layout, particles=particles)
    assert k.eval_path() == _path(precision, layout, 3)
    sel_pos = np.ascontiguousarray(c["pos"][:, particles])
    ge_ref, f_ref = _oracle(oracle_built, sub, pos=sel_pos)
    for mode in (gf.FORCE_F64_STORE, gf.FORCE_F64_ADD):
        forces = np.full(c["pos"].shape, 3.5)
        en, _, _ = k.execute_host(c["pos"], forces=forces, force_mode=mode)
        _check(en, None, None, ge_ref, f_ref, te, tf, f"subset mode {mode}")
        want = f_ref + (3.5 if mode == gf.FORCE_F64_ADD else 0.0)
        assert np.abs(forces[:, particles] - want).max() <= tf * np.abs(f_ref).max() + 1e-15 * 3.5, mode
        untouched = np.setdiff1d(np.arange(n_particles), particles)
        assert (forces[:, untouched] == 3.5).all(), mode
    # interleaved energy slots
    slots = (np.arange(a) % 3).astype(np.int32)
    k.set_energy_slots(slots, 3)
    assert k.eval_path() == _path(precision, layout, 3)
    forces = np.zeros_like(c["pos"])
    en, _, ge = k.execute_host(c["pos"], forces=forces, force_mode=gf.FORCE_F64_ADD, want_grid_energies=True)
    en, ge = en.reshape(r, 3), ge.reshape(r, 3, 3)
    for s in range(3):
        sel = np.nonzero(slots == s)[0]
        g_s, _ = _oracle(oracle_built, sub, pos=np.ascontiguousarray(sel_pos[:, sel]), scaling=sub["scaling"][:, sel])
        _check(en[:, s], ge[:, s], None, g_s, None, te, tf, f"slot {s}")
    assert np.abs(forces[:, particles] - f_ref).max() <= tf * np.abs(f_ref).max()
    k.set_energy_slots(None, 1)
    # per-atom energies against one-atom oracle runs
    k.request_atom_energies(True)
    en, _, _ = k.execute_host(c["pos"])
    ae = k.atom_energies(r)
    want = np.zeros((r, a))
    for ia in range(a):
        g1, _ = _oracle(oracle_built, sub, pos=np.ascontiguousarray(sel_pos[:, ia:ia + 1]), scaling=sub["scaling"][:, ia:ia + 1])
        want[:, ia] = g1.sum(axis=1)
    assert np.abs(ae - want).max() <= te * np.abs(want).max()
    assert np.abs(ae.sum(axis=1) - en).max() <= 1e-12 * np.abs(want).max() * a
    k.request_atom_energies(False)
    _close(grids, k)


@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
@pytest.mark.parametrize("method", [1, 2], ids=["bspline", "tricubic"])
def test_record_kernel_inv_power_batched(gpu_device, oracle_built, method, precision):
    """inv_power 4 on a positive grid (pow of the interpolated value and its derivative), 37 replicas x 47 atoms."""
    import openmmgridforce_b200 as gf
    layout = RECORD_LAYOUT[method]
    c = _case(2, 37, 47, seed=300 + method, method=method, edges=True)
    rng = np.random.default_rng(3)
    c["grids"] = [rng.uniform(0.5, 3.0, size=COUNTS).astype(np.float32).astype(np.float64) for _ in range(2)]
    c["inv_power"] = [4.0, 0.0]
    ge_ref, f_ref = _oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, precision, layout)
    assert k.eval_path() == _path(precision, layout, 2, lines_ok=False)
    en, forces, ge = k.execute_host(c["pos"], want_grid_energies=True)
    te, tf = _tol(precision, method)
    _check(en, ge, forces, ge_ref, f_ref, te, tf)
    _close(grids, k)


# ---------------------------------------------------------------------------------------------------------------------
# D. Dispatch and slot edges
# ---------------------------------------------------------------------------------------------------------------------
MANY_LAYOUTS = [(0, CELLS), (0, ROWS), (0, PAIRS), (0, BSPLINE), (0, BSPLINE_POINTS), (0, HERMITE), (0, POINTS),
                (1, CELLS), (1, ROWS), (1, BSPLINE), (1, BSPLINE_POINTS), (1, HERMITE), (1, POINTS)]
LAYOUT_IDS = {CELLS: "cells", ROWS: "rows", PAIRS: "pairs", BSPLINE: "bspline", BSPLINE_POINTS: "bspline_points",
              HERMITE: "hermite", POINTS: "points"}


@pytest.mark.parametrize("n_grids", [5, 8])
@pytest.mark.parametrize("mode", MANY_LAYOUTS, ids=[("mixed-" if p == 0 else "double-") + LAYOUT_IDS[l] for p, l in MANY_LAYOUTS])
def test_many_grids_one_geometry(gpu_device, oracle_built, mode, n_grids):
    """More than 4 grids: the general kernel with a run-time grid count (NG = 0, SAME) and the record kernels' grid loop
    beyond 4. Totals, per-grid energies and forces."""
    import openmmgridforce_b200 as gf
    precision, layout = mode
    method = METHOD[layout]
    c = _case(n_grids, 13, 47, seed=40 * n_grids + layout + precision, method=method, edges=True)
    ge_ref, f_ref = _oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, precision, layout)
    assert k.eval_path() == _path(precision, layout, n_grids)
    en, forces, ge = k.execute_host(c["pos"], want_grid_energies=True)
    te, tf = _tol(precision, method)
    _check(en, ge, forces, ge_ref, f_ref, te, tf)
    _close(grids, k)


@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
def test_eight_grids_of_mixed_geometry(gpu_device, oracle_built, precision):
    """Eight grids, no two of the same geometry: each is classified on its own (NG = 0, SAME = false)."""
    import openmmgridforce_b200 as gf
    rng = np.random.default_rng(88 + precision)
    r, a = 9, 47
    geoms = [((11 + g, 9 + (g * 3) % 5, 13 - g % 4), (0.09 + 0.01 * (g % 3), 0.1, 0.08 + 0.005 * g), (0.02 * g, -0.01 * g, 0.0))
             for g in range(8)]
    vals = [(rng.normal(size=cnt) * 4).astype(np.float32).astype(np.float64) for cnt, _, _ in geoms]
    sc = rng.normal(size=(8, a))
    sc[:, ::7] = 0.0
    pos = rng.uniform(-0.1, 1.3, size=(r, a, 3))
    grids = [gf.Grid(gpu_device, cnt, sp, og, v, precision, layout=CELLS) for (cnt, sp, og), v in zip(geoms, vals)]
    k = gf.Kernel(gpu_device, grids, sc, oob_k=OOB_K)
    assert k.eval_path() == 0
    en, forces, ge = k.execute_host(pos, want_grid_energies=True)
    ge_ref = np.zeros((r, 8))
    f_ref = np.zeros_like(pos)
    for g, ((cnt, sp, og), v) in enumerate(zip(geoms, vals)):
        port = oracle_built.PortOracle(cnt, sp, og, [v], sc[g:g + 1], oob_k=[OOB_K[g]])
        e, f = port.execute_batched(pos, n_threads=N_THREADS)
        ge_ref[:, g] = e[:, 0]
        f_ref += f
    te, tf = _tol(precision, 0)
    _check(en, ge, forces, ge_ref, f_ref, te, tf)
    _close(grids, k)


@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
def test_inv_power_on_one_grid_of_three(gpu_device, oracle_built, precision):
    """inv-power on grid 1 only: the record kernels (lines paths) refuse the state, the general kernel serves it."""
    import openmmgridforce_b200 as gf
    c = _case(3, 37, 47, seed=404)
    c["grids"][1] = np.random.default_rng(5).uniform(0.5, 3.0, size=COUNTS).astype(np.float32).astype(np.float64)
    c["inv_power"] = [0.0, 4.0, 0.0]
    ge_ref, f_ref = _oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, precision, CELLS)
    assert k.eval_path() == 0
    en, forces, ge = k.execute_host(c["pos"], want_grid_energies=True)
    te, tf = _tol(precision, 0)
    _check(en, ge, forces, ge_ref, f_ref, te, tf)
    _close(grids, k)


def test_update_parameters_moves_between_paths(gpu_device, oracle_built):
    """update_parameters(inv_power=...) takes a 3-grid MIXED CELLS state from the lines kernel to the general kernel and
    back; every step against the oracle with the same parameters."""
    import openmmgridforce_b200 as gf
    c = _case(3, 21, 47, seed=505)
    c["grids"][1] = np.random.default_rng(6).uniform(0.5, 3.0, size=COUNTS).astype(np.float32).astype(np.float64)
    grids, k = _make(gf, gpu_device, c, 0, CELLS)
    te, tf = _tol(0, 0)
    for inv_power, path in (([0.0, 0.0, 0.0], 1), ([0.0, 4.0, 0.0], 0), ([0.0, 0.0, 0.0], 1)):
        k.update_parameters(inv_power=inv_power)
        assert k.eval_path() == path
        ge_ref, f_ref = _oracle(oracle_built, dict(c, inv_power=inv_power))
        en, forces, ge = k.execute_host(c["pos"], want_grid_energies=True)
        _check(en, ge, forces, ge_ref, f_ref, te, tf, str(inv_power))
    _close(grids, k)


# every kernel family: (precision, layout, n_grids)
SLOT_FAMILIES = [(0, CELLS, 1), (0, CELLS, 3), (1, CELLS, 3), (0, ROWS, 1), (1, CELLS, 1), (0, BSPLINE, 1), (1, BSPLINE, 2),
                 (0, HERMITE, 2), (1, HERMITE, 1)]


@pytest.mark.parametrize("family", SLOT_FAMILIES,
                         ids=[f"{'mixed' if p == 0 else 'double'}-{LAYOUT_IDS[l]}{g}" for p, l, g in SLOT_FAMILIES])
def test_empty_energy_slots(gpu_device, oracle_built, family):
    """3 atoms in 200 energy slots, 2 replicas: 400 entries, more than the launch has threads. Slots without atoms read
    exactly 0 on the host path; on the device path the launch clears all 400 entries of the next accumulator."""
    import torch
    import openmmgridforce_b200 as gf
    precision, layout, n_grids = family
    method = METHOD[layout]
    r, a, n_slots = 2, 3, 200
    c = _case(n_grids, r, a, seed=600 + layout, method=method, frac_outside=0.0)
    c["scaling"] = np.random.default_rng(1).uniform(0.5, 1.5, size=(n_grids, a))
    slots = np.array([0, 117, 199], dtype=np.int32)
    grids, k = _make(gf, gpu_device, c, precision, layout)
    path = _path(precision, layout, n_grids)
    assert k.eval_path() == path
    k.set_energy_slots(slots, n_slots)
    assert k.eval_path() == path
    ge_ref, _ = _oracle(oracle_built, c)
    te, _ = _tol(precision, method)
    want = np.zeros((r, n_slots))
    for ia, s in enumerate(slots):
        g1, _ = _oracle(oracle_built, c, pos=np.ascontiguousarray(c["pos"][:, ia:ia + 1]), scaling=c["scaling"][:, ia:ia + 1])
        want[:, s] = g1.sum(axis=1)
    en, _, _ = k.execute_host(c["pos"])
    en = en.reshape(r, n_slots)
    empty = np.ones(n_slots, dtype=bool)
    empty[slots] = False
    assert (en[:, empty] == 0.0).all()
    assert np.abs(en[:, slots] - want[:, slots]).max() <= te * np.abs(ge_ref).max()
    dev = torch.device("cuda:0")
    d_pos = torch.from_numpy(c["pos"]).to(dev)
    d_e = torch.zeros(r * n_slots, dtype=torch.float64, device=dev)
    d_next = torch.full((r * n_slots,), 123.0, dtype=torch.float64, device=dev)
    d_f = torch.zeros(r * a * 3, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    k.execute_device(r, a, d_pos.data_ptr(), d_e.data_ptr(), None, d_f.data_ptr(), gf.FORCE_F64_STORE, 0, None,
                     torch.cuda.current_stream().cuda_stream, d_energies_clear=d_next.data_ptr())
    torch.cuda.synchronize()
    nxt = d_next.cpu().numpy()
    assert not nxt.any(), f"{int(np.count_nonzero(nxt))} of {nxt.size} entries not cleared"
    e_dev = d_e.cpu().numpy().reshape(r, n_slots)
    assert (e_dev[:, empty] == 0.0).all()
    assert np.abs(e_dev[:, slots] - want[:, slots]).max() <= te * np.abs(ge_ref).max()
    _close(grids, k)
