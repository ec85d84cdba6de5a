"""CPU tests of the parity oracle itself (no GPU):
  * the C restatement (oracle/gridforce_oracle.c) reproduces the committed golden vectors — outputs of the
    reference's own kernel — bit for bit;
  * where /root/reference is present (build container) it is also checked bit-for-bit against a fresh build of
    the reference kernel (oracle/_ref) on random inputs;
  * closed-form known answers (ones grid, linear field, restraint)."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import cases  # noqa: E402

GOLDEN = sorted(cases.CASES)


def _port(bindings, c):
    return bindings.PortOracle(c["counts"], c["spacing"], c["origin"], c["grids"], c["scaling"], oob_k=c["oob_k"],
                               inv_power=c["inv_power"], interpolation_method=c.get("interp", 0))


@pytest.mark.parametrize("name", GOLDEN)
def test_port_matches_golden_bit_exact(oracle_built, name):
    c, ref = cases.load_golden(name)
    port = _port(oracle_built, c)
    total_f = np.zeros_like(ref["forces"])
    for g in range(len(c["grids"])):
        e, f, _ = port.execute(c["pos"], g)
        assert e == ref["grid_energies"][g], f"{name} grid {g}: energy differs from the reference kernel"
        assert np.array_equal(f, ref["grid_forces"][g], equal_nan=True)
        total_f -= -f        # same accumulation order as forceData[ia] -= ... over forces 0..G-1
    assert np.array_equal(total_f, ref["forces"], equal_nan=True)


@pytest.mark.parametrize("name", GOLDEN)
def test_golden_inputs_match_generators(name):
    """The stored inputs are the ones cases.py generates (guards against a stale .npz)."""
    c, _ = cases.load_golden(name)
    fresh = cases.CASES[name]()
    assert c["counts"] == tuple(fresh["counts"])
    np.testing.assert_array_equal(c["pos"], np.asarray(fresh["pos"], dtype=np.float64))
    np.testing.assert_array_equal(c["scaling"], np.asarray(fresh["scaling"], dtype=np.float64))
    for a, b in zip(c["grids"], fresh["grids"]):
        np.testing.assert_array_equal(a, np.asarray(b, dtype=np.float64))


def test_port_matches_reference_build_random(oracle_built):
    if not oracle_built.ref_available():
        pytest.skip("oracle/_ref not built (no /root/reference on this machine); golden vectors cover it")
    rng = np.random.default_rng(42)
    for trial in range(6):
        counts = tuple(int(v) for v in rng.integers(2, 24, size=3))
        sp = tuple(rng.uniform(0.01, 0.3, size=3))
        og = tuple(rng.uniform(-2, 2, size=3))
        n, g = int(rng.integers(1, 400)), int(rng.integers(1, 4))
        grids = [rng.normal(size=counts) * 10 ** rng.uniform(-2, 4) for _ in range(g)]
        length = np.array(sp) * (np.array(counts) - 1)
        pos = np.array(og) + rng.uniform(-0.2, 1.2, size=(n, 3)) * length
        sc = rng.normal(size=(g, n))
        sc[:, rng.integers(0, n, size=max(1, n // 10))] = 0.0
        k = list(rng.uniform(10, 1e5, size=g))
        ref = oracle_built.RefOracle(n, counts, sp, og, grids, sc, oob_k=k)
        port = oracle_built.PortOracle(counts, sp, og, grids, sc, oob_k=k)
        for gi in range(g):
            er, fr = ref.execute(pos, groups=1 << gi)
            ep, fp, _ = port.execute(pos, gi)
            assert er == ep, f"trial {trial} grid {gi}"
            assert np.array_equal(fr, fp)
        ref.close()


def test_ligand_atoms_quirk_q1(oracle_built):
    """Position is read at ligand_atoms[ia] but the force is written at ia (ReferenceGridForceKernels.cpp:684 vs :1082)."""
    if not oracle_built.ref_available():
        pytest.skip("needs oracle/_ref")
    rng = np.random.default_rng(3)
    counts, sp = (8, 8, 8), (0.1, 0.1, 0.1)
    grid = rng.normal(size=counts)
    pos = rng.uniform(0.0, 0.7, size=(10, 3))
    la = [7, 2, 9]
    sc = np.array([[1.0, -2.0, 0.5]])
    ref = oracle_built.RefOracle(10, counts, sp, (0, 0, 0), [grid], sc, ligand_atoms=la)
    er, fr = ref.execute(pos)
    port = oracle_built.PortOracle(counts, sp, (0, 0, 0), [grid], sc)
    ep, fp, _ = port.execute(pos, 0, ligand_atoms=la)
    assert er == ep
    assert np.array_equal(fr[:3], fp) and not fr[3:].any()


def test_known_answers(oracle_built):
    c = cases.case_ones_grid()
    e, f, cls = _port(oracle_built, c).execute(c["pos"], 0, classify=True)
    assert abs(e - c["scaling"].sum()) < 1e-13 and not f.any() and cls["inside"].all()
    c = cases.case_linear_field()
    e, f, cls = _port(oracle_built, c).execute(c["pos"], 0, classify=True)
    np.testing.assert_allclose(f[0], [-20.0, -40.0, -60.0], rtol=1e-12)
    # atom 1: 0.5 nm beyond +x and 0.01 nm below -y, k = 1e4: F = -k*dev, E = k/2 * dev^2
    np.testing.assert_allclose(f[1], [-5000.0, 100.0, 0.0], rtol=1e-12)
    assert list(cls["inside"]) == [1, 0, 1, 1]
    assert tuple(cls["cell"][0]) == (3, 4, 2) and tuple(cls["cell"][1]) == (-1, -1, -1)
    assert tuple(cls["cell"][3]) == (-1, -1, -1)        # inside but scale == 0 -> restraint branch (Q3), adds 0
    v = lambda p: 2 * p[0] + 4 * p[1] + 6 * p[2] + 1    # noqa: E731
    expect = 10 * v(c["pos"][0]) + 0.5e4 * (0.5 ** 2 + 0.01 ** 2) + 2 * v(c["pos"][2])
    assert abs(e - expect) < 1e-9


def test_batched_threads_agree(oracle_built):
    c = cases.case_random_aniso()
    port = _port(oracle_built, c)
    pos = np.stack([c["pos"] + 0.001 * r for r in range(7)])
    e1, f1 = port.execute_batched(pos, n_threads=1)
    e4, f4 = port.execute_batched(pos, n_threads=4)
    assert np.array_equal(e1, e4) and np.array_equal(f1, f4)
    e0, f0, _ = port.execute(pos[3], 1)
    assert e1[3, 1] == e0


def test_reference_contexts_on_threads(oracle_built):
    """bench.py --impl reference drives one reference Context per host thread; the driver's stdout silencer is shared
    process state and must survive concurrent entry/exit (a crash here took the reference arm down on a 16-core box)."""
    if not oracle_built.ref_available():
        pytest.skip("needs oracle/_ref")
    import threading
    c = cases.case_random_aniso()
    n = c["pos"].shape[0]
    want = None
    oracles = [oracle_built.RefOracle(n, c["counts"], c["spacing"], c["origin"], c["grids"], c["scaling"],
                                      oob_k=c["oob_k"]) for _ in range(16)]
    want = oracles[0].execute_repeat(c["pos"], 3)
    got = [None] * len(oracles)

    def work(i):
        for _ in range(200):
            got[i] = oracles[i].execute_repeat(c["pos"], 1)

    th = [threading.Thread(target=work, args=(i,)) for i in range(len(oracles))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert all(g == want for g in got)
    for o in oracles:
        o.close()
    print("stdout still works", flush=True)


def test_port_bspline_matches_reference_build_random(oracle_built):
    """Interpolation method 1 (cubic B-spline, :727-795) incl. atoms on the faces and in edge cells, bit for bit."""
    if not oracle_built.ref_available():
        pytest.skip("oracle/_ref not built; golden vectors bspline_* cover it")
    rng = np.random.default_rng(7)
    for trial in range(8):
        counts = tuple(int(v) for v in rng.integers(2, 14, size=3))
        sp = tuple(rng.uniform(0.01, 0.3, size=3))
        og = tuple(rng.uniform(-2, 2, size=3))
        n = int(rng.integers(2, 300))
        grid = rng.normal(size=counts) * 10
        length = np.array(sp) * (np.array(counts) - 1)
        pos = np.array(og) + rng.uniform(-0.1, 1.1, size=(n, 3)) * length
        pos[0] = np.array(og) + length
        pos[1] = np.array(og)
        sc = rng.normal(size=(1, n))
        ref = oracle_built.RefOracle(n, counts, sp, og, [grid], sc, interpolation_method=1)
        port = oracle_built.PortOracle(counts, sp, og, [grid], sc, interpolation_method=1)
        er, fr = ref.execute(pos)
        ep, fp, _ = port.execute(pos, 0)
        assert er == ep and np.array_equal(fr, fp), trial
        ref.close()


def tricubic_positions(rng, counts, sp, og, n, outside_frac=0.05):
    """Positions for interpolation method 2 that stay where the reference is defined: off the upper faces (quirk Q2)
    and out of the last x layer (ix == nx-2 makes the reference read past the end of its value vector, :825-832); first
    cells and the last cells in y and z (whose neighbour reads land in the next row / x-slab) are included."""
    counts = np.array(counts)
    length = np.array(sp) * (counts - 1)
    hi = np.array([np.array(sp)[0] * (counts[0] - 2), length[1], length[2]]) * (1 - 1e-9)
    pos = np.array(og) + rng.uniform(0.0, 1.0, size=(n, 3)) * hi
    k = n // 5
    pos[:k] = np.array(og) + rng.uniform(0.0, 1.0, size=(k, 3)) * np.array(sp)                         # first cells
    pos[k:2 * k, 1:] = (np.array(og) + length - rng.uniform(1e-9, 1.0, size=(k, 3)) * np.array(sp))[:, 1:]   # last y/z cells
    m = max(1, int(outside_frac * n))
    pos[-m:] = np.array(og) + rng.uniform(-0.2, 1.2, size=(m, 3)) * length
    inside_last_x = (pos[-m:, 0] - og[0] >= hi[0]) & (pos[-m:, 0] - og[0] <= length[0])
    pos[-m:, 0] = np.where(inside_last_x, og[0] - 0.01, pos[-m:, 0])                                   # outside instead
    return pos


def test_port_tricubic_matches_reference_build_random(oracle_built):
    """Interpolation method 2 (tricubic Hermite, :796-893) incl. the first cells (derivative estimates off) and the last
    y/z cells (flat-index neighbours in the next row / slab), bit for bit, with and without inv-power."""
    if not oracle_built.ref_available():
        pytest.skip("oracle/_ref not built; golden vectors tricubic_* cover it")
    rng = np.random.default_rng(11)
    for trial in range(10):
        counts = tuple(int(v) for v in rng.integers(4, 14, size=3))
        sp = tuple(rng.uniform(0.01, 0.3, size=3))
        og = tuple(rng.uniform(-2, 2, size=3))
        n = int(rng.integers(20, 300))
        grid = rng.normal(size=counts) * 10
        inv_power = [0.0]
        if trial % 3 == 2:
            grid = np.abs(grid) + 0.5
            inv_power = [3.0]
        pos = tricubic_positions(rng, counts, sp, og, n)
        sc = rng.normal(size=(1, n))
        ref = oracle_built.RefOracle(n, counts, sp, og, [grid], sc, inv_power=inv_power, interpolation_method=2)
        port = oracle_built.PortOracle(counts, sp, og, [grid], sc, inv_power=inv_power, interpolation_method=2)
        er, fr = ref.execute(pos)
        ep, fp, _ = port.execute(pos, 0)
        assert er == ep and np.array_equal(fr, fp), trial
        ref.close()


def test_inv_power_transform_matches_reference(oracle_built):
    """RUNTIME inv-power mode: the restatement of GridForce::applyInvPowerTransformation against the reference's own
    method (where built) and against the committed fixture it produced."""
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "inv_power_transform.npz"))
    got = oracle_built.port_inv_power_transform(z["values"], float(z["inv_power"]))
    assert np.array_equal(got, z["ref_transformed"])
    assert int(z["mode_after"]) == 2        # STORED
    if oracle_built.ref_available():
        rng = np.random.default_rng(3)
        v = rng.normal(size=(7, 5, 9)) * 10 ** rng.uniform(-3, 4, size=(7, 5, 9))
        v[rng.integers(0, 7, 10), rng.integers(0, 5, 10), rng.integers(0, 9, 10)] = 0.0
        for n in (2.0, 4.0, 3.5):
            ref, mode = oracle_built.ref_inv_power_transform(v, n)
            assert mode == 2 and np.array_equal(ref, oracle_built.port_inv_power_transform(v, n))


def test_tricubic_known_answers(oracle_built):
    """Interpolation method 2 (:796-893) on fields whose answer can be written down, which also records what this branch
    of the reference is and is not: a constant field is reproduced exactly with zero force; a linear field
    V = 2x + 4y + 6z + 1 is reproduced in VALUE at cell midpoints and its x-force everywhere in the interior, but the
    y- and z-differences of the branch (one-sided, against neighbour rows interpolated with the value basis only,
    :849-867) are not derivative estimates of the field: at a midpoint the y- and z-forces come out at HALF the field's
    gradient, and off the midpoints the value itself is off. The restatement is bit-exact with the reference build on
    random inputs (test_port_tricubic_matches_reference_build_random); this test pins the same behaviour by hand."""
    counts, sp = (9, 9, 9), (0.1, 0.1, 0.1)
    i, j, k = np.meshgrid(*(np.arange(n) * 0.1 for n in counts), indexing="ij")
    rng = np.random.default_rng(3)
    pos = rng.uniform(0.0, 0.8, size=(60, 3)) * (1 - 1e-9)
    pos[:, 0] *= 0.875                                              # not the last x layer (its ix+2 neighbours are past the vector)
    sc = rng.uniform(0.5, 1.5, size=(1, 60))
    const = oracle_built.PortOracle(counts, sp, (0.0, 0.0, 0.0), [np.full(counts, 3.25)], sc, interpolation_method=2)
    e, f, _ = const.execute(pos, 0)
    assert abs(e - 3.25 * sc.sum()) <= 1e-12 * abs(e) and np.abs(f).max() <= 1e-9
    grid = 2 * i + 4 * j + 6 * k + 1
    cells = rng.integers(1, 7, size=(40, 3))                        # interior cells 1..6
    mid = (cells + 0.5) * 0.1
    one = np.ones((1, 40))
    lin = oracle_built.PortOracle(counts, sp, (0.0, 0.0, 0.0), [grid], one, interpolation_method=2)
    f_all = np.zeros((40, 3))
    for a in range(40):                                              # per-atom energies: one atom at a time
        pa = np.zeros((40, 3)) - 1.0                                 # the others outside (restraint, not interpolation)
        pa[a] = mid[a]
        ea, fa, _ = lin.execute(pa, 0)
        outside = 39 * 3 * 0.5 * 10000.0 * 1.0                       # 39 atoms at (-1,-1,-1): k/2 * dev^2 per axis
        v = 2 * mid[a, 0] + 4 * mid[a, 1] + 6 * mid[a, 2] + 1
        assert abs((ea - outside) - v) <= 1e-9, a
        f_all[a] = fa[a]
    assert np.abs(f_all - np.array([-2.0, -2.0, -3.0])).max() <= 1e-9
    off = np.array([[0.33, 0.41, 0.27]])
    one1 = oracle_built.PortOracle(counts, sp, (0.0, 0.0, 0.0), [grid], np.ones((1, 1)), interpolation_method=2)
    e_off, f_off, _ = one1.execute(off, 0)
    assert abs(f_off[0, 0] + 2.0) <= 1e-9                            # x: centred differences + cubic Hermite, exact
    assert abs(e_off - 4.92) > 1e-3                                  # the value is NOT the field's off the midpoints


def test_reference_method3_matrix_is_truncated():
    """Why interpolation method 3 (triquintic Hermite, ReferenceGridForceKernels.cpp:895-1015) is refused instead of
    reproduced: the 216 x 216 coefficient matrix the reference multiplies the 216 corner derivatives with
    (platforms/reference/src/TriquinticMatrix.h) holds 31 initialised rows in the reference tree; the other 185 are
    zero-initialised, so the "interpolant" ignores 180 of its 216 inputs (rank 31). There is no defined behaviour to match.
    Reads the header from the original project's source tree, located by the REFERENCE_DIR environment variable."""
    import re
    path = os.path.join(os.environ.get("REFERENCE_DIR", ""), "platforms", "reference", "src", "TriquinticMatrix.h")
    if not os.environ.get("REFERENCE_DIR") or not os.path.exists(path):
        pytest.skip("needs the original project's source tree (set REFERENCE_DIR)")
    text = open(path).read()
    body = text[text.index("TRIQUINTIC_COEFFICIENTS[216][216] = {") + len("TRIQUINTIC_COEFFICIENTS[216][216] = {"):]
    rows = re.findall(r"\{([^{}]*)\}", body[:body.rindex("};")])
    m = np.zeros((216, 216))
    for i, r in enumerate(rows[:216]):
        vals = [float(x) for x in r.replace("\n", " ").split(",") if x.strip()]
        m[i, :len(vals)] = vals
    assert len(rows) < 216
    assert np.linalg.matrix_rank(m) < 216
    assert int((np.abs(m).sum(axis=0) == 0).sum()) > 100        # inputs that cannot influence the result
