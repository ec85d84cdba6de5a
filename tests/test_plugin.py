"""The OpenMM-plugin path (C++: registerPlatforms/registerKernelFactories -> B200Platform -> GridForceImpl ->
B200CalcGridForceKernel), driven the way the reference's own tests drive a platform
(python/tests/test_grid_force.py:40-64, 117-159), and compared with the golden outputs of the reference kernel."""
import ctypes
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import cases  # noqa: E402


def test_plugin_exports_openmm_entry_points():
    """What OpenMM's plugin loader needs from a platform library (every reference platform lib exports the same two)."""
    import openmmgridforce_b200.gridforceplugin as gfp
    lib = ctypes.CDLL(gfp.plugin_library_path())
    for name in ("registerPlatforms", "registerKernelFactories", "registerB200GridForceKernelFactories"):
        assert hasattr(lib, name)


def test_platform_registers_and_lists_kernel():
    import openmmgridforce_b200.gridforceplugin as gfp
    p = gfp.Platform.getPlatformByName("B200")        # registers, then checks supportsKernels(["CalcGridForce"])
    assert p.getName() == "B200"
    with pytest.raises(RuntimeError):
        gfp.Platform.getPlatformByName("CUDA")


def test_api_validation_matches_reference_messages():
    import openmmgridforce_b200.gridforceplugin as gfp
    f = gfp.GridForce()
    with pytest.raises(RuntimeError, match="Invalid interpolation method"):
        f.setInterpolationMethod(4)
    with pytest.raises(RuntimeError, match="inv_power must be non-zero"):
        f.setInvPowerMode(gfp.InvPowerMode_STORED, 0.0)


def test_inv_power_mode_bookkeeping_matches_reference():
    """Mode transitions and their exceptions (reference GridForce.cpp:190-272); none of this needs a GPU because the
    checks come before any device work."""
    import openmmgridforce_b200.gridforceplugin as gfp
    f = gfp.GridForce()
    f.addGridCounts(2, 2, 2)
    f.addGridSpacing(0.1, 0.1, 0.1)
    with pytest.raises(RuntimeError, match="inv_power must be 0 when mode == NONE"):
        f.setInvPowerMode(gfp.InvPowerMode_NONE, 2.0)
    f.setInvPowerMode(gfp.InvPowerMode_STORED, 4.0)          # no values yet: any mode may be chosen
    f.setGridValues(np.ones(8))
    with pytest.raises(RuntimeError, match="already has STORED transformation"):
        f.setInvPowerMode(gfp.InvPowerMode_RUNTIME, 4.0)
    with pytest.raises(RuntimeError, match="when mode == RUNTIME"):
        f.applyInvPowerTransformation()                      # STORED grids are already transformed
    g = gfp.GridForce()
    g.setGridValues(np.ones(8))
    g.setInvPowerMode(gfp.InvPowerMode_RUNTIME, 4.0)
    with pytest.raises(RuntimeError, match="Call applyInvPowerTransformation"):
        g.setInvPowerMode(gfp.InvPowerMode_STORED, 4.0)
    h = gfp.GridForce()
    h.setInvPowerMode(gfp.InvPowerMode_RUNTIME, 4.0)
    with pytest.raises(RuntimeError, match="No grid values to transform"):
        h.applyInvPowerTransformation()


def _build_system(gfp, c, ligand_atoms=None):
    system = gfp.System()
    for _ in range(c["pos"].shape[0]):
        system.addParticle(1.0)
    forces = []
    for g, vals in enumerate(c["grids"]):
        force = gfp.GridForce()
        force.addGridCounts(*c["counts"])
        force.addGridSpacing(*c["spacing"])
        force.setGridOrigin(*c["origin"])
        if g == 0 and vals.size <= 5000:
            for v in vals.ravel():                    # the reference's per-value idiom (test_grid_force.py:58-59)
                force.addGridValue(v)
        else:
            force.setGridValues(vals)
        for s in c["scaling"][g]:
            force.addScalingFactor(s)
        if c["inv_power"][g] > 0:
            force.setInvPowerMode(gfp.InvPowerMode_STORED, c["inv_power"][g])
        force.setOutOfBoundsRestraint(c["oob_k"][g])
        force.setInterpolationMethod(c.get("interp", 0))
        force.setForceGroup(g)
        system.addForce(force)
        forces.append(force)
    return system, forces


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["mixed", "double"])
@pytest.mark.parametrize("name", sorted(cases.CASES))
def test_plugin_matches_reference_kernel(name, precision):
    import openmmgridforce_b200.gridforceplugin as gfp
    c, ref = cases.load_golden(name)
    platform = gfp.Platform.getPlatformByName("B200")
    platform.setPropertyDefaultValue("Precision", precision)
    system, forces = _build_system(gfp, c)
    context = gfp.Context(system, platform)
    context.setPositions(c["pos"])
    state = context.getState(getEnergy=True, getForces=True)
    te, tf = (1e-6, 1e-5) if precision == "mixed" else (1e-12, 1e-12)
    assert abs(state.getPotentialEnergy() - ref["energy"]) <= te * abs(ref["energy"])
    assert np.abs(state.getForces() - ref["forces"]).max() <= tf * np.abs(ref["forces"]).max()
    for g in range(len(forces)):                      # force groups gate each GridForce (GridForceImpl.cpp:64-68)
        s = context.getState(getEnergy=True, getForces=True, groups=1 << g)
        assert abs(s.getPotentialEnergy() - ref["grid_energies"][g]) <= te * max(abs(ref["grid_energies"][g]), 1e-300)
        assert np.abs(s.getForces() - ref["grid_forces"][g]).max() <= tf * np.abs(ref["grid_forces"][g]).max()
    platform.setPropertyDefaultValue("Precision", "mixed")


@pytest.mark.gpu
def test_plugin_batch_entry_point_and_groups(oracle_built):
    """GridForceBatch (one launch for R replicas x G forces) and particle groups, against the oracle."""
    import openmmgridforce_b200.gridforceplugin as gfp
    c, ref = cases.load_golden("ligand_three_grids")
    platform = gfp.Platform.getPlatformByName("B200")
    platform.setPropertyDefaultValue("Precision", "double")
    system, forces = _build_system(gfp, c)
    context = gfp.Context(system, platform)
    rng = np.random.default_rng(0)
    pos = np.stack([c["pos"] + rng.uniform(-0.05, 0.05, size=3) for _ in range(9)])
    en, f = context.evaluateBatch(pos, precision="double")
    port = oracle_built.PortOracle(c["counts"], c["spacing"], c["origin"], c["grids"], c["scaling"], oob_k=c["oob_k"])
    ge_ref, f_ref = port.execute_batched(pos)
    assert np.abs(en - ge_ref.sum(axis=1)).max() <= 1e-12 * np.abs(ge_ref).max()
    assert np.abs(f - f_ref).max() <= 1e-12 * np.abs(f_ref).max()
    # updateParametersInContext: doubled scaling factors on force 2
    forces[2].setScalingFactors(2.0 * c["scaling"][2])
    forces[2].updateParametersInContext(context)
    context.setPositions(c["pos"])
    s = context.getState(getEnergy=True, groups=1 << 2)
    assert abs(s.getPotentialEnergy() - 2.0 * ref["grid_energies"][2]) <= 1e-12 * abs(ref["grid_energies"][2]) * 2
    # particle groups: two groups of particles with their own scaling factors -> per-group energies
    system2 = gfp.System()
    for _ in range(47):
        system2.addParticle(1.0)
    force = gfp.GridForce()
    force.addGridCounts(*c["counts"])
    force.addGridSpacing(*c["spacing"])
    force.setGridOrigin(*c["origin"])
    force.setGridValues(c["grids"][0])
    ga, gb = list(range(0, 20)), list(range(20, 47))
    force.addParticleGroup("a", ga, list(c["scaling"][0][ga]))
    force.addParticleGroup("b", gb, list(c["scaling"][0][gb]))
    system2.addForce(force)
    ctx2 = gfp.Context(system2, platform)
    ctx2.setPositions(c["pos"])
    st = ctx2.getState(getEnergy=True, getForces=True)
    assert abs(st.getPotentialEnergy() - ref["grid_energies"][0]) <= 1e-12 * abs(ref["grid_energies"][0])
    assert np.abs(st.getForces() - ref["grid_forces"][0]).max() <= 1e-12 * np.abs(ref["grid_forces"][0]).max()
    eg = force.getParticleGroupEnergies(ctx2)
    assert len(eg) == 2 and abs(sum(eg) - ref["grid_energies"][0]) <= 1e-12 * abs(ref["grid_energies"][0])
    platform.setPropertyDefaultValue("Precision", "mixed")


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["mixed", "double"])
@pytest.mark.parametrize("method", [1, 2])
def test_plugin_batch_entry_point_other_interpolation_methods(oracle_built, method, precision):
    """GridForceBatch with cubic B-spline (1) and tricubic Hermite (2) forces: 33 replicas x 3 forces in one launch, against
    the oracle. MIXED runs the record kernels (BSPLINE / HERMITE records), DOUBLE the DOUBLE B-spline records and, for
    method 2, the raw-points layout."""
    import openmmgridforce_b200.gridforceplugin as gfp
    c, _ = cases.load_golden("ligand_three_grids")            # FP32-representable grids
    c = dict(c, interp=method)
    platform = gfp.Platform.getPlatformByName("B200")
    system, forces = _build_system(gfp, c)
    context = gfp.Context(system, platform, {"Precision": precision})
    rng = np.random.default_rng(method)
    pos = np.stack([c["pos"] + rng.uniform(-0.3, 0.3, size=3) for _ in range(33)])
    en, f = context.evaluateBatch(pos, precision=precision)
    port = oracle_built.PortOracle(c["counts"], c["spacing"], c["origin"], c["grids"], c["scaling"], oob_k=c["oob_k"],
                                   interpolation_method=method)
    ge_ref, f_ref = port.execute_batched(pos)
    te, tf = (1e-6, 1e-5) if precision == "mixed" else (1e-12, 1e-12)
    scale = np.maximum(np.abs(ge_ref.sum(axis=1)), np.abs(ge_ref).max(axis=1))
    assert (np.abs(en - ge_ref.sum(axis=1)) <= te * scale).all()
    assert np.abs(f - f_ref).max() <= tf * np.abs(f_ref).max()


@pytest.mark.gpu
def test_plugin_compact_layouts_when_records_do_not_fit():
    """Record layouts (methods 1 and 2) are 32x the raw grid; when that copy is refused (GFB_ERR_NOMEM) the platform runs
    the same method on the raw points. B200_COMPACT_LAYOUTS=1 takes that branch on purpose: a fresh interpreter (the switch
    is read once) evaluates the B-spline and tricubic golden cases through the plugin in both precisions."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = """
import os, sys, numpy as np
sys.path.insert(0, os.path.join(%r, "tests", "golden")); sys.path.insert(0, os.path.join(%r, "tests")); sys.path.insert(0, %r)
import cases
import openmmgridforce_b200.gridforceplugin as gfp
from test_plugin import _build_system
for name in ("bspline_random_aniso", "bspline_thin_grid", "tricubic_random_aniso", "tricubic_inv_power"):
    for precision, te, tf in (("mixed", 1e-6, 1e-5), ("double", 1e-12, 1e-12)):
        c, ref = cases.load_golden(name)
        system, forces = _build_system(gfp, c)
        ctx = gfp.Context(system, gfp.Platform.getPlatformByName("B200"), {"Precision": precision})
        ctx.setPositions(c["pos"])
        st = ctx.getState(getEnergy=True, getForces=True)
        assert abs(st.getPotentialEnergy() - ref["energy"]) <= te * abs(ref["energy"]), (name, precision)
        assert np.abs(st.getForces() - ref["forces"]).max() <= tf * np.abs(ref["forces"]).max(), (name, precision)
print("compact ok")
""" % (root, root, root)
    env = dict(os.environ, B200_COMPACT_LAYOUTS="1")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "compact ok" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


@pytest.mark.gpu
def test_plugin_refuses_what_it_does_not_implement():
    import openmmgridforce_b200.gridforceplugin as gfp
    c, _ = cases.load_golden("ramp_grid")
    platform = gfp.Platform.getPlatformByName("B200")
    system, forces = _build_system(gfp, c)
    forces[0].setInterpolationMethod(3)               # quintic Hermite needs the 27 derivative grids: loud refusal, no fallback
    with pytest.raises(RuntimeError, match="not implemented on this platform"):
        gfp.Context(system, platform)


@pytest.mark.gpu
def test_plugin_runtime_inv_power_mode(oracle_built):
    """RUNTIME mode through the GridForce API: applyInvPowerTransformation() stores G^(1/n) (on the GPU), flips the mode to
    STORED, and the evaluation then recovers the untransformed field (python/gridforceplugin.i:181, GridForce.cpp:221-272)."""
    import openmmgridforce_b200.gridforceplugin as gfp
    c, _ = cases.load_golden("inv_power")
    raw = c["grids"][0] ** 4                              # an untransformed, strictly positive field
    force = gfp.GridForce()
    force.addGridCounts(*c["counts"])
    force.addGridSpacing(*c["spacing"])
    force.setGridValues(raw)
    with pytest.raises(RuntimeError, match="when mode == RUNTIME"):
        force.applyInvPowerTransformation()
    force.setInvPowerMode(gfp.InvPowerMode_RUNTIME, 4.0)
    force.applyInvPowerTransformation()
    assert force.getInvPowerMode() == gfp.InvPowerMode_STORED
    want = oracle_built.port_inv_power_transform(raw, 4.0)
    got = force.getGridValues().reshape(raw.shape)
    assert np.abs(got - want).max() <= 1e-14 * np.abs(want).max()
    for s in c["scaling"][0]:
        force.addScalingFactor(s)
    system = gfp.System()
    for _ in range(c["pos"].shape[0]):
        system.addParticle(1.0)
    system.addForce(force)
    platform = gfp.Platform.getPlatformByName("B200")
    platform.setPropertyDefaultValue("Precision", "double")
    ctx = gfp.Context(system, platform)
    ctx.setPositions(c["pos"])
    st = ctx.getState(getEnergy=True, getForces=True)
    port = oracle_built.PortOracle(c["counts"], c["spacing"], c["origin"], [want], c["scaling"], inv_power=[4.0])
    e, f, _ = port.execute(c["pos"], 0)
    assert abs(st.getPotentialEnergy() - e) <= 1e-11 * abs(e)
    assert np.abs(st.getForces() - f).max() <= 1e-11 * np.abs(f).max()
    platform.setPropertyDefaultValue("Precision", "mixed")


def test_plugin_has_no_cpu_fallback():
    """Without a usable GPU, Context creation must raise (the product never routes through a CPU path)."""
    import openmmgridforce_b200 as gf
    import openmmgridforce_b200.gridforceplugin as gfp
    try:
        n = gf.Device.count()
    except gf.GridForceB200Error:
        n = 0
    if n > 0:
        pytest.skip("a GPU is present")
    c, _ = cases.load_golden("ramp_grid")
    system, _ = _build_system(gfp, c)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        gfp.Context(system, gfp.Platform.getPlatformByName("B200"))


def test_gridforce_file_round_trip(tmp_path):
    """GridForce.saveToFile / loadFromFile round trip, as python/tests/test_auto_grid.py:54-102 does it."""
    import openmmgridforce_b200.gridforceplugin as gfp
    c = cases.case_ramp_grid()
    f = gfp.GridForce()
    f.addGridCounts(*c["counts"])
    f.addGridSpacing(*c["spacing"])
    f.setGridOrigin(0.25, -1.5, 3.0)
    f.setGridValues(c["grids"][0])
    f.setInvPowerMode(gfp.InvPowerMode_STORED, 4.0)
    path = str(tmp_path / "ramp.grid")
    f.saveToFile(path)
    g = gfp.GridForce()
    g.loadFromFile(path)
    assert g._counts == list(c["counts"]) and g._spacing == list(c["spacing"]) and g.getGridOrigin() == (0.25, -1.5, 3.0)
    assert np.array_equal(np.asarray(g._vals), c["grids"][0].ravel()) and g.getInvPower() == 4.0
    with pytest.raises(RuntimeError, match="Cannot open"):
        gfp.GridForce().loadFromFile(str(tmp_path / "nope.grid"))


@pytest.mark.gpu
def test_many_contexts_share_grids_and_run_from_threads():
    """The sampler pattern (example/sampler.py:130-151): several Contexts over Systems with the same three grids. Device
    grids are shared through the plugin's cache, and Contexts may be driven from different threads."""
    import threading
    import openmmgridforce_b200.gridforceplugin as gfp
    c, ref = cases.load_golden("ligand_three_grids")
    platform = gfp.Platform.getPlatformByName("B200")
    platform.setPropertyDefaultValue("Precision", "double")
    contexts = []
    for _ in range(4):
        system, _forces = _build_system(gfp, c)
        contexts.append(gfp.Context(system, platform))
    results = [None] * 4

    def run(i):
        ctx = contexts[i]
        for _ in range(20):
            ctx.setPositions(c["pos"] + 1e-3 * i)
            s = ctx.getState(getEnergy=True, getForces=True)
        ctx.setPositions(c["pos"])
        s = ctx.getState(getEnergy=True, getForces=True)
        results[i] = (s.getPotentialEnergy(), s.getForces())

    threads = [threading.Thread(target=run, args=(i,)) for i in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for e, f in results:
        assert abs(e - ref["energy"]) <= 1e-12 * abs(ref["energy"])
        assert np.abs(f - ref["forces"]).max() <= 1e-12 * np.abs(ref["forces"]).max()
    platform.setPropertyDefaultValue("Precision", "mixed")


def _auto_system(gfp, grid_type, with_nonbonded=True):
    """20 ligand particles + 280 receptor particles with NonbondedForce parameters; a GridForce that derives its grid
    (setAutoGenerateGrid) and its scaling factors (setAutoCalculateScalingFactors) from them, as
    python/tests/test_auto_grid.py:135-202 and test_auto_scaling.py do in the reference."""
    rng = np.random.default_rng(5)
    n_lig, n_rec = 20, 280
    counts, sp, og = (15, 14, 13), (0.12, 0.13, 0.14), (0.2, 0.1, 0.0)
    length = np.array(sp) * (np.array(counts) - 1)
    rec_pos = rng.uniform(-0.4, 2.2, size=(n_rec, 3))
    lig_pos = np.array(og) + rng.uniform(0.1, 0.9, size=(n_lig, 3)) * length
    q = rng.normal(size=n_lig + n_rec) * 0.4
    sg = rng.uniform(0.1, 0.2, size=n_lig + n_rec)
    ep = rng.uniform(0.1, 1.0, size=n_lig + n_rec)
    system = gfp.System()
    for _ in range(n_lig + n_rec):
        system.addParticle(1.0)
    if with_nonbonded:
        nb = gfp.NonbondedForce()
        for i in range(n_lig + n_rec):
            nb.addParticle(q[i], sg[i], ep[i])
        system.addForce(nb)
    force = gfp.GridForce()
    force.addGridCounts(*counts)
    force.addGridSpacing(*sp)
    force.setGridOrigin(*og)
    force.setAutoGenerateGrid(True)
    force.setGridType(grid_type)
    force.setReceptorAtoms(range(n_lig, n_lig + n_rec))
    force.setReceptorPositionsFromLists(rec_pos[:, 0], rec_pos[:, 1], rec_pos[:, 2])
    force.setAutoCalculateScalingFactors(True)
    force.setScalingProperty(grid_type)
    system.addForce(force)
    pos = np.concatenate([lig_pos, rec_pos])
    return system, force, dict(counts=counts, spacing=sp, origin=og, rec_pos=rec_pos, pos=pos, q=q, sg=sg, ep=ep, n_lig=n_lig)


@pytest.mark.gpu
@pytest.mark.parametrize("grid_type", ["charge", "ljr", "lja"])
def test_plugin_auto_generated_grid_and_scaling(oracle_built, grid_type):
    import openmmgridforce_b200.gridforceplugin as gfp
    system, force, d = _auto_system(gfp, grid_type)
    platform = gfp.Platform.getPlatformByName("B200")
    platform.setPropertyDefaultValue("Precision", "double")
    ctx = gfp.Context(system, platform)
    n_lig = d["n_lig"]
    # the kernel wrote both derived inputs back into the force (ReferenceGridForceKernels.cpp:209, :272)
    want_grid = oracle_built.port_generate_grid(d["counts"], d["spacing"], d["origin"], grid_type, d["rec_pos"], d["q"][n_lig:],
                                                d["sg"][n_lig:], d["ep"][n_lig:], grid_cap=41840.0, n_threads=4)
    got_grid = force.getGridValues().reshape(d["counts"])
    assert np.abs(got_grid - want_grid).max() <= 1e-10 * np.abs(want_grid).max()
    want_sc = {"charge": d["q"], "ljr": np.sqrt(d["ep"]) * (2 * d["sg"]) ** 6, "lja": np.sqrt(d["ep"]) * (2 * d["sg"]) ** 3}[grid_type]
    got_sc = force.getScalingFactors()
    assert got_sc.shape == want_sc.shape and np.abs(got_sc - want_sc).max() <= 1e-14 * np.abs(want_sc).max()
    # evaluation: every particle has a scaling factor now, so every particle is evaluated (as in the reference's tests)
    ctx.setPositions(d["pos"])
    st = ctx.getState(getEnergy=True, getForces=True)
    port = oracle_built.PortOracle(d["counts"], d["spacing"], d["origin"], [want_grid], want_sc[None, :])
    e, f, _ = port.execute(d["pos"], 0)
    assert abs(st.getPotentialEnergy() - e) <= 1e-9 * abs(e)
    assert np.abs(st.getForces() - f).max() <= 1e-9 * np.abs(f).max()
    platform.setPropertyDefaultValue("Precision", "mixed")


@pytest.mark.gpu
def test_plugin_auto_inputs_errors():
    import openmmgridforce_b200.gridforceplugin as gfp
    platform = gfp.Platform.getPlatformByName("B200")
    system, force, _ = _auto_system(gfp, "charge", with_nonbonded=False)
    with pytest.raises(RuntimeError, match="requires a NonbondedForce"):
        gfp.Context(system, platform)
    system, force, _ = _auto_system(gfp, "dipole")
    with pytest.raises(RuntimeError, match="Invalid scaling property|Invalid grid type"):
        gfp.Context(system, platform)
    system, force, _ = _auto_system(gfp, "ljr")
    force.setReceptorPositions(np.zeros((0, 3)))
    with pytest.raises(RuntimeError, match="Receptor positions must be set"):
        gfp.Context(system, platform)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["mixed", "double"])
def test_step_fusion_matches_separate_launches(precision, monkeypatch):
    """Three GridForces of one geometry in one Context share a launch per evaluation (B200StepFusion). Every force-group
    subset must give what the per-force golden outputs say — all three, pairs (a smaller fused launch), singles (no
    fusion) — in any order, and updateParametersInContext must invalidate the fused state."""
    import openmmgridforce_b200.gridforceplugin as gfp
    c, ref = cases.load_golden("ligand_three_grids")
    platform = gfp.Platform.getPlatformByName("B200")
    platform.setPropertyDefaultValue("Precision", precision)
    system, forces = _build_system(gfp, c)
    ctx = gfp.Context(system, platform)
    ctx.setPositions(c["pos"])
    te, tf = (1e-6, 1e-5) if precision == "mixed" else (1e-12, 1e-12)
    scale_f = np.abs(ref["forces"]).max()
    for groups in (0b111, 0b011, 0b101, 0b110, 0b001, 0b100, 0b111, 0b010, 0b111):
        st = ctx.getState(getEnergy=True, getForces=True, groups=groups)
        sel = [g for g in range(3) if (groups >> g) & 1]
        e_ref = sum(ref["grid_energies"][g] for g in sel)
        f_ref = sum(ref["grid_forces"][g] for g in sel)
        assert abs(st.getPotentialEnergy() - e_ref) <= te * max(abs(ref["grid_energies"][g]) for g in sel), bin(groups)
        assert np.abs(st.getForces() - f_ref).max() <= tf * scale_f, bin(groups)
    forces[1].setScalingFactors(3.0 * c["scaling"][1])
    forces[1].updateParametersInContext(ctx)
    st = ctx.getState(getEnergy=True, getForces=True)
    e_ref = ref["grid_energies"][0] + 3.0 * ref["grid_energies"][1] + ref["grid_energies"][2]
    f_ref = ref["grid_forces"][0] + 3.0 * ref["grid_forces"][1] + ref["grid_forces"][2]
    assert abs(st.getPotentialEnergy() - e_ref) <= te * max(abs(e) for e in ref["grid_energies"]) * 3
    assert np.abs(st.getForces() - f_ref).max() <= tf * np.abs(f_ref).max()
    secs, e = ctx.timeEvaluations(200)
    assert abs(e - e_ref) <= te * max(abs(x) for x in ref["grid_energies"]) * 3 and secs > 0
    print(f"{precision}: {secs * 1e6:.1f} us per fused 3-force evaluation")
    platform.setPropertyDefaultValue("Precision", "mixed")


@pytest.mark.gpu
def test_step_fusion_keeps_unlike_forces_apart():
    """Forces on different geometries, or with particle groups, never join a fused launch; a second Context on the same
    System has its own fusion state."""
    import openmmgridforce_b200.gridforceplugin as gfp
    a, ref_a = cases.load_golden("ligand_three_grids")
    platform = gfp.Platform.getPlatformByName("B200")
    platform.setPropertyDefaultValue("Precision", "double")
    system, forces = _build_system(gfp, a)
    # a fourth force on a coarser grid cut out of grid 0 (different geometry, same atoms)
    extra = gfp.GridForce()
    extra.addGridCounts(20, 20, 20)
    extra.addGridSpacing(0.1, 0.1, 0.1)
    extra.setGridOrigin(*a["origin"])
    extra.setGridValues(a["grids"][0][::2, ::2, ::2])
    for s in a["scaling"][0]:
        extra.addScalingFactor(s)
    extra.setForceGroup(3)
    system.addForce(extra)
    ctx1 = gfp.Context(system, platform)
    ctx2 = gfp.Context(system, platform)
    for ctx in (ctx1, ctx2, ctx1):
        ctx.setPositions(a["pos"])
        e_all = ctx.getState(getEnergy=True, getForces=True).getPotentialEnergy()
        e_3 = ctx.getState(getEnergy=True, groups=0b0111).getPotentialEnergy()
        e_x = ctx.getState(getEnergy=True, groups=0b1000).getPotentialEnergy()
        assert abs(e_3 - ref_a["energy"]) <= 1e-12 * max(abs(x) for x in ref_a["grid_energies"])
        assert abs(e_all - (e_3 + e_x)) <= 1e-12 * (abs(e_3) + abs(e_x))
    platform.setPropertyDefaultValue("Precision", "mixed")


def _extra_force(gfp, a, group, counts=(20, 20, 20), spacing=0.1, stride=2):
    """A force on a coarser grid cut out of grid 0 (different geometry, same atoms): never fusable with the others."""
    extra = gfp.GridForce()
    extra.addGridCounts(*counts)
    extra.addGridSpacing(spacing, spacing, spacing)
    extra.setGridOrigin(*a["origin"])
    extra.setGridValues(a["grids"][0][::stride, ::stride, ::stride])
    for s in a["scaling"][0]:
        extra.addScalingFactor(s)
    extra.setForceGroup(group)
    return extra


@pytest.mark.gpu
@pytest.mark.parametrize("order", ["unlike_between", "two_interleaved_sets"])
def test_step_fusion_with_other_forces_between_members(order):
    """System order [A, X, B, C] with X unfusable, and two interleaved fusable sets [A1, A2, B1, B2]: a member that does
    not belong to a fused launch must not disturb the others' pending results — forces must come out ONCE (a second
    fused launch would add them twice) and a second evaluation must not return the first one's energies."""
    import openmmgridforce_b200.gridforceplugin as gfp
    a, ref = cases.load_golden("ligand_three_grids")
    platform = gfp.Platform.getPlatformByName("B200")
    system = gfp.System()
    for _ in range(a["pos"].shape[0]):
        system.addParticle(1.0)
    _, members = _build_system(gfp, a)                  # three fusable forces (groups 0, 1, 2)
    if order == "unlike_between":
        seq = [members[0], _extra_force(gfp, a, 3), members[1], members[2]]
        fused_groups = [(0b0111, [0, 1, 2])]
    else:
        twin = [_extra_force(gfp, a, 3), _extra_force(gfp, a, 4)]       # a second fusable set (same coarse geometry)
        seq = [members[0], twin[0], members[1], twin[1], members[2]]
        fused_groups = [(0b00111, [0, 1, 2])]
    for f in seq:
        system.addForce(f)
    ctx = gfp.Context(system, platform, {"Precision": "double"})
    all_groups = (1 << 5) - 1
    for shift in (0.0, 0.013):                          # second pass: moved atoms, nothing cached may survive
        pos = a["pos"] + shift
        ctx.setPositions(pos)
        singles = {}
        for g in range(5):
            st = ctx.getState(getEnergy=True, getForces=True, groups=1 << g)
            singles[g] = (st.getPotentialEnergy(), st.getForces().copy())
        st = ctx.getState(getEnergy=True, getForces=True, groups=all_groups)
        e_sum = sum(v[0] for v in singles.values())
        f_sum = sum(v[1] for v in singles.values())
        assert abs(st.getPotentialEnergy() - e_sum) <= 1e-11 * sum(abs(v[0]) for v in singles.values())
        assert np.abs(st.getForces() - f_sum).max() <= 1e-11 * np.abs(f_sum).max()
        if shift == 0.0:
            for mask, sel in fused_groups:
                s2 = ctx.getState(getEnergy=True, getForces=True, groups=mask)
                assert abs(s2.getPotentialEnergy() - ref["energy"]) <= 1e-12 * max(abs(x) for x in ref["grid_energies"])
                assert np.abs(s2.getForces() - ref["forces"]).max() <= 1e-12 * np.abs(ref["forces"]).max()


@pytest.mark.gpu
def test_platform_properties_the_openmm_way():
    """Property names are registered with the platform: the BASE class's setPropertyDefaultValue accepts them and rejects
    others; per-Context properties win over the defaults and are reported by getPropertyValue."""
    import openmmgridforce_b200.gridforceplugin as gfp
    c, ref = cases.load_golden("ligand_three_grids")
    platform = gfp.Platform.getPlatformByName("B200")
    assert platform.getPropertyDefaultValue("Precision") == "mixed" and platform.getPropertyDefaultValue("DeviceIndex") == "0"
    with pytest.raises(RuntimeError, match="Illegal property name"):
        platform.setPropertyDefaultValue("NoSuchProperty", "1")
    system, _ = _build_system(gfp, c)
    with pytest.raises(RuntimeError, match="Illegal property name"):
        gfp.Context(system, platform, {"Presicion": "double"})
    system, _ = _build_system(gfp, c)
    with pytest.raises(RuntimeError, match="Precision must be"):
        gfp.Context(system, platform, {"Precision": "single"})
    system, _ = _build_system(gfp, c)
    ctx_d = gfp.Context(system, platform, {"Precision": "double"})
    system2, _ = _build_system(gfp, c)
    ctx_m = gfp.Context(system2, platform)
    assert platform.getPropertyValue(ctx_d, "Precision") == "double" and platform.getPropertyValue(ctx_m, "Precision") == "mixed"
    assert platform.getPropertyDefaultValue("Precision") == "mixed"          # the default did not move
    ctx_d.setPositions(c["pos"])
    ctx_m.setPositions(c["pos"])
    e_d = ctx_d.getState(getEnergy=True).getPotentialEnergy()
    e_m = ctx_m.getState(getEnergy=True).getPotentialEnergy()
    assert abs(e_d - ref["energy"]) <= 1e-12 * abs(ref["energy"])
    assert abs(e_m - ref["energy"]) <= 1e-6 * abs(ref["energy"]) and e_m != e_d


@pytest.mark.gpu
def test_set_particles_filter_and_atom_energies(oracle_built):
    """GridForce::setParticles (only the listed particles feel the grid, each with the scaling factor of ITS particle
    index — the reference CUDA platform's semantics, CudaGridForceKernels.cpp:122-127) and getParticleAtomEnergies."""
    import openmmgridforce_b200.gridforceplugin as gfp
    c, ref = cases.load_golden("ligand_three_grids")
    platform = gfp.Platform.getPlatformByName("B200")
    keep = [1, 4, 5, 9, 20, 33, 46]
    system = gfp.System()
    for _ in range(47):
        system.addParticle(1.0)
    force = gfp.GridForce()
    force.addGridCounts(*c["counts"])
    force.addGridSpacing(*c["spacing"])
    force.setGridOrigin(*c["origin"])
    force.setGridValues(c["grids"][0])
    force.setScalingFactors(c["scaling"][0])
    force.setParticles(keep)
    system.addForce(force)
    ctx = gfp.Context(system, platform, {"Precision": "double"})
    ctx.setPositions(c["pos"])
    st = ctx.getState(getEnergy=True, getForces=True)
    port = oracle_built.PortOracle(c["counts"], c["spacing"], c["origin"], c["grids"][:1], c["scaling"][:1, keep], oob_k=c["oob_k"][:1])
    ge, f = port.execute_batched(np.ascontiguousarray(c["pos"][keep])[None])
    assert abs(st.getPotentialEnergy() - ge[0, 0]) <= 1e-12 * abs(ge[0, 0])
    got = st.getForces()
    assert np.abs(got[keep] - f[0]).max() <= 1e-12 * np.abs(f[0]).max()
    others = np.setdiff1d(np.arange(47), keep)
    assert not got[others].any()
    assert len(force.getParticleAtomEnergies(ctx)) == 0          # no particle groups: empty, as the reference
    # particle groups: per-atom energies in group order, summing to the group energies
    system2 = gfp.System()
    for _ in range(47):
        system2.addParticle(1.0)
    f2 = gfp.GridForce()
    f2.addGridCounts(*c["counts"])
    f2.addGridSpacing(*c["spacing"])
    f2.setGridOrigin(*c["origin"])
    f2.setGridValues(c["grids"][0])
    ga, gb = list(range(30, 47)), list(range(0, 12))
    f2.addParticleGroup("a", ga, list(c["scaling"][0][ga]))
    f2.addParticleGroup("b", gb, list(c["scaling"][0][gb]))
    system2.addForce(f2)
    ctx2 = gfp.Context(system2, platform, {"Precision": "double"})
    ctx2.setPositions(c["pos"])
    ctx2.getState(getEnergy=True, getForces=True)
    eg = f2.getParticleGroupEnergies(ctx2)
    ae = f2.getParticleAtomEnergies(ctx2)
    assert len(ae) == len(ga) + len(gb)
    assert abs(ae[:len(ga)].sum() - eg[0]) <= 1e-12 * np.abs(ae).sum() and abs(ae[len(ga):].sum() - eg[1]) <= 1e-12 * np.abs(ae).sum()
    order = ga + gb
    for j in (0, 5, len(ga), len(order) - 1):                    # spot-check single atoms against the oracle
        ia = order[j]
        p1 = oracle_built.PortOracle(c["counts"], c["spacing"], c["origin"], c["grids"][:1], c["scaling"][:1, ia:ia + 1], oob_k=c["oob_k"][:1])
        ge1, _ = p1.execute_batched(c["pos"][ia:ia + 1][None])
        assert abs(ae[j] - ge1[0, 0]) <= 1e-12 * max(abs(ge1[0, 0]), 1e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["mixed", "double"])
def test_batch_buffer_overloads(oracle_built, precision):
    """GridForceBatch's pointer overloads on caller-owned numpy buffers: E+F in float64 and float32, energy only, with
    pageable and page-locked (pinBuffer) arrays; all against the oracle and against the std::vector overloads."""
    import openmmgridforce_b200.gridforceplugin as gfp
    c, ref = cases.load_golden("ligand_three_grids")
    platform = gfp.Platform.getPlatformByName("B200")
    system, forces = _build_system(gfp, c)
    ctx = gfp.Context(system, platform, {"Precision": precision})
    rng = np.random.default_rng(4)
    r = 301
    pos = np.stack([c["pos"] + rng.uniform(-0.05, 0.05, size=3) for _ in range(r)])
    port = oracle_built.PortOracle(c["counts"], c["spacing"], c["origin"], c["grids"], c["scaling"], oob_k=c["oob_k"])
    ge_ref, f_ref = port.execute_batched(pos, n_threads=4)
    e_ref = ge_ref.sum(axis=1)
    te, tf = (1e-6, 1e-5) if precision == "mixed" else (1e-12, 1e-12)
    e_vec, f_vec = ctx.evaluateBatch(pos, precision=precision)
    en = np.full(r, np.nan)
    f64 = np.full(pos.shape, np.nan)
    ctx.evaluateBatchBuffers(pos, en, f64, precision=precision)
    assert np.abs(en - e_ref).max() <= te * max(np.abs(e_ref).max(), np.abs(ge_ref).max())
    assert np.abs(f64 - f_ref).max() <= tf * np.abs(f_ref).max()
    assert np.array_equal(f64, f_vec) and np.abs(en - e_vec).max() <= 1e-13 * np.abs(e_vec).max()
    f32 = np.full(pos.shape, np.nan, dtype=np.float32)
    gfp.pin_buffer(pos)
    gfp.pin_buffer(f32)
    try:
        en32 = np.zeros(r)
        ctx.evaluateBatchBuffers(pos, en32, f32, precision=precision)
    finally:
        gfp.pin_buffer(f32, False)
        gfp.pin_buffer(pos, False)
    assert np.abs(f32 - f_ref).max() <= max(tf, 1.2e-7) * np.abs(f_ref).max()
    assert np.abs(en32 - en).max() <= 1e-13 * np.abs(en).max()
    e_only = np.zeros(r)
    ctx.evaluateBatchBuffers(pos, e_only, None, precision=precision)
    assert np.abs(e_only - en).max() <= 1e-13 * np.abs(en).max()


def test_plugin_sources_compile_against_the_reference_headers():
    """`make plugin-check-reference`: the three platform sources compiled with the REFERENCE's openmmapi/include in place
    of the in-repo stand-ins (only where the original project's source tree is given by the REFERENCE_DIR environment
    variable)."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ref = os.environ.get("REFERENCE_DIR")
    if not ref or not os.path.isdir(os.path.join(ref, "openmmapi", "include")):
        pytest.skip("needs the original project's source tree (set REFERENCE_DIR)")
    out = subprocess.run(["make", "-C", root, "plugin-check-reference", f"REFERENCE_DIR={ref}"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
