"""GPU parity tests (-m gpu) of the evaluation variants added in round 2, each against the C oracle
(oracle/gridforce_oracle.c, bit-exact with the reference's ReferenceCalcGridForceKernel) on the same inputs:

  * energy-only launches (forces == NULL; CalcGridForceKernel::execute with includeForces == false,
    ReferenceGridForceKernels.cpp:646-648) in every record kernel and the general kernel;
  * FP32 force stores (GFB_FORCE_F32_STORE) through pinned (zero-copy) and pageable host buffers and on the device;
  * gf_eval_lines_f64_kernel — DOUBLE 256-byte records — at 1e-12;
  * evaluation order from the library's own counting sort (gfb_kernel_sort_atoms) through the record kernels;
  * per-atom energies (GridForce::getParticleAtomEnergies);
  * caller buffers page-locked with gfb_host_register; CUDA-graph replay of a launch sequence.

Tolerances (BASELINE.json north_star): MIXED energies 1e-6 relative, forces 1e-5 relative (max-norm); DOUBLE 1e-12.
"""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL = {0: (1e-6, 1e-5), 1: (1e-12, 1e-12)}


def _case(n_grids, n_replicas, n_atoms, seed, counts=(23, 19, 31), frac_outside=0.08):
    rng = np.random.default_rng(seed)
    sp, og = (0.05, 0.07, 0.04), (0.3, -0.2, 1.0)
    grids = [(rng.normal(size=counts) * 4).astype(np.float32).astype(np.float64) for _ in range(n_grids)]
    length = np.array(sp) * (np.array(counts) - 1)
    pos = np.array(og) + rng.uniform(0.0, 1.0, size=(n_replicas, n_atoms, 3)) * length
    out = rng.uniform(size=(n_replicas, n_atoms)) < frac_outside
    pos[out] += rng.choice([-1.0, 1.0], size=(int(out.sum()), 3)) * rng.uniform(0.0, 0.3, size=(int(out.sum()), 3)) * length
    sc = rng.normal(size=(n_grids, n_atoms))
    sc[:, ::7] = 0.0
    oob = [10000.0, 1234.0, 777.0, 5000.0][:n_grids]
    return dict(counts=counts, spacing=sp, origin=og, grids=grids, scaling=sc, pos=pos, oob_k=oob)


def _oracle(bindings, c):
    port = bindings.PortOracle(c["counts"], c["spacing"], c["origin"], c["grids"], c["scaling"], oob_k=c["oob_k"])
    return port.execute_batched(c["pos"], n_threads=4)           # ([R][G] energies, [R][A][3] forces)


def _make(gf, dev, c, precision=0, layout=None, particles=None):
    layout = gf.LAYOUT_CELLS if layout is None else layout
    grids = [gf.Grid(dev, c["counts"], c["spacing"], c["origin"], g, precision, layout=layout) for g in c["grids"]]
    return grids, gf.Kernel(dev, grids, c["scaling"], particles=particles, oob_k=c["oob_k"])


def _close(grids, k):
    k.close()
    for g in grids:
        g.close()


SHAPES = [(1, 5), (1, 300), (3, 47), (37, 47), (130, 9), (1, 4099)]


@pytest.mark.parametrize("shape", SHAPES, ids=[f"{r}x{a}" for r, a in SHAPES])
@pytest.mark.parametrize("n_grids", [2, 3, 4])
def test_double_record_kernel_vs_oracle(gpu_device, oracle_built, n_grids, shape):
    import openmmgridforce_b200 as gf
    r, a = shape
    c = _case(n_grids, r, a, seed=900 + 10 * n_grids + r + a)
    ge_ref, f_ref = _oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, precision=gf.PRECISION_DOUBLE)
    assert load_path(k) == 2
    en, forces, ge = k.execute_host(c["pos"], want_grid_energies=True)
    scale_e = np.abs(ge_ref).max()
    assert np.abs(ge - ge_ref).max() <= 1e-12 * scale_e
    assert np.abs(en - ge_ref.sum(axis=1)).max() <= 1e-12 * max(np.abs(ge_ref.sum(axis=1)).max(), scale_e)
    assert np.abs(forces - f_ref).max() <= 1e-12 * np.abs(f_ref).max()
    # accumulate onto existing forces, no per-grid energies (the other instantiation)
    f0 = np.random.default_rng(1).normal(size=c["pos"].shape)
    facc = f0.copy()
    en2, _, _ = k.execute_host(c["pos"], forces=facc, force_mode=gf.FORCE_F64_ADD)
    assert np.abs(en2 - ge_ref.sum(axis=1)).max() <= 1e-12 * max(np.abs(ge_ref.sum(axis=1)).max(), scale_e)
    assert np.abs(facc - f0 - f_ref).max() <= 1e-12 * np.abs(f_ref).max() + 1e-15 * np.abs(f0).max()
    # bit-exact classification (the DOUBLE kernels divide exactly as the reference does)
    port = oracle_built.PortOracle(c["counts"], c["spacing"], c["origin"], c["grids"], c["scaling"], oob_k=c["oob_k"])
    got = k.classify_host(c["pos"], 0)
    _, _, want = port.execute(c["pos"][0], 0, classify=True)
    assert np.array_equal(got["cell"][:a], want["cell"]) and np.array_equal(got["inside"][:a], want["inside"])
    _close(grids, k)


def load_path(k):
    import openmmgridforce_b200 as gf
    return int(gf.load_library().gfb_kernel_eval_path(k._h))


def test_double_record_kernel_device_fixed_point_and_upper_face(gpu_device, oracle_built):
    """Device path of the DOUBLE record kernel: OpenMM fixed-point forces over two launches, energies accumulated, next
    accumulator cleared; plus atoms exactly on the upper faces (last cell at fraction 1)."""
    import torch
    import openmmgridforce_b200 as gf
    r, a = 41, 47
    c = _case(3, r, a, seed=77)
    length = np.array(c["spacing"]) * (np.array(c["counts"]) - 1)
    c["pos"][0, 1] = np.array(c["origin"]) + length                       # corner of the box
    c["pos"][0, 2, 0] = c["origin"][0] + length[0]                        # on one upper face
    c["scaling"][:, 1] = 1.0
    c["scaling"][:, 2] = -0.5
    ge_ref, f_ref = _oracle(oracle_built, c)
    grids, k = _make(gf, gpu_device, c, precision=gf.PRECISION_DOUBLE)
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
    e_ref = ge_ref.sum(axis=1)
    assert np.abs(d_e.cpu().numpy() - 2 * e_ref).max() <= 1e-12 * 2 * max(np.abs(e_ref).max(), np.abs(ge_ref).max())
    # the fixed-point format itself resolves 2^-32 kJ/mol/nm
    assert np.abs(d_out.cpu().numpy().reshape(r, a, 3) - 2 * f_ref).max() <= 2 * 2.0 ** -32 + 1e-12 * np.abs(f_ref).max()
    assert not d_next.cpu().numpy().any()
    _close(grids, k)


@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
@pytest.mark.parametrize("n_grids", [1, 3])
@pytest.mark.parametrize("layout", ["cells", "rows"])
def test_energy_only_matches_energy_and_force_run(gpu_device, oracle_built, precision, n_grids, layout):
    """forces == NULL: the record kernels run their energy-only instantiation (no gradient arithmetic, no force
    read-modify-write), the general kernel skips the store. Energies must equal the oracle's and those of an E+F call."""
    import openmmgridforce_b200 as gf
    r, a = 53, 47
    c = _case(n_grids, r, a, seed=40 + n_grids)
    ge_ref, _ = _oracle(oracle_built, c)
    lay = gf.LAYOUT_CELLS if layout == "cells" else gf.LAYOUT_ROWS
    grids, k = _make(gf, gpu_device, c, precision=precision, layout=lay)
    te, _ = TOL[precision]
    en_f, f, _ = k.execute_host(c["pos"])
    en, none, ge = k.execute_host(c["pos"], want_forces=False, want_grid_energies=True)
    assert none is None
    scale = np.abs(ge_ref).max()
    assert np.abs(ge - ge_ref).max() <= te * scale
    assert np.abs(en - ge_ref.sum(axis=1)).max() <= te * max(scale, np.abs(ge_ref.sum(axis=1)).max())
    assert np.abs(en - en_f).max() <= 1e-13 * max(scale, 1.0)          # same FP64 value path, different atomics order
    _close(grids, k)


@pytest.mark.parametrize("buffers", ["pinned", "pageable", "registered"])
@pytest.mark.parametrize("n_grids", [1, 3])
def test_f32_force_store_host_path(gpu_device, oracle_built, n_grids, buffers):
    """GFB_FORCE_F32_STORE through gfb_kernel_execute_host: the lines kernel's warps emit 384-byte runs of float forces
    straight into page-locked caller memory (cudaHostAlloc or gfb_host_register), or into staging for pageable memory.
    Odd replica counts exercise the chunk boundaries; the F32 forces equal the F64_STORE forces rounded to float."""
    import torch
    import openmmgridforce_b200 as gf
    from openmmgridforce_b200 import workloads as W
    w = W.c5_sharded_replicas(n_local=9001, n=64)
    grids = [gf.Grid(gpu_device, w.counts, w.spacing, w.origin, v, gf.PRECISION_MIXED) for v in w.grids[:n_grids]]
    k = gf.Kernel(gpu_device, grids, w.scaling[:n_grids], oob_k=w.oob_k[:n_grids])
    port = oracle_built.PortOracle(w.counts, w.spacing, w.origin, w.grids[:n_grids], w.scaling[:n_grids], oob_k=w.oob_k[:n_grids])
    ge_ref, f_ref = port.execute_batched(w.pos, n_threads=8)
    e64, f64, _ = k.execute_host(w.pos)
    keep = []
    if buffers == "pinned":
        tp, tf = torch.from_numpy(w.pos.copy()).pin_memory(), torch.full(w.pos.shape, 7.0, dtype=torch.float32).pin_memory()
        pos, f32 = tp.numpy(), tf.numpy()
        keep = [tp, tf]
    else:
        pos, f32 = w.pos.copy(), np.full(w.pos.shape, 7.0, dtype=np.float32)
        if buffers == "registered":
            gf.host_register(pos)
            gf.host_register(f32)
    en, _, _ = k.execute_host(pos, forces=f32, force_mode=gf.FORCE_F32_STORE)
    if buffers == "registered":
        gf.host_unregister(pos)
        gf.host_unregister(f32)
    assert np.array_equal(f32, f64.astype(np.float32)), int((f32 != f64.astype(np.float32)).sum())
    assert np.abs(f32 - f_ref).max() <= 1e-5 * np.abs(f_ref).max()
    assert np.abs(en - ge_ref.sum(axis=1)).max() <= 1e-6 * max(np.abs(ge_ref).max(), np.abs(ge_ref.sum(axis=1)).max())
    assert np.abs(en - e64).max() <= 1e-13 * np.abs(e64).max()
    del keep
    k.close()
    for g in grids:
        g.close()


@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
def test_f32_force_store_other_kernels_and_subsets(gpu_device, oracle_built, precision):
    """F32 stores with a particle subset (entries of untouched particles stay as they were) through CELLS (the MIXED lines
    kernel / the DOUBLE record kernel) and ROWS (the general kernel). The B-spline and tricubic record kernels' F32 stores
    are checked in test_gpu_coverage.py::test_record_kernel_modes."""
    import openmmgridforce_b200 as gf
    rng = np.random.default_rng(8)
    r, n_particles, a = 7, 90, 60
    c = _case(3, r, n_particles, seed=13)
    particles = np.sort(rng.choice(n_particles, size=a, replace=False)).astype(np.int32)
    sc = rng.normal(size=(3, a))
    _, tf = TOL[precision]
    tf = max(tf, 1.2e-7)      # float output
    for layout in (gf.LAYOUT_CELLS, gf.LAYOUT_ROWS):
        grids = [gf.Grid(gpu_device, c["counts"], c["spacing"], c["origin"], g, precision, layout=layout) for g in c["grids"]]
        k = gf.Kernel(gpu_device, grids, sc, particles=particles, oob_k=c["oob_k"])
        port = oracle_built.PortOracle(c["counts"], c["spacing"], c["origin"], c["grids"], sc, oob_k=c["oob_k"])
        _, f_ref = port.execute_batched(np.ascontiguousarray(c["pos"][:, particles]), n_threads=2)
        forces = np.full(c["pos"].shape, 3.5, dtype=np.float32)
        k.execute_host(c["pos"], forces=forces, force_mode=gf.FORCE_F32_STORE)
        assert np.abs(forces[:, particles] - f_ref).max() <= tf * np.abs(f_ref).max()
        untouched = np.setdiff1d(np.arange(n_particles), particles)
        assert (forces[:, untouched] == 3.5).all()
        _close(grids, k)


def test_sort_atoms_is_a_permutation_and_order_is_honoured(gpu_device, oracle_built):
    """gfb_kernel_sort_atoms (own counting sort by 4^3-cell brick along a Morton curve): the result is a permutation,
    atoms of one brick are adjacent, outside atoms come last; evaluating in that order through the record kernels leaves
    bit-identical fixed-point forces and the same energies."""
    import torch
    import openmmgridforce_b200 as gf
    rng = np.random.default_rng(2)
    counts, sp, og = (70, 50, 90), (0.02, 0.03, 0.025), (0.1, 0.2, -0.3)
    r, a = 300, 47
    grids_v = [(rng.normal(size=counts) * 2).astype(np.float32).astype(np.float64) for _ in range(3)]
    length = np.array(sp) * (np.array(counts) - 1)
    pos = np.array(og) + rng.uniform(-0.03, 1.03, size=(r, a, 3)) * length
    sc = rng.uniform(0.5, 1.5, size=(3, a))
    c = dict(counts=counts, spacing=sp, origin=og, grids=grids_v, scaling=sc, pos=pos, oob_k=[10000.0] * 3)
    ge_ref, f_ref = _oracle(oracle_built, c)
    dev = torch.device("cuda:0")
    n = r * a
    stride = ((n + 31) // 32) * 32
    for precision in (gf.PRECISION_MIXED, gf.PRECISION_DOUBLE):
        grids, k = _make(gf, gpu_device, c, precision=precision)
        assert load_path(k) in (1, 2)
        d_pos = torch.from_numpy(pos).to(dev)
        d_order = torch.full((n,), -1, dtype=torch.int32, device=dev)
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        k.sort_atoms(r, a, d_pos.data_ptr(), d_order.data_ptr(), side.cuda_stream)
        torch.cuda.synchronize()
        order = d_order.cpu().numpy()
        assert np.array_equal(np.sort(order), np.arange(n))
        # brick keys along the order are non-decreasing; outside atoms last
        flat = pos.reshape(n, 3)[order]
        rel = flat - np.array(og)
        inside = ((rel >= 0) & (rel <= length)).all(axis=1)
        n_in = int(inside.sum())
        assert inside[:n_in].all() and not inside[n_in:].any()
        cell = np.minimum((rel[:n_in] / np.array(sp)).astype(np.int64), np.array(counts) - 2) >> 2

        def spread(v):
            out = np.zeros_like(v)
            for b in range(10):
                out |= ((v >> b) & 1) << (3 * b)
            return out
        key = (spread(cell[:, 0]) << 2) | (spread(cell[:, 1]) << 1) | spread(cell[:, 2])
        assert (np.diff(key) >= 0).all()
        res = []
        for use_order in (False, True):
            d_f = torch.zeros(3 * stride, dtype=torch.int64, device=dev)
            d_e = torch.zeros(r, dtype=torch.float64, device=dev)
            k.execute_device(r, a, d_pos.data_ptr(), d_e.data_ptr(), None, d_f.data_ptr(), gf.FORCE_FIXED_ADD, stride,
                             d_order.data_ptr() if use_order else None, side.cuda_stream)
            torch.cuda.synchronize()
            res.append((d_e.cpu().numpy(), d_f.cpu().numpy()))
        assert np.array_equal(res[0][1], res[1][1])
        assert np.abs(res[0][0] - res[1][0]).max() <= 1e-12 * np.abs(res[0][0]).max()
        te, _ = TOL[precision]
        assert np.abs(res[1][0] - ge_ref.sum(axis=1)).max() <= te * max(np.abs(ge_ref).max(), np.abs(ge_ref.sum(axis=1)).max())
        _close(grids, k)


@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
@pytest.mark.parametrize("n_grids", [1, 3])
def test_per_atom_energies(gpu_device, oracle_built, precision, n_grids):
    """gfb_kernel_request_atom_energies: per-atom energies (summed over the kernel's grids) against the oracle run on
    one-atom 'replicas' with that atom's scaling factor; their sum is the replica energy."""
    import openmmgridforce_b200 as gf
    r, a = 9, 47
    c = _case(n_grids, r, a, seed=60 + n_grids)
    grids, k = _make(gf, gpu_device, c, precision=precision)
    k.request_atom_energies(True)
    en, _, _ = k.execute_host(c["pos"])
    ae = k.atom_energies(r)
    te, _ = TOL[precision]
    want = np.zeros((r, a))
    for ia in range(a):
        port = oracle_built.PortOracle(c["counts"], c["spacing"], c["origin"], c["grids"], c["scaling"][:, ia:ia + 1], oob_k=c["oob_k"])
        ge1, _ = port.execute_batched(np.ascontiguousarray(c["pos"][:, ia:ia + 1]), n_threads=1)
        want[:, ia] = ge1.sum(axis=1)
    assert np.abs(ae - want).max() <= te * np.abs(want).max()
    assert np.abs(ae.sum(axis=1) - en).max() <= 1e-12 * np.abs(want).max() * a
    # the single-ligand (host-mapped) path
    en1, _, _ = k.execute_host(c["pos"][:1])
    ae1 = k.atom_energies(1)
    assert np.abs(ae1 - want[:1]).max() <= te * np.abs(want).max()
    k.request_atom_energies(False)
    _close(grids, k)


def test_cuda_graph_replay_matches_direct_launches(gpu_device):
    """gfb_graph_*: K evaluation launches (programmatic dependent launch on) captured once and replayed must leave the
    fixed-point forces of K direct launches, bit for bit, and the same energies."""
    import torch
    import openmmgridforce_b200 as gf
    from openmmgridforce_b200 import workloads as W
    w = W.c5_sharded_replicas(n_local=2048, n=64)
    grids = [gf.Grid(gpu_device, w.counts, w.spacing, w.origin, v, gf.PRECISION_MIXED) for v in w.grids]
    k = gf.Kernel(gpu_device, grids, w.scaling, oob_k=w.oob_k)
    k.set_launch_overlap(True)
    tdev = torch.device("cuda:0")
    r, a = w.n_replicas, w.n_atoms
    stride = ((r * a + 31) // 32) * 32
    rng = np.random.default_rng(5)
    sets = [torch.from_numpy(w.pos + rng.uniform(-0.01, 0.01, size=3)).to(tdev) for _ in range(3)]
    stream = torch.cuda.Stream()
    steps = 6

    def run(graph):
        d_f = torch.zeros(3 * stride, dtype=torch.int64, device=tdev)
        d_e = [torch.zeros(r, dtype=torch.float64, device=tdev) for _ in range(2)]
        torch.cuda.synchronize()

        def launches():
            for i in range(steps):
                k.execute_device(r, a, sets[i % 3].data_ptr(), d_e[i % 2].data_ptr(), None, d_f.data_ptr(), gf.FORCE_FIXED_ADD,
                                 stride, None, stream.cuda_stream, d_energies_clear=d_e[(i + 1) % 2].data_ptr())
        if graph:
            gf.Graph.begin(gpu_device, stream.cuda_stream)
            launches()
            g = gf.Graph.end(gpu_device, stream.cuda_stream)
            assert not d_f.cpu().numpy().any()            # capture records, it does not run
            g.launch(stream.cuda_stream)
            stream.synchronize()
            g.close()
        else:
            launches()
            stream.synchronize()
        return d_f.cpu().numpy(), d_e[(steps - 1) % 2].cpu().numpy()
    f0, e0 = run(False)
    f1, e1 = run(True)
    assert f0.any() and np.array_equal(f0, f1)
    assert np.abs(e0 - e1).max() <= 1e-13 * np.abs(e0).max()
    k.close()
    for g in grids:
        g.close()


def test_host_copy_probe_and_large_layout_refusal(gpu_device):
    import openmmgridforce_b200 as gf
    h2d, d2h, both = gpu_device.bench_host_copy(16 << 20, 3)
    assert 1.0 < h2d < 200.0 and 1.0 < d2h < 200.0 and both > 0.0
    # a 3000^3 grid cannot be repacked into B-spline records (32x the raw grid = 3.4 TB): the library says what does not
    # fit instead of returning a bare cudaMalloc error (the device pointer is never touched)
    import ctypes as C
    lib = gf.load_library()
    h = C.c_void_p()
    n = 3000
    rc = lib.gfb_grid_create_from_device(gpu_device._h, (C.c_int * 3)(n, n, n), (C.c_double * 3)(0.1, 0.1, 0.1),
                                         (C.c_double * 3)(0, 0, 0), C.c_void_p(0x1000), n ** 3, 0, gf.LAYOUT_BSPLINE, C.byref(h))
    assert rc == -4 and b"needs" in lib.gfb_last_error() and b"B-spline records" in lib.gfb_last_error()


@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
def test_release_cells_keeps_record_kernels_working(gpu_device, oracle_built, precision):
    """gfb_grid_release_cells: once a kernel over 2-4 grids has woven the packed cells into its records, the per-grid copies
    can be freed (3 x 192^3: 638 MB of 1.5 GB). The record kernels must give the same results afterwards, the grids must
    report zero device bytes, and building another kernel on a released grid must fail with a clear error instead of
    reading freed memory."""
    import openmmgridforce_b200 as gf
    from openmmgridforce_b200 import workloads as W
    w = W.c5_sharded_replicas(n_local=300, n=48)
    grids = [gf.Grid(gpu_device, w.counts, w.spacing, w.origin, v, precision) for v in w.grids]
    k = gf.Kernel(gpu_device, grids, w.scaling, oob_k=w.oob_k)
    assert k.eval_path() == (1 if precision == 0 else 2)
    e0, f0, _ = k.execute_host(w.pos)
    before = [g.device_bytes for g in grids]
    assert all(b > 0 for b in before)
    for g in grids:
        g.release_cells()
        g.release_cells()                      # idempotent
    assert all(g.device_bytes == 0 for g in grids)
    e1, f1, _ = k.execute_host(w.pos)
    assert np.array_equal(f0, f1) and np.abs(e0 - e1).max() <= 1e-13 * np.abs(e0).max()
    with pytest.raises(gf.GridForceB200Error, match="released its packed cells"):     # a new kernel would need them again
        gf.Kernel(gpu_device, grids[:1], w.scaling[:1], oob_k=w.oob_k[:1])
    k.close()
    for g in grids:
        g.close()


@pytest.mark.parametrize("precision", [0, 1], ids=["mixed", "double"])
@pytest.mark.parametrize("n_replicas", [2, 4, 5, 21, 87])
def test_small_batches_on_host_mapped_memory(gpu_device, oracle_built, n_replicas, precision):
    """gfb_kernel_execute_host with a handful of replicas (<= 4096 particles in all): one launch on host-mapped staging;
    up to 16 accumulators (4 replicas x 3 grids + totals) the energies are summed in the mapped array itself, beyond that
    on the device. Energies, per-grid energies, forces (STORE and ADD) and the energy-only call against the oracle."""
    import openmmgridforce_b200 as gf
    import sys as _sys
    _sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import cases
    c, _ = cases.load_golden("ligand_three_grids")
    rng = np.random.default_rng(n_replicas)
    pos = np.stack([c["pos"] + rng.uniform(-0.6, 0.6, size=3) for _ in range(n_replicas)])
    port = oracle_built.PortOracle(c["counts"], c["spacing"], c["origin"], c["grids"], c["scaling"], oob_k=c["oob_k"])
    ge_ref, f_ref = port.execute_batched(pos)
    grids = [gf.Grid(gpu_device, c["counts"], c["spacing"], c["origin"], g, precision) for g in c["grids"]]
    k = gf.Kernel(gpu_device, grids, c["scaling"], oob_k=c["oob_k"])
    te, tf = (1e-6, 1e-5) if precision == 0 else (1e-12, 1e-12)
    scale = np.maximum(np.abs(ge_ref.sum(axis=1)), np.abs(ge_ref).max(axis=1))
    for _ in range(3):                                   # repeated calls: accumulators start from zero every time
        en, f, ge = k.execute_host(pos, want_grid_energies=True)
        assert (np.abs(en - ge_ref.sum(axis=1)) <= te * scale).all()
        assert (np.abs(ge - ge_ref) <= te * scale[:, None]).all()
        assert np.abs(f - f_ref).max() <= tf * np.abs(f_ref).max()
    acc = np.ones_like(pos)
    k.execute_host(pos, forces=acc, force_mode=gf.FORCE_F64_ADD)
    assert np.abs(acc - (1.0 + f_ref)).max() <= tf * np.abs(f_ref).max()
    e0, none, _ = k.execute_host(pos, want_forces=False)
    assert none is None and (np.abs(e0 - ge_ref.sum(axis=1)) <= te * scale).all()
    # a run of calls without per-grid energies on moving poses (the two device accumulator arrays take turns and each
    # launch clears the other's totals), with a per-grid call and a smaller batch in between
    for step in range(6):
        p2 = pos + rng.uniform(-0.05, 0.05, size=3)
        g2, f2 = port.execute_batched(p2)
        s2 = np.maximum(np.abs(g2.sum(axis=1)), np.abs(g2).max(axis=1))
        if step == 3:
            en, f, ge = k.execute_host(p2, want_grid_energies=True)
            assert (np.abs(ge - g2) <= te * s2[:, None]).all()
        elif step == 4 and n_replicas > 2:
            en, f, _ = k.execute_host(p2[:-1])
            assert (np.abs(en - g2.sum(axis=1)[:-1]) <= te * s2[:-1]).all()
            continue
        else:
            en, f, _ = k.execute_host(p2)
        assert (np.abs(en - g2.sum(axis=1)) <= te * s2).all(), step
        assert np.abs(f - f2).max() <= tf * np.abs(f2).max()
    k.close()
    for g in grids:
        g.close()
