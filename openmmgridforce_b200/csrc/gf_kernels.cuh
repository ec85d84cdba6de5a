// Hand-written sm_100a kernels of the GridForce evaluation path.
//
// What is evaluated is the trilinear branch of the reference's Reference-platform kernel
// (platforms/reference/src/ReferenceGridForceKernels.cpp:646-1121); how it is evaluated is new:
//   * every stencil is read with aligned 32-byte loads (LDG.E.256, sm_100+): 4 (ROWS), 2 (PAIRS) or 1 (CELLS)
//     per stencil depending on the grid's layout, instead of 8 scattered 4-byte loads (reference CUDA kernel,
//     platforms/cuda/src/kernels/gridForce.cu:349-417);
//   * positions of a block are staged through shared memory with fully coalesced 16-byte loads;
//   * all grids acting on an atom (ele/LJr/LJa) are evaluated by the same thread in one pass, so the
//     position, the index math and the force write are paid once per atom, not once per grid;
//   * index/fraction math is FP64 and bit-exact with the reference (:687-715); interpolation is FP32 in
//     MIXED mode, FP64 in DOUBLE mode;
//   * energy: per-replica segmented warp reduction (__shfl_down_sync), one atomic per run of equal
//     replica ids per warp — or one per block when there is a single replica;
//   * forces: OpenMM 64-bit fixed point (RED.ADD.64, no return value), or doubles.
#ifndef GF_KERNELS_CUH_
#define GF_KERNELS_CUH_

#include <cuda_runtime.h>
#include <stdint.h>

#include "gf_params.h"

namespace gfb {

constexpr int kBlock = 256;
constexpr unsigned kFull = 0xffffffffu;

// ------------------------------------------------------------------------------------------------
// Classification: inside test + cell index + in-cell fraction for one axis.
// Reference: pi = pos - origin (:687-688); inside iff 0 <= pi <= hCorner (:690-696, upper face
// inclusive); ix = (int)(pi/spacing), f = pi/spacing - ix (:708-715, true FP64 division).
//
// The quotient is first formed as pi * fl(1/spacing) (one DMUL instead of a ~10-instruction IEEE
// division). That product is within 2^-51 relative of the correctly rounded quotient, so its
// truncation can only differ when an integer lies within that distance; in that (probability ~1e-13)
// case the division is redone exactly. EXACT=true (DOUBLE mode) always divides, so the fraction is the
// reference's bit for bit as well.
// ------------------------------------------------------------------------------------------------
// IEEE division kept out of line: ptxas otherwise if-converts the rare branch below and runs the ~12-instruction
// FP64 division sequence for every atom on every axis.
static __device__ __noinline__ double exact_quotient(double pi, double spacing) { return pi / spacing; }

template <bool EXACT>
__device__ __forceinline__ void axis_index(double pi, double spacing, double inv_spacing, int ncell,
                                           int& idx, double& frac) {
    double q;
    if (EXACT) {
        q = pi / spacing;
    } else {
        q = pi * inv_spacing;
        const double r = rint(q);
        if (fabs(q - r) <= 1.8e-15 * fmax(q, 1.0)) q = exact_quotient(pi, spacing);
    }
    int i = __double2int_rz(q);
    // pi == hCorner gives i == ncell (== counts-1): the reference then reads past the grid (UB, its
    // quirk Q2). Evaluate the last cell at fraction 1 instead — the limit from inside.
    i = min(i, ncell - 1);
    idx = i;
    frac = q - (double) i;
}

struct AtomCell {
    int ix, iy, iz;
    double fx, fy, fz;     // in-cell fractions
    bool inside;
};

template <bool EXACT>
__device__ __forceinline__ AtomCell classify(const GridView& g, double x, double y, double z) {
    AtomCell c;
    const double px = x - g.origin[0];
    const double py = y - g.origin[1];
    const double pz = z - g.origin[2];
    c.inside = (px >= 0.0 && px <= g.hcorner[0]) && (py >= 0.0 && py <= g.hcorner[1]) &&
               (pz >= 0.0 && pz <= g.hcorner[2]);
    c.ix = c.iy = c.iz = 0;
    c.fx = c.fy = c.fz = 0.0;
    if (c.inside) {
        axis_index<EXACT>(px, g.spacing[0], g.inv_spacing[0], g.nc[0], c.ix, c.fx);
        axis_index<EXACT>(py, g.spacing[1], g.inv_spacing[1], g.nc[1], c.iy, c.fy);
        axis_index<EXACT>(pz, g.spacing[2], g.inv_spacing[2], g.nc[2], c.iz, c.fz);
    }
    return c;
}

// ------------------------------------------------------------------------------------------------
// 32-byte aligned load = one L2 sector = one LDG.E.256: the unit every layout is built from.
// .nc: the grid is read-only for the life of the kernel. L2::evict_last: the grid is the only data
// with reuse across atoms/steps; positions and forces stream through.
// ------------------------------------------------------------------------------------------------
// The stencil load carries the L2 prefetch-size hint .L2::64B (SASS LDG.E.ELL2.LTC64B.256): measured on C3 (one random
// 32-byte stencil per atom out of 530 MB of packed cells) against no hint / .L2::128B in A/B builds
// (-DGFB_STENCIL_LD_VARIANT=0/2/3): FIXED_ADD 31.8 -> 29.8 us, F32 stores 25.4 -> 24.2 us.
#ifndef GFB_STENCIL_LD_VARIANT
#define GFB_STENCIL_LD_VARIANT 1
#endif
#if GFB_STENCIL_LD_VARIANT == 0
#define GFB_STENCIL_LD "ld.global.nc.L2::evict_last.v8.f32"
#elif GFB_STENCIL_LD_VARIANT == 1
#define GFB_STENCIL_LD "ld.global.nc.L2::evict_last.L2::64B.v8.f32"
#elif GFB_STENCIL_LD_VARIANT == 2
#define GFB_STENCIL_LD "ld.global.nc.L2::evict_last.L2::128B.v8.f32"
#elif GFB_STENCIL_LD_VARIANT == 3
#define GFB_STENCIL_LD "ld.global.nc.v8.f32"
#else
#define GFB_STENCIL_LD "ld.global.nc.L2::64B.v8.f32"
#endif
__device__ __forceinline__ void load32(const float* p, float v[8]) {
    asm volatile(GFB_STENCIL_LD " {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                 : "l"(p));
}
__device__ __forceinline__ void load32(const double* p, double v[4]) {
    asm volatile("ld.global.nc.L2::evict_last.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3])
                 : "l"(p));
}
__device__ __forceinline__ void load_cell(const float* p, float v[8]) { load32(p, v); }
__device__ __forceinline__ void load_cell(const double* p, double v[8]) {
    load32(p, v);
    load32(p + 4, v + 4);
}

// (c[o], c[o+1]) for a per-lane offset o in [0, W-2]: compare/select chain, no local memory.
template <typename S, int W>
__device__ __forceinline__ void pick_pair(const S* c, int o, S& a, S& b) {
    a = c[0];
    b = c[1];
#pragma unroll
    for (int k = 1; k < W - 1; k++)
        if (o == k) {
            a = c[k];
            b = c[k + 1];
        }
}

// The 8 corners {v000,v001,v010,v011,v100,v101,v110,v111} (last index z) of cell (ix,iy,iz).
template <typename S, int LAYOUT>
__device__ __forceinline__ void load_stencil(const GridView& G, int ix, int iy, int iz, S v[8]) {
    const S* base = static_cast<const S*>(G.cells);
    if constexpr (LAYOUT == GFB_LAYOUT_CELLS) {
        const size_t cell = ((size_t) ix * G.nc[1] + iy) * G.nc[2] + iz;
        load_cell(base + (size_t) G.cell_stride * cell, v);
    } else if constexpr (LAYOUT == GFB_LAYOUT_ROWS) {
        constexpr int W = 32 / (int) sizeof(S);     // values per chunk; consecutive chunks advance by W-1
        const int j = iz / (W - 1);
        const int o = iz - j * (W - 1);
        const int ny = G.nc[1] + 1;
        const size_t row = (size_t) ix * ny + iy;
        const S* p00 = base + (row * G.row_chunks + j) * W;
        const size_t dy = (size_t) G.row_chunks * W, dx = dy * ny;
        S c0[W], c1[W], c2[W], c3[W];
        load32(p00, c0);
        load32(p00 + dy, c1);
        load32(p00 + dx, c2);
        load32(p00 + dx + dy, c3);
        pick_pair<S, W>(c0, o, v[0], v[1]);
        pick_pair<S, W>(c1, o, v[2], v[3]);
        pick_pair<S, W>(c2, o, v[4], v[5]);
        pick_pair<S, W>(c3, o, v[6], v[7]);
    } else {  // PAIRS (float only): entry = {row iy: z=3j..3j+3 | row iy+1: z=3j..3j+3}
        const int j = iz / 3;
        const int o = iz - 3 * j;
        const size_t ent = ((size_t) ix * G.nc[1] + iy) * G.row_chunks + j;
        const size_t dx = (size_t) G.nc[1] * G.row_chunks * 8;
        S e0[8], e1[8];
        load_cell(base + ent * 8, e0);
        load_cell(base + ent * 8 + dx, e1);
        pick_pair<S, 4>(e0, o, v[0], v[1]);
        pick_pair<S, 4>(e0 + 4, o, v[2], v[3]);
        pick_pair<S, 4>(e1, o, v[4], v[5]);
        pick_pair<S, 4>(e1 + 4, o, v[6], v[7]);
    }
}

// Positions are read once per step: stream them (evict-first) so they do not displace grid sectors.
__device__ __forceinline__ double load_stream(const double* p) {
    double v;
    asm volatile("ld.global.cs.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}

// ------------------------------------------------------------------------------------------------
// Trilinear value and analytic gradient, in the reference's evaluation order (z -> y -> x, :1044-1053;
// gradient :1066-1071). v[] = {v000,v001,v010,v011,v100,v101,v110,v111}, last index z.
// ------------------------------------------------------------------------------------------------
template <typename C>
__device__ __forceinline__ void trilinear(const C v[8], C fx, C fy, C fz, C& val, C& dx, C& dy, C& dz) {
    const C one = (C) 1;
    const C ax = one - fx, ay = one - fy, az = one - fz;
    const C vmm = az * v[0] + fz * v[1];
    const C vmp = az * v[2] + fz * v[3];
    const C vpm = az * v[4] + fz * v[5];
    const C vpp = az * v[6] + fz * v[7];
    const C vm = ay * vmm + fy * vmp;
    const C vp = ay * vpm + fy * vpp;
    val = ax * vm + fx * vp;
    if constexpr (sizeof(C) == 4) {
        // MIXED: the stored corners are differenced first, as dz is. vp - vm subtracts two rounded lerps of size |V|, so
        // its error grows with |V| (a field C + noise loses digits in proportion to C); a difference of two nearby FP32
        // corners is exact or nearly so, which leaves an error proportional to |grad V| * spacing.
        dx = ((v[4] - v[0]) * az + (v[5] - v[1]) * fz) * ay + ((v[6] - v[2]) * az + (v[7] - v[3]) * fz) * fy;
        dy = ((v[2] - v[0]) * az + (v[3] - v[1]) * fz) * ax + ((v[6] - v[4]) * az + (v[7] - v[5]) * fz) * fx;
    } else {   // DOUBLE: the reference's expressions (:1066-1068)
        dx = vp - vm;
        dy = (vmp - vmm) * ax + (vpp - vpm) * fx;
    }
    dz =((v[1] - v[0]) * ay + (v[3] - v[2]) * fy) * ax + ((v[5] - v[4]) * ay + (v[7] - v[6]) * fy) * fx;
}

// MIXED mode energy path: the interpolated VALUE is formed in FP64 from the FP32-stored corners and the FP64
// fractions (7 lerps, z -> y -> x as :1044-1053). A replica's energy is a sum of terms of both signs, so FP32
// rounding of each term (6e-8 of |s*v|) would not meet 1e-6 of the much smaller total; in FP64 the only error left
// is the FP32 rounding of the stored grid values. The kernel is memory-bound: the ~25 extra FP64 ops are hidden.
__device__ __forceinline__ double trilinear_value_f64(const float v[8], double fx, double fy, double fz) {
    const double ax = 1.0 - fx, ay = 1.0 - fy, az = 1.0 - fz;
    const double vmm = az * (double) v[0] + fz * (double) v[1];
    const double vmp = az * (double) v[2] + fz * (double) v[3];
    const double vpm = az * (double) v[4] + fz * (double) v[5];
    const double vpp = az * (double) v[6] + fz * (double) v[7];
    const double vm = ay * vmm + fy * vmp;
    const double vp = ay * vpm + fy * vpp;
    return ax * vm + fx * vp;
}
__device__ __forceinline__ double trilinear_value_f64(const double*, double, double, double) { return 0.0; }  // unused (DOUBLE)

// Number of lanes that follow `lane` inside its run of equal keys (runs = maximal stretches of consecutive lanes with
// the same key). `heads` gets the ballot of run heads. Equal keys that are not adjacent form separate runs, which is
// still correct: each run issues its own atomic.
__device__ __forceinline__ unsigned run_span(int key, unsigned lane, unsigned& heads) {
    const int kprev = __shfl_up_sync(kFull, key, 1);
    heads = __ballot_sync(kFull, lane == 0 || kprev != key);
    const unsigned above = (heads >> 1) >> lane;   // bit i: lane+1+i starts a new run
    return above ? (unsigned) __ffs((int) above) - 1u : 31u - lane;
}

// Segmented sum over a run; the total lands in the run's first lane.
__device__ __forceinline__ void run_sum(double& e, unsigned span) {
#pragma unroll
    for (unsigned off = 1; off < 32; off <<= 1) {
        const double ev = __shfl_down_sync(kFull, e, off);
        if (off <= span) e += ev;
    }
}

__device__ __forceinline__ void red_add_f64(double* addr, double v) {
    asm volatile("red.global.add.f64 [%0], %1;" ::"l"(addr), "d"(v) : "memory");
}
__device__ __forceinline__ void red_add_u64(unsigned long long* addr, unsigned long long v) {
    asm volatile("red.global.add.u64 [%0], %1;" ::"l"(addr), "l"(v) : "memory");
}

// ------------------------------------------------------------------------------------------------
// The evaluation kernel. One thread per atom; that thread evaluates every grid.
//   S      stored corner type (float MIXED / double DOUBLE); also the interpolation type
//   LAYOUT gfb_layout of every grid of this launch
//   NG     number of grids when > 0 (fully unrolled), 0 = runtime p.n_grids
//   SAME   all grids share counts/spacing/origin: classify once
//   SINGLE one replica: block-level energy reduction, one atomic per block
// The force mode (gfb_force_mode) is a run-time, launch-uniform switch here (p.force_mode): this kernel is the general
// path, and one instantiation per mode tripled the library's build time for nothing measurable.
// ------------------------------------------------------------------------------------------------
// Occupancy: the kernel waits on DRAM/L2 round trips, so resident warps are what hides them. ptxas fits the
// one-grid kernel in 40 registers (6 blocks = 1536 threads per SM) and the three-grid kernel in 64 (4 blocks)
// without meaningful spills; left alone it takes 46 / 78 registers and occupancy drops to 5 / 3 blocks.

// One grid's contribution for an atom whose stencil v[] is already in registers (:1039-1082).
template <typename S>
__device__ __forceinline__ void accumulate_inside(const GridView& G, const S v[8], const AtomCell& c, double sd,
                                                  double& e_g, double& Fx, double& Fy, double& Fz) {
    constexpr bool EXACT = sizeof(S) == 8;
    S val, dx, dy, dz;
    trilinear<S>(v, (S) c.fx, (S) c.fy, (S) c.fz, val, dx, dy, dz);
    double gx, gy, gz;
    if (EXACT) {  // DOUBLE: divide, as the reference does (:1072)
        gx = (double) dx / G.spacing[0];
        gy = (double) dy / G.spacing[1];
        gz = (double) dz / G.spacing[2];
    } else {
        gx = (double) (dx * (S) G.inv_spacing[0]);
        gy = (double) (dy * (S) G.inv_spacing[1]);
        gz = (double) (dz * (S) G.inv_spacing[2]);
    }
    double dval = EXACT ? (double) val : trilinear_value_f64(v, c.fx, c.fy, c.fz);
    if (G.inv_power > 0.0) {  // :1057-1059, :1076-1080 (plain pow: NaN for a negative base, as the oracle)
        const double base = dval;
        dval = pow(base, G.inv_power);
        const double pf = G.inv_power * pow(base, G.inv_power - 1.0);
        gx *= pf;
        gy *= pf;
        gz *= pf;
    }
    e_g = sd * dval;  // :1061
    Fx -= sd * gx;    // :1082
    Fy -= sd * gy;
    Fz -= sd * gz;
}

// ------------------------------------------------------------------------------------------------
// Cubic B-spline interpolation (GridForce::setInterpolationMethod(1); ReferenceGridForceKernels.cpp:727-795):
// 4x4x4 points ix-1..ix+2 (indices clamped into the grid), separable weights bx[i]*by[j]*bz[k].
//
// Layout GFB_LAYOUT_BSPLINE (gf_repack_bspline_kernel) — the "brick" layout SURVEY.md §8f anticipates: the clamping is
// baked into a padded copy P[a][b][c] = V[clamp(a-1)][clamp(b-1)][clamp(c-1)], so the stencil of cell (ix,iy,iz) is
// P[ix..ix+3][iy..iy+3][iz..iz+3]. For EVERY cell (iy,iz) and every padded plane a <= nx, the two 4x4 (y,z) windows
// P[a][iy..iy+3][iz..iz+3] and P[a+1][..][..] are stored back to back as one record of 2 x 16 values (128 bytes of floats
// = exactly one L2/HBM line, 256 bytes of doubles), z fastest: record (a, iy, iz) at ((a*(ny-1) + iy)*(nz-1) + iz).
// A stencil is the TWO records a = ix and a = ix+2: 8 aligned 32-byte loads (16 in FP64) of exactly the 64 values it
// needs, in two full lines — no unaligned windows, no zero-padded weights, no partly used lines — instead of 64
// scattered 4-byte loads to 16 lines (reference CUDA kernel, gridForce.cu:103-147). Copy size: 32x the raw grid
// (192^3: 906 MB). Earlier layouts, for the record: tiles of 4 rows x 8 z-values advancing by 5 (6.4x; twice the bytes
// per stencil, half of the FMAs on zero weights) and single 64-byte bricks (16x; a brick still cost 89 bytes of DRAM).
//
// Arithmetic: S = double -> everything FP64. S = float -> gradient FP32, interpolated VALUE FP64 from the FP32-stored
// points and FP64 weights (same reasoning as trilinear_value_f64). The FP32 gradient sums run over the points minus the
// stencil's first point `ref`: each axis's derivative weights sum to 0, so the result is the same in exact arithmetic,
// but the rounding error then scales with the spread of the stencil (|grad V| * spacing) instead of with |V|.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void bspline_basis(double t, double b[4], double d[4]) {   // :54-63
    const double u = 1.0 - t, t2 = t * t, t3 = t2 * t;
    const double sixth = 1.0 / 6.0;
    b[0] = u * u * u * sixth;
    b[1] = (3.0 * t3 - 6.0 * t2 + 4.0) * sixth;
    b[2] = (-3.0 * t3 + 3.0 * t2 + 3.0 * t + 1.0) * sixth;
    b[3] = t3 * sixth;
    d[0] = -u * u * 0.5;
    d[1] = (3.0 * t2 - 4.0 * t) * 0.5;
    d[2] = (-3.0 * t2 + 2.0 * t + 1.0) * 0.5;
    d[3] = t2 * 0.5;
}

// The 16 values [row][z] of one brick.
__device__ __forceinline__ void load_brick(const float* p, float v[16]) {
    load32(p, v);
    load32(p + 8, v + 8);
}
__device__ __forceinline__ void load_brick(const double* p, double v[16]) {
    load32(p, v);
    load32(p + 4, v + 4);
    load32(p + 8, v + 8);
    load32(p + 12, v + 12);
}

template <typename S>
__device__ __forceinline__ void bspline_interpolate(const GridView& G, int ix, int iy, int iz, double fx, double fy, double fz,
                                                    double& val, S& gx, S& gy, S& gz) {
    constexpr bool F64 = sizeof(S) == 8;
    double bx[4], dbx[4], by[4], dby[4], bz[4], dbz[4];
    bspline_basis(fx, bx, dbx);   // :741-748
    bspline_basis(fy, by, dby);
    bspline_basis(fz, bz, dbz);
    const S* rec = static_cast<const S*>(G.cells) + (((size_t) ix * G.nc[1] + iy) * G.nc[2] + iz) * 32;
    const size_t plane2 = (size_t) G.nc[1] * G.nc[2] * 64;    // records two x-planes further on
    val = 0.0;
    gx = gy = gz = (S) 0;
    S ref = (S) 0;                // MIXED: the stencil's first point, subtracted in the FP32 gradient sums
#pragma unroll
    for (int i = 0; i < 4; i++) {
        S v[16];
        load_brick(rec + (i >> 1) * plane2 + (i & 1) * 16, v);   // planes ix, ix+1 | ix+2, ix+3
        if (!F64 && i == 0) ref = v[0];
        double pv = 0.0;          // sum over (j,k) of by*bz*V in this x-plane
        S pdy = (S) 0, pdz = (S) 0;
#pragma unroll
        for (int r = 0; r < 4; r++) {
            double rz = 0.0;
            S rzs = (S) 0, drz = (S) 0;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const S d = F64 ? v[4 * r + k] : v[4 * r + k] - ref;
                rz = fma(bz[k], (double) v[4 * r + k], rz);
                if (!F64) rzs = fma((S) bz[k], d, rzs);
                drz = fma((S) dbz[k], d, drz);
            }
            if (F64) rzs = (S) rz;
            pv = fma(by[r], rz, pv);
            pdy = fma((S) dby[r], rzs, pdy);
            pdz = fma((S) by[r], drz, pdz);
        }
        val = fma(bx[i], pv, val);
        gx = fma((S) dbx[i], F64 ? (S) pv : (S) (pv - (double) ref), gx);
        gy = fma((S) bx[i], pdy, gy);
        gz = fma((S) bx[i], pdz, gz);
    }
}

// The same sums over the raw points (GFB_LAYOUT_BSPLINE_POINTS), indices clamped when they are formed as the reference
// does (:754-775): 64 scalar loads per stencil, 1/64 of the records' memory — the fallback for grids whose records do
// not fit. The atom's cell comes from classify(), which maps the upper face to (n-2, fraction 1); the reference uses
// (n-1, fraction 0) there: the same 4x4x4 polynomial on the clamped neighbourhood (DESIGN.md, deviations table).
template <typename S>
__device__ __forceinline__ void bspline_interpolate_points(const GridView& G, int ix, int iy, int iz, double fx, double fy, double fz,
                                                           double& val, S& gx, S& gy, S& gz) {
    constexpr bool F64 = sizeof(S) == 8;
    double bx[4], dbx[4], by[4], dby[4], bz[4], dbz[4];
    bspline_basis(fx, bx, dbx);
    bspline_basis(fy, by, dby);
    bspline_basis(fz, bz, dbz);
    const int nx = G.nc[0] + 1, ny = G.nc[1] + 1, nz = G.nc[2] + 1;
    const S* base = static_cast<const S*>(G.cells);
    int zi[4];
#pragma unroll
    for (int k = 0; k < 4; k++) zi[k] = min(max(iz - 1 + k, 0), nz - 1);
    val = 0.0;
    gx = gy = gz = (S) 0;
    S ref = (S) 0;                // MIXED: the stencil's first point, as in bspline_interpolate
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const size_t px = (size_t) min(max(ix - 1 + i, 0), nx - 1) * ny;
        double pv = 0.0;
        S pdy = (S) 0, pdz = (S) 0;
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const S* row = base + (px + (size_t) min(max(iy - 1 + r, 0), ny - 1)) * nz;
            double rz = 0.0;
            S rzs = (S) 0, drz = (S) 0;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const S v = __ldg(row + zi[k]);
                if (!F64 && i == 0 && r == 0 && k == 0) ref = v;
                const S d = F64 ? v : v - ref;
                rz = fma(bz[k], (double) v, rz);
                if (!F64) rzs = fma((S) bz[k], d, rzs);
                drz = fma((S) dbz[k], d, drz);
            }
            if (F64) rzs = (S) rz;
            pv = fma(by[r], rz, pv);
            pdy = fma((S) dby[r], rzs, pdy);
            pdz = fma((S) by[r], drz, pdz);
        }
        val = fma(bx[i], pv, val);
        gx = fma((S) dbx[i], F64 ? (S) pv : (S) (pv - (double) ref), gx);
        gy = fma((S) bx[i], pdy, gy);
        gz = fma((S) bx[i], pdz, gz);
    }
}

// One grid's B-spline contribution for an inside atom (:727-795), same epilogue as accumulate_inside.
template <typename S, int LAYOUT = GFB_LAYOUT_BSPLINE>
__device__ __forceinline__ void accumulate_bspline(const GridView& G, const AtomCell& c, double sd, double& e_g, double& Fx,
                                                   double& Fy, double& Fz) {
    constexpr bool EXACT = sizeof(S) == 8;
    double dval;
    S dx, dy, dz;
    if constexpr (LAYOUT == GFB_LAYOUT_BSPLINE_POINTS) bspline_interpolate_points<S>(G, c.ix, c.iy, c.iz, c.fx, c.fy, c.fz, dval, dx, dy, dz);
    else bspline_interpolate<S>(G, c.ix, c.iy, c.iz, c.fx, c.fy, c.fz, dval, dx, dy, dz);
    double gx, gy, gz;
    if (EXACT) {  // :790
        gx = (double) dx / G.spacing[0];
        gy = (double) dy / G.spacing[1];
        gz = (double) dz / G.spacing[2];
    } else {
        gx = (double) (dx * (S) G.inv_spacing[0]);
        gy = (double) (dy * (S) G.inv_spacing[1]);
        gz = (double) (dz * (S) G.inv_spacing[2]);
    }
    if (G.inv_power > 0.0) {  // :778-787
        const double base = dval;
        dval = pow(base, G.inv_power);
        const double pf = G.inv_power * pow(base, G.inv_power - 1.0);
        gx *= pf;
        gy *= pf;
        gz *= pf;
    }
    e_g = sd * dval;  // :793
    Fx -= sd * gx;    // :794
    Fy -= sd * gy;
    Fz -= sd * gz;
}

// ------------------------------------------------------------------------------------------------
// Tricubic Hermite interpolation (GridForce::setInterpolationMethod(2); ReferenceGridForceKernels.cpp:796-893): cubic
// Hermite along x on the cell's four x-edges with centred-difference x-derivatives, then along y and along z with
// one-sided differences of the partly interpolated values against the value-basis interpolant of the neighbour rows.
// 32 of the 64 points ix-1..ix+2 x iy-1..iy+2 x iz-1..iz+2 are read: 16 on the four x-lines of the cell's edges, 8 in
// the rows iy-1 / iy+2, 8 at iz-1 / iz+2. What the reference does and a derivation from scratch would not is kept:
// dvdy comes from the z = iz plane only (:863), and a derivative estimate is 0 in the first cell layer of its axis.
//
// Layout GFB_LAYOUT_POINTS: the raw x-major array in S plus one zero x-slab. The reference addresses the neighbours by
// flat index without clamping (:817-867), so in the last y / z cell they are the first values of the next row / slab;
// the same flat indices are formed here. In the last x layer its reads leave the vector (undefined); here they hit the
// zero slab. Lower neighbours are only read where the reference reads them (ix, iy, iz > 0): nothing precedes the array.
// Per stencil 12 (x,y) rows are touched, 2 or 4 consecutive z-values each: 12-16 sectors.
// Arithmetic FP64 for both storage types; d*spacing products of the reference ((v1 - v0)/(2s) * s) are formed as
// 0.5*(v1 - v0), equal to rounding.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void hermite_basis(double t, double h[4], double d[4]) {   // :68-77; order h00, h01, h10, h11
    const double u = 1.0 - t, t2 = t * t;
    h[0] = (1.0 + 2.0 * t) * u * u;
    h[1] = t2 * (3.0 - 2.0 * t);
    h[2] = t * u * u;
    h[3] = t2 * (t - 1.0);
    d[0] = 6.0 * t2 - 6.0 * t;
    d[1] = -d[0];
    d[2] = 3.0 * t2 - 4.0 * t + 1.0;
    d[3] = 3.0 * t2 - 2.0 * t;
}

// The arithmetic of :806-876 over an accessor V(i, r, k) = the point at offsets (i-1, r-1, k-1) from (ix, iy, iz),
// i, r, k in 0..3 — always called with literal indices, so an accessor over registers costs nothing. Lower neighbours
// (index 0) are only touched when xin / yin / zin hold, as in the reference.
struct TricubicWeights {
    double hx[4], dhx[4], hy[4], dhy[4], hz[4], dhz[4];
};
__device__ __forceinline__ void tricubic_weights(double fx, double fy, double fz, TricubicWeights& w) {
    hermite_basis(fx, w.hx, w.dhx);
    hermite_basis(fy, w.hy, w.dhy);
    hermite_basis(fz, w.hz, w.dhz);
}
template <typename Acc>
__device__ __forceinline__ void tricubic_eval(const Acc& V, bool xin, bool yin, bool zin, const TricubicWeights& w, double& val,
                                              double& gx, double& gy, double& gz) {
    const double* hx = w.hx;
    const double* hy = w.hy;
    // x: the four edges (iy+j, iz+k), :806-846
    double vv[2][2], dv[2][2];
#pragma unroll
    for (int j = 0; j < 2; j++) {
#pragma unroll
        for (int k = 0; k < 2; k++) {
            const double f0 = V(1, 1 + j, 1 + k), f1 = V(2, 1 + j, 1 + k);
            double d0 = 0.0, d1 = 0.0;   // derivative x spacing at ix and ix+1
            if (xin) {
                d0 = 0.5 * (f1 - V(0, 1 + j, 1 + k));
                d1 = 0.5 * (V(3, 1 + j, 1 + k) - f0);
            }
            vv[j][k] = hx[0] * f0 + hx[1] * f1 + hx[2] * d0 + hx[3] * d1;
            dv[j][k] = w.dhx[0] * f0 + w.dhx[1] * f1 + w.dhx[2] * d0 + w.dhx[3] * d1;
        }
    }
    // y: rows iy-1 and iy+2 interpolated in x with the value basis only, :849-863
    double vk[2], dxk[2], dvdy = 0.0;
#pragma unroll
    for (int k = 0; k < 2; k++) {
        double dy0 = 0.0, dy1 = 0.0;
        if (yin) {
            const double rm = hx[0] * V(1, 0, 1 + k) + hx[1] * V(2, 0, 1 + k);
            const double rp = hx[0] * V(1, 3, 1 + k) + hx[1] * V(2, 3, 1 + k);
            dy0 = vv[1][k] - rm;
            dy1 = rp - vv[0][k];
        }
        vk[k] = hy[0] * vv[0][k] + hy[1] * vv[1][k] + hy[2] * dy0 + hy[3] * dy1;
        dxk[k] = hy[0] * dv[0][k] + hy[1] * dv[1][k];
        if (k == 0) dvdy = w.dhy[0] * vv[0][0] + w.dhy[1] * vv[1][0] + w.dhy[2] * dy0 + w.dhy[3] * dy1;   // z = iz plane only, :863
    }
    // z: points iz-1 and iz+2 interpolated in x and y with the value basis only, :866-876
    double dz0 = 0.0, dz1 = 0.0;
    if (zin) {
        const double zm = hy[0] * (hx[0] * V(1, 1, 0) + hx[1] * V(2, 1, 0)) + hy[1] * (hx[0] * V(1, 2, 0) + hx[1] * V(2, 2, 0));
        const double zp = hy[0] * (hx[0] * V(1, 1, 3) + hx[1] * V(2, 1, 3)) + hy[1] * (hx[0] * V(1, 2, 3) + hx[1] * V(2, 2, 3));
        dz0 = vk[1] - zm;
        dz1 = zp - vk[0];
    }
    val = w.hz[0] * vk[0] + w.hz[1] * vk[1] + w.hz[2] * dz0 + w.hz[3] * dz1;          // :873
    gx = w.hz[0] * dxk[0] + w.hz[1] * dxk[1];                                          // :875
    gy = dvdy;
    gz = w.dhz[0] * vk[0] + w.dhz[1] * vk[1] + w.dhz[2] * dz0 + w.dhz[3] * dz1;       // :876
}

// POINTS: scalar reads by flat index.
template <typename S>
struct TricubicPoints {
    const S* v;          // &V[im]
    long long nz, nyz;
    __device__ __forceinline__ double operator()(int i, int r, int k) const {
        return (double) __ldg(v + (i - 1) * nyz + (r - 1) * nz + (k - 1));
    }
};
// HERMITE records read into registers: b[i][4 * r + k] (load_brick order).
template <typename S>
struct TricubicBricks {
    const S (*b)[16];
    __device__ __forceinline__ double operator()(int i, int r, int k) const { return (double) b[i][4 * r + k]; }
};

// LAYOUT = GFB_LAYOUT_POINTS or GFB_LAYOUT_HERMITE (MIXED only: the BSPLINE record format, filled by flat index — see
// gf_repack_bspline_kernel — so that a stencil is two full lines; gf_eval_bspline_kernel<.., 2> is its fast reader and
// this one the fallback for grids of different geometry or an evaluation order).
template <typename S, int LAYOUT>
__device__ __forceinline__ void tricubic_interpolate(const GridView& G, const AtomCell& c, double& val, double& gx, double& gy,
                                                     double& gz) {
    const bool xin = c.ix > 0 && c.ix < G.nc[0];   // :817 (ix < counts-1 always holds for an inside atom)
    const bool yin = c.iy > 0 && c.iy < G.nc[1];   // :849
    const bool zin = c.iz > 0 && c.iz < G.nc[2];   // :866
    TricubicWeights w;
    tricubic_weights(c.fx, c.fy, c.fz, w);
    if constexpr (LAYOUT == GFB_LAYOUT_POINTS) {
        TricubicPoints<S> V;
        V.nz = G.nc[2] + 1;
        V.nyz = (long long) (G.nc[1] + 1) * V.nz;
        V.v = static_cast<const S*>(G.cells) + ((long long) c.ix * V.nyz + (long long) c.iy * V.nz + c.iz);   // :801
        tricubic_eval(V, xin, yin, zin, w, val, gx, gy, gz);
    } else {
        const S* rec = static_cast<const S*>(G.cells) + (((size_t) c.ix * G.nc[1] + c.iy) * G.nc[2] + c.iz) * 32;
        const size_t plane2 = (size_t) G.nc[1] * G.nc[2] * 64;    // records two x-planes further on
        S b[4][16];
#pragma unroll
        for (int i = 0; i < 4; i++) load_brick(rec + (i >> 1) * plane2 + (i & 1) * 16, b[i]);
        TricubicBricks<S> V;
        V.b = b;
        tricubic_eval(V, xin, yin, zin, w, val, gx, gy, gz);
    }
}

// One grid's tricubic contribution for an inside atom (:796-893), same epilogue as accumulate_bspline.
__device__ __forceinline__ void tricubic_epilogue(const GridView& G, double sd, double dval, double gx, double gy, double gz,
                                                  double& e_g, double& Fx, double& Fy, double& Fz) {
    if (G.inv_power > 0.0) {  // :879-886
        const double base = dval;
        dval = pow(base, G.inv_power);
        const double pf = G.inv_power * pow(base, G.inv_power - 1.0);
        gx *= pf;
        gy *= pf;
        gz *= pf;
    }
    e_g = sd * dval;                     // :892
    Fx -= sd * (gx / G.spacing[0]);      // :889, :893
    Fy -= sd * (gy / G.spacing[1]);
    Fz -= sd * (gz / G.spacing[2]);
}
template <typename S, int LAYOUT>
__device__ __forceinline__ void accumulate_tricubic(const GridView& G, const AtomCell& c, double sd, double& e_g, double& Fx,
                                                    double& Fy, double& Fz) {
    double dval, gx, gy, gz;
    tricubic_interpolate<S, LAYOUT>(G, c, dval, gx, gy, gz);
    tricubic_epilogue(G, sd, dval, gx, gy, gz, e_g, Fx, Fy, Fz);
}

// :1093-1117 — harmonic wall outside the grid (unscaled). Inside atoms with scale == 0 land here too and contribute
// exactly 0 (quirk Q3). Rare (1-2 % of atoms): kept out of line so its FP64 temporaries do not cost registers.
struct Restraint {
    double e, fx, fy, fz;
};
static __device__ __noinline__ Restraint restraint_terms(const GridView& G, double x, double y, double z) {
    const double px = x - G.origin[0], py = y - G.origin[1], pz = z - G.origin[2];
    const double devx = px < 0.0 ? px : (px > G.hcorner[0] ? px - G.hcorner[0] : 0.0);
    const double devy = py < 0.0 ? py : (py > G.hcorner[1] ? py - G.hcorner[1] : 0.0);
    const double devz = pz < 0.0 ? pz : (pz > G.hcorner[2] ? pz - G.hcorner[2] : 0.0);
    const double hk = 0.5 * G.oob_k;
    Restraint r;
    r.e = hk * devx * devx;
    r.e += hk * devy * devy;
    r.e += hk * devz * devz;
    r.fx = G.oob_k * devx;
    r.fy = G.oob_k * devy;
    r.fz = G.oob_k * devz;
    return r;
}
__device__ __forceinline__ void accumulate_restraint(const GridView& G, double x, double y, double z, double& e_g, double& Fx,
                                                     double& Fy, double& Fz) {
    const Restraint r = restraint_terms(G, x, y, z);
    e_g = r.e;
    Fx -= r.fx;
    Fy -= r.fy;
    Fz -= r.fz;
}

template <typename S, int LAYOUT, int NG>
__host__ __device__ constexpr int eval_min_blocks() {
    return (LAYOUT == GFB_LAYOUT_BSPLINE || LAYOUT >= GFB_LAYOUT_POINTS) ? 2 : ((NG == 1 && sizeof(S) == 4) ? 6 : 4);
}

template <typename S, int LAYOUT, int NG, bool SAME, bool SINGLE>
__global__ void __launch_bounds__(kBlock, eval_min_blocks<S, LAYOUT, NG>()) gf_eval_kernel(const __grid_constant__ EvalParams p) {
    constexpr bool EXACT = sizeof(S) == 8;
    constexpr int NGC = NG > 0 ? NG : 1;
    // With a compile-time grid count, one shared geometry and the one-load-per-stencil layout, every grid's stencil
    // load is issued before any arithmetic, so the G memory round trips overlap instead of following one another
    // (C5: 157 -> 138 us). ROWS/PAIRS would need 4x/2x the registers in flight and spill (C5 ROWS: 205 -> 261 us),
    // so they keep one grid at a time.
    constexpr bool BATCHED = NG > 0 && SAME && LAYOUT == GFB_LAYOUT_CELLS;
    const unsigned t0 = blockIdx.x * kBlock;          // total <= 2e9 (checked by the launcher): 32-bit indices
    const unsigned t = t0 + threadIdx.x;
    const unsigned total = (unsigned) p.total;
    const int lane = threadIdx.x & 31;
    const bool active = t < total;
    if (p.energies_clear)   // grid-stride: with energy slots the next accumulator can have more entries than the launch has threads
        for (unsigned c = t; c < (unsigned) (p.n_replicas * p.n_slots); c += gridDim.x * blockDim.x) p.energies_clear[c] = 0.0;

    int rep = -1;
    unsigned ia = 0;
    long long gidx = 0;
    if (active) {
        const unsigned a = p.order ? (unsigned) p.order[t] : t;
        if (SINGLE) {
            rep = 0;
            ia = a;
        } else {
            rep = (int) (a / (unsigned) p.n_atoms);
            ia = a - (unsigned) rep * (unsigned) p.n_atoms;
        }
        const int particle = p.particles ? p.particles[ia] : (int) ia;
        gidx = (long long) rep * p.n_particles + particle;
        // Particle groups (GridForce::addParticleGroup): every atom carries the energy slot of its group, and the
        // energy of replica r, group s accumulates at [r * n_slots + s]. Runs of equal key reduce together.
        if (p.slots) rep = rep * p.n_slots + p.slots[ia];
    }

    // Scaling factors depend on the atom ordinal only: their loads go out first and overlap the position fetch.
    double sd[NGC];
#pragma unroll
    for (int g = 0; g < NGC; g++) sd[g] = (NG > 0 && active) ? p.grid[g].scaling[ia] : 0.0;

    // Positions of the block's 256 consecutive atoms are 6144 contiguous bytes when no index indirection is in
    // play: read them as 384 16-byte vectors (4 lines per warp instruction instead of 24 sectors x 3 instructions
    // for stride-24 scalar loads), then pick x,y,z out of shared memory (stride 3 doubles: conflict-free).
    __shared__ double2 s_pos2[kBlock * 3 / 2];
    const bool staged = p.order == nullptr && p.particles == nullptr && p.n_particles == p.n_atoms &&
                        (reinterpret_cast<uintptr_t>(p.pos) & 15) == 0;
    if (staged) {
        const double2* src = reinterpret_cast<const double2*>(p.pos + 3 * (size_t) t0);   // t0*24 bytes: 16-byte aligned
        const unsigned left = 3u * (total - t0);                                          // doubles left in the array
        for (unsigned i = threadIdx.x; i < kBlock * 3 / 2; i += kBlock) {
            double2 v = make_double2(0.0, 0.0);
            if (2 * i + 1 < left) {
                asm volatile("ld.global.cs.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(src + i));
            } else if (2 * i < left) {   // odd tail: the last double of the array
                v.x = load_stream(reinterpret_cast<const double*>(src + i));
            }
            s_pos2[i] = v;
        }
        __syncthreads();
    }
    const double* my_pos = staged ? reinterpret_cast<const double*>(s_pos2) + 3 * threadIdx.x : p.pos + 3 * gidx;
    double x = 0.0, y = 0.0, z = 0.0;
    if (active) {
        if (staged) {
            x = my_pos[0];
            y = my_pos[1];
            z = my_pos[2];
        } else {
            x = load_stream(my_pos);
            y = load_stream(my_pos + 1);
            z = load_stream(my_pos + 2);
        }
    }

    double e_total = 0.0;
    double Fx = 0.0, Fy = 0.0, Fz = 0.0;
    const int ng = NG > 0 ? NG : p.n_grids;
    __shared__ double s_warp_ge[SINGLE ? kBlock / 32 : 1][SINGLE ? GFB_MAX_GRIDS : 1];
    unsigned heads;
    const unsigned span = run_span(rep, (unsigned) lane, heads);   // runs of equal energy key inside the warp
    const bool head = rep >= 0 && ((heads >> lane) & 1u);

    if constexpr (BATCHED) {
        const AtomCell c = classify<EXACT>(p.grid[0], x, y, z);
        S v[NGC][8];
        bool interp[NGC];
#pragma unroll
        for (int g = 0; g < NGC; g++) {
            interp[g] = active && c.inside && sd[g] != 0.0;
            if (interp[g]) load_stencil<S, LAYOUT>(p.grid[g], c.ix, c.iy, c.iz, v[g]);
        }
#pragma unroll
        for (int g = 0; g < NGC; g++) {
            double e_g = 0.0;
            if (interp[g]) accumulate_inside<S>(p.grid[g], v[g], c, sd[g], e_g, Fx, Fy, Fz);
            else if (active) accumulate_restraint(p.grid[g], my_pos[0], my_pos[1], my_pos[2], e_g, Fx, Fy, Fz);
            e_total += e_g;
            if (p.grid_energies) {  // uniform branch
                double eg = e_g;
                if (SINGLE) {   // warp sums now, one atomic (or plain store) per block and grid after the loop
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) eg += __shfl_xor_sync(kFull, eg, off);
                    if (lane == 0) s_warp_ge[threadIdx.x >> 5][g] = eg;
                } else {
                    run_sum(eg, span);
                    if (head) red_add_f64(p.grid_energies + (size_t) rep * ng + g, eg);
                }
            }
        }
    } else {
        AtomCell c;
        if (SAME) c = classify<EXACT>(p.grid[0], x, y, z);
#pragma unroll
        for (int g = 0; g < (NG > 0 ? NG : GFB_MAX_GRIDS); g++) {
            if (NG == 0 && g >= ng) break;
            const GridView& G = p.grid[g];
            double e_g = 0.0;
            if (active) {
                if (!SAME) c = classify<EXACT>(G, x, y, z);
                const double s = NG > 0 ? sd[NG > 0 ? g : 0] : G.scaling[ia];
                if (c.inside && s != 0.0) {
                    if constexpr (LAYOUT == GFB_LAYOUT_BSPLINE || LAYOUT == GFB_LAYOUT_BSPLINE_POINTS) {
                        accumulate_bspline<S, LAYOUT>(G, c, s, e_g, Fx, Fy, Fz);
                    } else if constexpr (LAYOUT == GFB_LAYOUT_POINTS || LAYOUT == GFB_LAYOUT_HERMITE) {
                        accumulate_tricubic<S, LAYOUT>(G, c, s, e_g, Fx, Fy, Fz);
                    } else {
                        S v[8];
                        load_stencil<S, LAYOUT>(G, c.ix, c.iy, c.iz, v);
                        accumulate_inside<S>(G, v, c, s, e_g, Fx, Fy, Fz);
                    }
                } else {
                    accumulate_restraint(G, x, y, z, e_g, Fx, Fy, Fz);
                }
            }
            e_total += e_g;
            if (p.grid_energies) {  // uniform branch
                double eg = e_g;
                if (SINGLE) {   // warp sums now, one atomic (or plain store) per block and grid after the loop
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) eg += __shfl_xor_sync(kFull, eg, off);
                    if (lane == 0) s_warp_ge[threadIdx.x >> 5][g] = eg;
                } else {
                    run_sum(eg, span);
                    if (head) red_add_f64(p.grid_energies + (size_t) rep * ng + g, eg);
                }
            }
        }
    }

    if (SINGLE && p.grid_energies) {  // uniform branch
        __syncthreads();
        if ((int) threadIdx.x < ng) {
            double b = 0.0;
#pragma unroll
            for (int w = 0; w < kBlock / 32; w++) b += s_warp_ge[SINGLE ? w : 0][SINGLE ? threadIdx.x : 0];
            if (p.energy_store) p.grid_energies[threadIdx.x] = b;
            else red_add_f64(p.grid_energies + threadIdx.x, b);
        }
    }

    if (p.atom_energies && active) p.atom_energies[p.order ? p.order[t] : t] = e_total;   // uniform branch

    // ---- forces -------------------------------------------------------------------------------
    if (active && p.forces) {
        const int fmode = p.force_mode;   // launch-uniform
        if (fmode == GFB_FORCE_FIXED_ADD) {
            unsigned long long* f = static_cast<unsigned long long*>(p.forces);
            const double scale = 4294967296.0;  // 2^32, gridForce.cu:487-499
            red_add_u64(f + gidx, (unsigned long long) (long long) (Fx * scale));
            red_add_u64(f + p.force_stride + gidx, (unsigned long long) (long long) (Fy * scale));
            red_add_u64(f + 2 * p.force_stride + gidx, (unsigned long long) (long long) (Fz * scale));
        } else if (fmode == GFB_FORCE_F64_ADD) {
            double* f = static_cast<double*>(p.forces) + 3 * gidx;
            red_add_f64(f, Fx);
            red_add_f64(f + 1, Fy);
            red_add_f64(f + 2, Fz);
        } else if (fmode == GFB_FORCE_F32_STORE) {
            float* f = static_cast<float*>(p.forces) + 3 * gidx;
            f[0] = (float) Fx;
            f[1] = (float) Fy;
            f[2] = (float) Fz;
        } else {
            double* f = static_cast<double*>(p.forces) + 3 * gidx;
            f[0] = Fx;
            f[1] = Fy;
            f[2] = Fz;
        }
    }

    // ---- energy -------------------------------------------------------------------------------
    if (p.energies) {  // uniform branch
        if (SINGLE) {
            __shared__ double warp_sum[kBlock / 32];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) e_total += __shfl_xor_sync(kFull, e_total, off);
            if (lane == 0) warp_sum[threadIdx.x >> 5] = e_total;
            __syncthreads();
            if (threadIdx.x < 32) {
                double b = threadIdx.x < kBlock / 32 ? warp_sum[threadIdx.x] : 0.0;
#pragma unroll
                for (int off = kBlock / 64; off > 0; off >>= 1) b += __shfl_xor_sync(kFull, b, off);
                if (threadIdx.x == 0) {
                    if (p.energy_store) *p.energies = b;
                    else red_add_f64(p.energies, b);
                }
            }
        } else {
            run_sum(e_total, span);
            if (head) red_add_f64(p.energies + rep, e_total);
        }
    }
}

}  // namespace gfb
#endif
