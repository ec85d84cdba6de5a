// The evaluation kernel of the named configurations: MIXED precision, packed cells, grids of one geometry, no inv-power.
//
// What differs from the general kernel (gf_kernels.cuh, gf_eval_kernel); measurements in DESIGN.md §4/§6:
//   * LINES. HBM and L2 move 128-byte lines, a stencil is 32 bytes. With 2-4 grids the packed cells of all grids are
//     woven into ONE 128-byte record per cell (gf_interleave_cells_kernel), so everything an atom needs is one line.
//     A warp fetches the lines of its 32 atoms with 8 warp-wide cp.async (LDGSTS.128) in which the eight lanes of an
//     octet copy the eight 16-byte granules of the SAME line: 4 full lines per instruction (one L2 request per line)
//     instead of 3 x 32 single-sector requests to 96 different lines. The data lands in a swizzled, conflict-free
//     slice of shared memory without passing through registers, and the lane that owns the atom reads each grid's
//     8 corners right before it uses them (2 LDS.128 per grid): 48 registers, 10 blocks of 128 threads per SM.
//     C5: DRAM traffic 842 -> 495 MB per launch (= the algorithmic bytes), 137 -> 86 us.
//   * INSTRUCTIONS. The general kernel issues 693 warp instructions per 32 atoms (ncu, r1). Here: replica/atom split by a
//     host magic multiplier, one 32-bit cell index, one near-integer test on fractions that are needed anyway, gradient
//     scaled by 1/spacing once per atom instead of once per grid, FP32 force accumulation, no pow code, restraint and
//     exact re-division out of line, no block barrier (positions are staged per warp).
//   * FORCES. The force lines an ADD mode will touch are prefetched into L2 at kernel start (FPATH 1): the RED that
//     arrives ~2 DRAM round trips later finds them there. One grid (C3): 45.5 -> 35.1 us.
//
// Reference semantics implemented (platforms/reference/src/ReferenceGridForceKernels.cpp): inside test :687-696,
// cell index/fraction :708-715 (bit-exact), trilinear value z->y->x :1039-1053, gradient :1066-1072, scaling and
// accumulation :1061-1063/:1082, restraint :1093-1117.
#ifndef GF_EVAL_LINES_CUH_
#define GF_EVAL_LINES_CUH_

#include "gf_kernels.cuh"
#include "gf_gather.cuh"

namespace gfb {

// Exact IEEE re-division of all three axes, taken when one fast quotient lies within rounding distance of an integer
// (probability ~1e-12 per atom) or on the upper face. Out of line: the FP64 division sequence must not be if-converted
// into the main path.
struct ExactCell {
    int ix, iy, iz;
    double fx, fy, fz;
};
static __device__ __noinline__ ExactCell exact_cell(const GridView& G, double px, double py, double pz) {
    ExactCell c;
    const double qx = px / G.spacing[0], qy = py / G.spacing[1], qz = pz / G.spacing[2];
    c.ix = min(__double2int_rz(qx), G.nc[0] - 1);
    c.iy = min(__double2int_rz(qy), G.nc[1] - 1);
    c.iz = min(__double2int_rz(qz), G.nc[2] - 1);
    c.fx = qx - (double) c.ix;
    c.fy = qy - (double) c.iy;
    c.fz = qz - (double) c.iz;
    return c;
}

// Inside test + cell index + in-cell fractions of the lines kernel (and of gf_classify_lines_kernel, which the bit-exact
// parity tests call). The quotient is pi * fl(1/spacing); it is within 3.3e-16*q of the correctly rounded pi/spacing, so
// the truncation can only differ when the fraction is that close to 0 or 1. near_int[k] = 1.8e-15 * cells on axis k
// covers that with margin; such atoms (and the upper face, where ix == nc and the fraction is 0) redo the division
// exactly, out of line.
struct FastCell {
    int ix, iy, iz;
    double fx, fy, fz;
    bool inside;
};
__device__ __forceinline__ FastCell classify_fast(const GridView& G, const double near_int[3], double x, double y, double z,
                                                  bool active) {
    FastCell c;
    const double px = x - G.origin[0], py = y - G.origin[1], pz = z - G.origin[2];
    c.inside = active && (px >= 0.0 && px <= G.hcorner[0]) && (py >= 0.0 && py <= G.hcorner[1]) &&
               (pz >= 0.0 && pz <= G.hcorner[2]);
    c.ix = c.iy = c.iz = 0;
    c.fx = c.fy = c.fz = 0.0;
    if (c.inside) {
        const double qx = px * G.inv_spacing[0], qy = py * G.inv_spacing[1], qz = pz * G.inv_spacing[2];
        c.ix = __double2int_rz(qx);
        c.iy = __double2int_rz(qy);
        c.iz = __double2int_rz(qz);
        c.fx = qx - (double) c.ix;
        c.fy = qy - (double) c.iy;
        c.fz = qz - (double) c.iz;
        const bool near = c.fx <= near_int[0] || c.fx >= 1.0 - near_int[0] || c.fy <= near_int[1] ||
                          c.fy >= 1.0 - near_int[1] || c.fz <= near_int[2] || c.fz >= 1.0 - near_int[2];
        if (near) {
            const ExactCell e = exact_cell(G, px, py, pz);
            c.ix = e.ix;
            c.iy = e.iy;
            c.iz = e.iz;
            c.fx = e.fx;
            c.fy = e.fy;
            c.fz = e.fz;
        }
    }
    return c;
}

// Restraint of an atom outside the (shared) grid box for all NG GridForces (:1093-1117): every force adds its own
// harmonic wall with its own constant. Rare; out of line.
template <int NG>
struct RestraintAll {
    double e[NG];
    float fx, fy, fz;
};
template <int NG>
static __device__ __noinline__ RestraintAll<NG> restraint_all(const EvalParams& p, double x, double y, double z) {
    RestraintAll<NG> r;
    double fx = 0.0, fy = 0.0, fz = 0.0;
#pragma unroll
    for (int g = 0; g < NG; g++) {
        const Restraint t = restraint_terms(p.grid[g], x, y, z);
        r.e[g] = t.e;
        fx += t.fx;
        fy += t.fy;
        fz += t.fz;
    }
    r.fx = (float) fx;
    r.fy = (float) fy;
    r.fz = (float) fz;
    return r;
}

__device__ __forceinline__ void lds128(unsigned addr, float* v) {
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(addr) : "memory");
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

constexpr int kForceRed = 0, kForcePrefetch = 1;
// Internal force mode of an energy-only launch (forces == NULL; GridForceBatch::evaluate, includeForces = false): no
// gradient arithmetic, no force read-modify-write.
constexpr int kForceNone = 4;

// Threads per block: no block barrier is used, so the block is only the scheduling granule. 128 threads keep the tail
// of a launch short (C4 is 1.02 waves of 256-thread blocks); one grid + one replica keeps 256 because it ends in one
// atomic per block on a single address.
#ifndef GFB_LINES_BLOCK_MULTI
#define GFB_LINES_BLOCK_MULTI 64    // threads per block of the 2-4 grid kernels: 20 blocks per SM. Measured against 128
                                    // (A/B builds, -DGFB_LINES_BLOCK_MULTI=128): C5 83.7 -> 81.8 us, a 1/8 shard of it
                                    // 13.5 -> 13.3 us, C4 unchanged
#endif
__host__ __device__ constexpr int lines_block(int ng) { return ng == 1 ? 256 : GFB_LINES_BLOCK_MULTI; }
#ifndef GFB_PERSIST_THREADS_PER_SM
#define GFB_PERSIST_THREADS_PER_SM 1024   // resident threads per SM of the tile-striding variant: 64 registers. At 1280 (48
                                          // registers) the loop-carried state spills and a 1/8 shard of C5 takes 14.05 us
                                          // instead of 11.60 (13.43 with one block per tile)
#endif
#ifndef GFB_PERSIST_DEFER
#define GFB_PERSIST_DEFER 3               // tiles whose energy sums a block of the tile-striding variant can park (12 bytes per thread each)
#endif
#ifndef GFB_PERSIST_BLOCKS_NG1
#define GFB_PERSIST_BLOCKS_NG1 6
#endif
__host__ __device__ constexpr int lines_blocks_per_sm(int ng, bool persist) {
    return ng == 1 ? (persist ? GFB_PERSIST_BLOCKS_NG1 : 6) : (persist ? GFB_PERSIST_THREADS_PER_SM : 1280) / lines_block(ng);
}

__device__ __forceinline__ void cp_async16(unsigned smem_addr, const void* gptr) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gptr) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
}

//   NG     grids evaluated per atom, 1..4 (1: the grid's own packed cells; 2..4: 128-byte records of 4 slots)
//   FMODE  gfb_force_mode, or kForceNone (energy only)
//   FPATH  kForceRed | kForcePrefetch (ADD modes only)
//   SINGLE one replica and no energy slots: block-level energy reduction, one atomic per block
//   GE     per-grid energies wanted (p.grid_energies): a template flag so that the per-grid terms cost no registers
//          in the common case
// Occupancy: 40 registers x 6 blocks of 256 (one grid), 48 registers x 10 blocks of 128 with 16 KB of smem each (2-4 grids;
// 12 blocks / 40 registers measured no faster on C5 and slower on C4).
//   PERSIST the launch's blocks stride over the tiles and park their energy sums (small launches under launch overlap,
//          see the tile loop below); false = one tile per block, code as if the loop were not there
template <int NG, int FMODE, int FPATH, bool SINGLE, bool GE, bool PERSIST = false>
__global__ void __launch_bounds__(lines_block(NG), lines_blocks_per_sm(NG, PERSIST)) gf_eval_lines_kernel(const __grid_constant__ EvalParams p) {
    constexpr int kBlock = lines_block(NG);
    // One slice per warp: first the warp's 32 positions (768 bytes), then (NG > 1) its 32 records of 128 bytes.
    constexpr unsigned kWarpSlice16 = NG == 1 ? 48 : 256;                // slice size in 16-byte units
    __shared__ __align__(128) double2 s_pos2[(kBlock / 32) * kWarpSlice16];
    float4* const s_rec = reinterpret_cast<float4*>(s_pos2);

    const unsigned total = (unsigned) p.total;
    // Programmatic dependent launch (sm_90+): let the NEXT launch on this stream start its blocks as soon as all of ours
    // have started, so that its position/record fetches overlap our tail; it blocks at griddepcontrol.wait (below, before
    // the first global write) until this grid has completed. Both are no-ops in a launch without the PDL attribute.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    // Tiles of kBlock atoms, block b takes tiles b, b + gridDim.x, ... The host launches one block per tile, except for
    // SMALL launches under launch overlap (p.defer, a few waves of blocks: a 1/8 shard of C5 is two): those get a grid
    // that is resident all at once. Every block then starts — and fires launch_dependents — right away, so the next
    // launch is already pending when our blocks begin to exit and takes their SM slots one by one; with one block per
    // tile the last blocks of a launch start (and release the next launch) only a block lifetime before its end, and the
    // slots freed meanwhile sit empty for the launch latency (measured ~3 us per launch whatever its size).
    // In that mode nothing the kernel writes needs the previous launch before the very end: forces are commutative
    // atomics (or absent), and the per-replica energy sums of up to kDefer tiles are parked in shared memory; the block
    // waits for the previous grid once, after its last tile, and only then issues its energy atomics and its share of
    // the accumulator clear.
    constexpr bool kAddMode = FMODE == GFB_FORCE_F64_ADD || FMODE == GFB_FORCE_FIXED_ADD;
    constexpr bool kCanDefer = PERSIST && !SINGLE && !GE && (kAddMode || FMODE == kForceNone);
    static_assert(!PERSIST || kCanDefer, "the tile-striding variant exists for the deferred-energy modes only");
    constexpr int kDefer = GFB_PERSIST_DEFER;
    __shared__ double s_def_e[kCanDefer ? kDefer * kBlock : 1];
    __shared__ int s_def_k[kCanDefer ? kDefer * kBlock : 1];
    constexpr bool defer = kCanDefer;   // the host launches the PERSIST instantiations for deferred launches only (p.defer)
    auto flush_parked = [&](unsigned n) {
        if (kCanDefer && p.energies) {
            for (unsigned j = 0; j < n; j++) {
                const int k = s_def_k[j * kBlock + threadIdx.x];
                if (k >= 0) red_add_f64(p.energies + k, s_def_e[j * kBlock + threadIdx.x]);
            }
        }
    };
    const unsigned n_tiles = (total + (unsigned) kBlock - 1u) / (unsigned) kBlock;
    // Loop state is ONE register (it): the tile follows from it, and "has this block waited for the previous grid" is
    // it > kDefer. tid is laundered through an empty asm every iteration so that the lane-derived addresses below are
    // recomputed (a few integer instructions) instead of being hoisted out of the loop and kept alive across it — hoisted,
    // they cost 48 bytes of spills at 48 registers.
    unsigned it = 0;
    do {
    unsigned tid = threadIdx.x;
    if (PERSIST) asm volatile("" : "+r"(tid));
    const unsigned lane = tid & 31u;
    const unsigned tile = blockIdx.x + it * gridDim.x;
    const bool waited = PERSIST ? it > (unsigned) kDefer : false;   // uniform
    const unsigned t0 = tile * kBlock;
    const unsigned t = t0 + tid;
    const bool active = t < total;

    // ---- who am I: replica, atom ordinal, particle -------------------------------------------------------------
    // Evaluation order (gfb_kernel_sort_atoms): thread t evaluates atom order[t] of the flattened [replica][atom] list.
    // PERSIST launches are "plain" by the launcher's choice: no evaluation order, no particle map, no energy slots,
    // 16-byte aligned positions, energies wanted — the run-time switches for those fold away (fewer registers live across
    // the tile loop, ~10 % fewer instructions).
    const unsigned a = (!PERSIST && p.order != nullptr && active) ? (unsigned) p.order[t] : t;
    unsigned rep = 0, ia = a;
    if (!SINGLE) {   // a / n_atoms by the host's magic multiplier floor(2^32 / n_atoms): estimate is q or q-1
        rep = __umulhi(a, p.div_magic);
        ia = a - rep * (unsigned) p.n_atoms;
        if (ia >= (unsigned) p.n_atoms) {
            ia -= (unsigned) p.n_atoms;
            rep++;
        }
    }
    if (!active) ia = 0;
    const bool plain = PERSIST || (p.particles == nullptr && p.n_particles == p.n_atoms && p.order == nullptr);   // uniform
    unsigned gidx = t;                                                         // particle slot in pos / forces
    if (!plain) gidx = rep * (unsigned) p.n_particles + (p.particles ? (unsigned) p.particles[ia] : ia);
    int key = -1;
    if (active) key = (!PERSIST && p.slots) ? (int) rep * p.n_slots + p.slots[ia] : (int) rep;

    // ---- loads that depend on the atom ordinal only go out first -------------------------------------------------
    const double sd0 = (NG == 1 && active) ? p.grid[0].scaling[ia] : 0.0;

    unsigned long long* const ffix = static_cast<unsigned long long*>(p.forces);
    double* const fdbl = static_cast<double*>(p.forces);
    if (p.forces && (FMODE == GFB_FORCE_F64_ADD || FMODE == GFB_FORCE_FIXED_ADD) && FPATH == kForcePrefetch) {
        if (FMODE == GFB_FORCE_FIXED_ADD) {
            if (active && (lane & 15u) == 0) {   // 16 lanes x 8 bytes = one line per plane
                prefetch_l2(ffix + gidx);
                prefetch_l2(ffix + p.force_stride + gidx);
                prefetch_l2(ffix + 2 * p.force_stride + gidx);
            }
        } else if (active && (lane & 3u) == 0) {   // 4 lanes x 24 bytes < one line
            prefetch_l2(fdbl + 3 * (size_t) gidx);
        }
    }

    // Positions of the block that will run in this block's SM slot NEXT (p.ahead_blocks = resident blocks of the launch)
    // are pulled into L2 now: when that block starts, its first dependent load is an L2 hit instead of a DRAM round trip.
    if (p.ahead_blocks && plain) {   // PERSIST: that block is this one, at its next tile
        const unsigned long long first = ((unsigned long long) tile + (PERSIST ? gridDim.x : p.ahead_blocks)) * kBlock;   // its first atom
        if (first < total && tid < (kBlock * 24u + 127u) / 128u) {
            const char* line = reinterpret_cast<const char*>(p.pos + 3 * first) + 128u * tid;
            if (line < reinterpret_cast<const char*>(p.pos + 3 * (size_t) total)) prefetch_l2(line);
        }
    }

    // ---- positions: a warp's 32 atoms are 768 contiguous bytes -> 48 coalesced 16-byte loads through the warp's own
    //      slice of shared memory (no block barrier anywhere on this path; the slice is reused for the records below)
    double x = 0.0, y = 0.0, z = 0.0;
    const bool staged = PERSIST || (plain && (reinterpret_cast<uintptr_t>(p.pos) & 15) == 0);   // uniform
    if (staged) {
        const unsigned w0 = t - lane;                                               // first atom of this warp
        double2* const s_warp = s_pos2 + (tid >> 5) * kWarpSlice16;
        if (w0 < total) {
            const double2* src = reinterpret_cast<const double2*>(p.pos + 3 * (size_t) w0);
            const unsigned left = 3u * (total - w0);                                // doubles left in the array (>= 3)
            double2 a = make_double2(0.0, 0.0), b = make_double2(0.0, 0.0);
            if (left >= 96u) {                                                      // every warp but the last
                asm volatile("ld.global.cs.v2.f64 {%0,%1}, [%2];" : "=d"(a.x), "=d"(a.y) : "l"(src + lane));
                if (lane < 16) asm volatile("ld.global.cs.v2.f64 {%0,%1}, [%2];" : "=d"(b.x), "=d"(b.y) : "l"(src + 32 + lane));
            } else {
                if (2 * lane + 1 < left) asm volatile("ld.global.cs.v2.f64 {%0,%1}, [%2];" : "=d"(a.x), "=d"(a.y) : "l"(src + lane));
                else if (2 * lane < left) a.x = load_stream(reinterpret_cast<const double*>(src + lane));
                if (lane < 16) {
                    if (2 * (32 + lane) + 1 < left) asm volatile("ld.global.cs.v2.f64 {%0,%1}, [%2];" : "=d"(b.x), "=d"(b.y) : "l"(src + 32 + lane));
                    else if (2 * (32 + lane) < left) b.x = load_stream(reinterpret_cast<const double*>(src + 32 + lane));
                }
            }
            s_warp[lane] = a;
            if (lane < 16) s_warp[32 + lane] = b;
        }
        __syncwarp();
        const double* mine = reinterpret_cast<const double*>(s_warp) + 3 * lane;
        x = mine[0];
        y = mine[1];
        z = mine[2];
        __syncwarp();   // the slice is overwritten by the records next
    } else if (active) {
        const double* mine = p.pos + 3 * (size_t) gidx;
        x = load_stream(mine);
        y = load_stream(mine + 1);
        z = load_stream(mine + 2);
    }

    // ---- classification (:687-715), bit-exact ------------------------------------------------------------------------
    const GridView& G = p.grid[0];
    const FastCell fc = classify_fast(G, p.near_int, x, y, z, active);
    const bool inside = fc.inside;
    unsigned cell = 0xffffffffu;
    if (inside) cell = ((unsigned) fc.ix * (unsigned) G.nc[1] + (unsigned) fc.iy) * (unsigned) G.nc[2] + (unsigned) fc.iz;
    const double dfx = fc.fx, dfy = fc.fy, dfz = fc.fz;
    const float fx = (float) dfx, fy = (float) dfy, fz = (float) dfz;

    // ---- stencils + interpolation: gradient FP32, value FP64 (see trilinear_value_f64) -----------------------------------
    double e_g[GE ? NG : 1];
    double e_total = 0.0;
    float sx = 0.f, sy = 0.f, sz = 0.f;   // sum over grids of scaling * (corner-difference gradient), before 1/spacing
    if (GE) {
#pragma unroll
        for (int g = 0; g < (GE ? NG : 1); g++) e_g[g] = 0.0;
    }
    auto one_grid = [&](int g, const float* v, double s) {
        if (FMODE != kForceNone) {
            float val, dx, dy, dz;
            trilinear<float>(v, fx, fy, fz, val, dx, dy, dz);
            const float sf = (float) s;
            sx = fmaf(sf, dx, sx);
            sy = fmaf(sf, dy, sy);
            sz = fmaf(sf, dz, sz);
        }
        const double e = s * trilinear_value_f64(v, dfx, dfy, dfz);   // :1061
        e_total += e;
        if (GE) e_g[GE ? g : 0] = e;
    };
    if (NG == 1) {
        if (inside && sd0 != 0.0) {   // :706
            float v[8];
            load32(static_cast<const float*>(G.cells) + 8 * (size_t) cell, v);
            one_grid(0, v, sd0);
        }
    } else {
        // The record of atom A (lane A of this warp) lives at warp_base + 128*A, its 16-byte granule c (slot c/2, half
        // c%2) at position c ^ (A & 7). Round i: the eight lanes of an octet copy the eight granules of the record of the
        // atom owned by lane 4i + octet -> 4 full lines per instruction, each written to one 128-byte smem row.
        const unsigned warp_base = (unsigned) __cvta_generic_to_shared(s_rec) + (tid >> 5) * 4096u;
        const unsigned gran = lane & 7u, octet = lane >> 3;
        const char* lane_base = static_cast<const char*>(p.lines) + 16u * gran;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const unsigned A = 4u * i + octet;
            const unsigned c = __shfl_sync(kFull, cell, (int) A);
            if (c != 0xffffffffu && gran < 2u * NG) cp_async16(warp_base + A * 128u + ((gran ^ (A & 7u)) << 4), lane_base + 128ull * c);
        }
        cp_async_wait_all();
        __syncwarp();
        const unsigned rbase = (warp_base + lane * 128u) ^ ((lane & 7u) << 4);   // 128-byte aligned base: xor == or
        if (inside) {
            {   // (the one_grid lambda above serves the one-grid kernel only)
                // Trilinear interpolation is linear in the corner values, and all NG grids share the cell and the
                // fractions: the scaled corners are summed over the grids first (FP64: s * corner is exact to 1e-16,
                // and nothing is rounded to FP32 before corners are differenced), and value and gradient are formed ONCE
                // from the eight sums — 8 conversions + 8 DFMA per grid and 32 FP64 operations per atom instead of a
                // full FP64 value and FP32 gradient interpolation per grid (168 -> ~105 instructions for three grids; the
                // kernel is issue-bound on small launches). Forces come out of FP64 arithmetic on the stored corners.
                double C[8];
#pragma unroll
                for (int k = 0; k < 8; k++) C[k] = 0.0;
#pragma unroll
                for (int g = 0; g < NG; g++) {
                    const double s = p.grid[g].scaling[ia];
                    if (s != 0.0) {   // :706
                        if (GE) {   // per-grid energies wanted: this grid's value on its own as well (the forces below are
                                    // formed from the summed corners either way, so both instantiations give the same forces)
                            float v[8];
                            lds128(rbase ^ (32u * g), v);
                            lds128(rbase ^ (32u * g + 16u), v + 4);
                            e_g[GE ? g : 0] = s * trilinear_value_f64(v, dfx, dfy, dfz);
#pragma unroll
                            for (int k = 0; k < 8; k++) C[k] = fma(s, (double) v[k], C[k]);
                        } else {
                            float v[4];
                            lds128(rbase ^ (32u * g), v);
#pragma unroll
                            for (int k = 0; k < 4; k++) C[k] = fma(s, (double) v[k], C[k]);
                            lds128(rbase ^ (32u * g + 16u), v);
#pragma unroll
                            for (int k = 0; k < 4; k++) C[4 + k] = fma(s, (double) v[k], C[4 + k]);
                        }
                    }
                }
                const double ax = 1.0 - dfx, ay = 1.0 - dfy, az = 1.0 - dfz;
                const double vmm = az * C[0] + dfz * C[1];   // z -> y -> x as :1044-1053
                const double vmp = az * C[2] + dfz * C[3];
                const double vpm = az * C[4] + dfz * C[5];
                const double vpp = az * C[6] + dfz * C[7];
                const double vm = ay * vmm + dfy * vmp;
                const double vp = ay * vpm + dfy * vpp;
                e_total = ax * vm + dfx * vp;                // :1061 summed over the grids
                if (FMODE != kForceNone) {                   // :1066-1071
                    const double gx = vp - vm;
                    const double gy = (vmp - vmm) * ax + (vpp - vpm) * dfx;
                    const double gz = ((C[1] - C[0]) * ay + (C[3] - C[2]) * dfy) * ax + ((C[5] - C[4]) * ay + (C[7] - C[6]) * dfy) * dfx;
                    sx = (float) (gx * G.inv_spacing[0]);
                    sy = (float) (gy * G.inv_spacing[1]);
                    sz = (float) (gz * G.inv_spacing[2]);
                }
            }
        }
    }
    float Fx, Fy, Fz;   // :1072, :1082
    if (NG == 1) {
        Fx = -sx * (float) G.inv_spacing[0];
        Fy = -sy * (float) G.inv_spacing[1];
        Fz = -sz * (float) G.inv_spacing[2];
    } else {
        Fx = -sx;
        Fy = -sy;
        Fz = -sz;
    }
    if (active && !inside) {   // :1093-1117 (inside atoms with scale 0 take that branch too and add exactly 0)
        const double* mine = p.pos + 3 * (size_t) gidx;   // re-read (rare path): x, y, z need not stay in registers
        const RestraintAll<NG> r = restraint_all<NG>(p, mine[0], mine[1], mine[2]);
#pragma unroll
        for (int g = 0; g < NG; g++) {
            e_total += r.e[g];
            if (GE) e_g[GE ? g : 0] = r.e[g];
        }
        Fx -= r.fx;
        Fy -= r.fy;
        Fz -= r.fz;
    }

    // ---- forces --------------------------------------------------------------------------------------------------------
    // STORE modes without indirection: a full warp's 32 forces are 768 (F64) or 384 (F32) contiguous bytes. They go
    // through the warp's smem slice and leave as coalesced 16-byte stores (the mirror image of the position staging)
    // instead of 96 scalar stores at stride 24/12 — which matters most when `forces` is host-mapped memory (PCIe write
    // TLPs of 128 bytes instead of 8): gfb_kernel_execute_host's zero-copy path.
    // Everything above only READ inputs that no evaluation launch writes (positions, grids, scaling factors). From here on
    // the kernel writes what the previous launch may still be writing or accumulating: wait for it to finish.
    // Exception: the ADD modes under programmatic dependent launch. Their force updates are commutative atomics, so they
    // may interleave with the previous evaluation launch's (the caller's promise for launch overlap covers d_forces: the
    // kernel launched just before only ACCUMULATES into it); issuing them before the wait leaves a block parked at the
    // wait with nothing but its energy atomics to do, which shortens the bubble between two small launches.
    constexpr bool kAdd = kAddMode;
    const bool early_forces = kAdd && p.pdl != 0u && p.gather == nullptr;   // uniform
    auto add_forces = [&]() {
        if (FMODE == GFB_FORCE_FIXED_ADD) {   // OpenMM's 2^32 fixed point, gridForce.cu:487-499
            const unsigned long long ax = (unsigned long long) __float2ll_rz(Fx * 4294967296.f);
            const unsigned long long ay = (unsigned long long) __float2ll_rz(Fy * 4294967296.f);
            const unsigned long long az = (unsigned long long) __float2ll_rz(Fz * 4294967296.f);
            red_add_u64(ffix + gidx, ax);
            red_add_u64(ffix + p.force_stride + gidx, ay);
            red_add_u64(ffix + 2 * p.force_stride + gidx, az);
        } else {
            double* f = fdbl + 3 * (size_t) gidx;
            red_add_f64(f, (double) Fx);
            red_add_f64(f + 1, (double) Fy);
            red_add_f64(f + 2, (double) Fz);
        }
    };
    if (kAdd && early_forces && active && p.forces) add_forces();
    const bool park = defer && !waited && it < (unsigned) kDefer;   // uniform: this tile's energies are parked
    if (!park && !waited) {   // PERSIST: exactly the tile it == kDefer
        asm volatile("griddepcontrol.wait;" ::: "memory");
        if (defer) flush_parked((unsigned) kDefer);
    }
    if (!defer && p.energies_clear)   // grid-stride, as below: the next accumulator can outnumber the launch's threads
        for (unsigned c = t; c < (unsigned) (p.n_replicas * p.n_slots); c += gridDim.x * blockDim.x) p.energies_clear[c] = 0.0;
    if (p.atom_energies && active) p.atom_energies[a] = e_total;   // uniform branch (never with p.defer)
    // Force writes. In a launch that carries the fused energy gather they come AFTER the energies and the block's gather
    // ticket (the ticket's fence then waits for the energy atomics only); otherwise right here.
    auto write_forces = [&]() {
        constexpr bool kStore = FMODE == GFB_FORCE_F64_STORE || FMODE == GFB_FORCE_F32_STORE;
        const bool stage_f = kStore && p.forces != nullptr && plain && (t - lane) + 32u <= total &&
                             (reinterpret_cast<uintptr_t>(p.forces) & 15) == 0;   // warp-uniform
        if (kStore && stage_f) {
            __syncwarp();   // every lane has consumed its record from this slice
            if (FMODE == GFB_FORCE_F64_STORE) {
                double* const s_f = reinterpret_cast<double*>(s_pos2 + (tid >> 5) * kWarpSlice16);
                s_f[3 * lane] = (double) Fx;
                s_f[3 * lane + 1] = (double) Fy;
                s_f[3 * lane + 2] = (double) Fz;
                __syncwarp();
                const double2* const s_f2 = reinterpret_cast<const double2*>(s_f);
                double2* const dst = reinterpret_cast<double2*>(static_cast<double*>(p.forces) + 3 * (size_t) (t - lane));
                dst[lane] = s_f2[lane];
                if (lane < 16) dst[32 + lane] = s_f2[32 + lane];
            } else {   // F32: 384 bytes = 24 x 16
                float* const s_f = reinterpret_cast<float*>(s_pos2 + (tid >> 5) * kWarpSlice16);
                s_f[3 * lane] = Fx;
                s_f[3 * lane + 1] = Fy;
                s_f[3 * lane + 2] = Fz;
                __syncwarp();
                const float4* const s_f4 = reinterpret_cast<const float4*>(s_f);
                float4* const dst = reinterpret_cast<float4*>(static_cast<float*>(p.forces) + 3 * (size_t) (t - lane));
                if (lane < 24) dst[lane] = s_f4[lane];
            }
        }
        if (kAdd && !early_forces && active && p.forces) add_forces();
        if (kStore && active && p.forces && !stage_f) {
            if (FMODE == GFB_FORCE_F32_STORE) {
                float* f = static_cast<float*>(p.forces) + 3 * (size_t) gidx;
                f[0] = Fx;
                f[1] = Fy;
                f[2] = Fz;
            } else {
                double* f = fdbl + 3 * (size_t) gidx;
                f[0] = (double) Fx;
                f[1] = (double) Fy;
                f[2] = (double) Fz;
            }
        }
    };
    if (p.gather == nullptr && !park) write_forces();   // parked tiles: forces went out early (ADD) or are not wanted

    // ---- energies ------------------------------------------------------------------------------------------------------
    if (SINGLE) {
        __shared__ double warp_sum[kBlock / 32];
        if (GE) {   // per-grid energies: warp sums -> one atomic per block and grid (a plain store when one block is the call)
            __shared__ double warp_ge[kBlock / 32][GE ? NG : 1];
#pragma unroll
            for (int g = 0; g < (GE ? NG : 1); g++) {
                double eg = e_g[g];
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) eg += __shfl_xor_sync(kFull, eg, off);
                if (lane == 0) warp_ge[tid >> 5][g] = eg;
            }
            __syncthreads();
            if (tid < (GE ? NG : 1)) {
                double b = 0.0;
#pragma unroll
                for (int w = 0; w < kBlock / 32; w++) b += warp_ge[w][tid];
                if (p.energy_store) p.grid_energies[tid] = b;
                else red_add_f64(p.grid_energies + tid, b);
            }
        }
        if (p.energies) {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) e_total += __shfl_xor_sync(kFull, e_total, off);
            if (lane == 0) warp_sum[tid >> 5] = e_total;
            __syncthreads();
            if (tid < 32) {
                double b = tid < kBlock / 32 ? warp_sum[tid] : 0.0;
#pragma unroll
                for (int off = kBlock / 64; off > 0; off >>= 1) b += __shfl_xor_sync(kFull, b, off);
                if (tid == 0) {
                    if (p.energy_store) *p.energies = b;
                    else red_add_f64(p.energies, b);
                }
            }
        }
    } else if (p.energies || GE) {
        unsigned heads;
        const unsigned span = run_span(key, lane, heads);
        const bool head = key >= 0 && ((heads >> lane) & 1u);
        if (GE) {
#pragma unroll
            for (int g = 0; g < (GE ? NG : 1); g++) {
                double eg = e_g[g];
                run_sum(eg, span);
                if (head) red_add_f64(p.grid_energies + (size_t) key * NG + g, eg);
            }
        }
        if (p.energies) {
            run_sum(e_total, span);
            if (kCanDefer && park) {
                s_def_e[(kCanDefer ? it : 0u) * kBlock + tid] = e_total;
                s_def_k[(kCanDefer ? it : 0u) * kBlock + tid] = head ? key : -1;
            } else if (head) {
                red_add_f64(p.energies + key, e_total);
            }
        }
    }
    if (p.gather) {   // uniform branch: fused energy gather of a replica-sharded run (one tile per block)
        const int copier = gather_ticket<kBlock>(p);
        write_forces();
        if (copier >= 0) gather_copy<kBlock>(p, (unsigned) copier);
    }
    if (PERSIST) __syncwarp();   // the warp's smem slice is rewritten by the next tile's positions
    it++;
    } while (PERSIST && blockIdx.x + it * gridDim.x < n_tiles);
    if (defer) {
        if (it <= (unsigned) kDefer) {   // every tile of this block was parked: the one wait comes here
            asm volatile("griddepcontrol.wait;" ::: "memory");
            flush_parked(it);
        }
        if (p.energies_clear) {
            const unsigned n_clear = (unsigned) (p.n_replicas * p.n_slots);
            for (unsigned c = blockIdx.x * kBlock + threadIdx.x; c < n_clear; c += gridDim.x * kBlock) p.energies_clear[c] = 0.0;
        }
    }
}

}  // namespace gfb
#endif
