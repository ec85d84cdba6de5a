// DOUBLE-precision twin of gf_eval_lines_kernel (gf_eval_lines.cuh) for 2-4 packed-cell grids of one geometry without
// inv-power: the reference's own arithmetic (ReferenceGridForceKernels.cpp:646-715, 1016-1121 is FP64 throughout), at the
// MIXED kernel's traffic efficiency.
//
// Layout: the FP64 packed cells of all grids are woven into ONE 256-byte record per cell (4 slots x 8 doubles,
// gf_interleave_cells_kernel with 64-byte slots) = two full 128-byte lines, instead of one 64-byte stencil out of a
// different 128-byte line per grid (general kernel: 3 lines fetched for 192 useful bytes, C5 1.18 GB of DRAM traffic for
// 825 MB algorithmic). A warp fetches its 32 records with 16 warp-wide cp.async (LDGSTS.128): sixteen lanes copy the
// sixteen 16-byte granules of the SAME record, two records = four full lines per instruction. The data lands in an
// XOR-swizzled 8 KB slice of shared memory per warp; the owning lane reads each grid's 8 corners with 4 LDS.128 right
// before use. Index math divides exactly, as the reference does (classify<true>); the gradient is divided by the spacing
// (:1072). Forces FP64 (or OpenMM fixed point), energies FP64.
#ifndef GF_EVAL_LINES_F64_CUH_
#define GF_EVAL_LINES_F64_CUH_

#include "gf_eval_lines.cuh"

namespace gfb {

constexpr int kLinesF64Block = 128;

__device__ __forceinline__ void lds128d(unsigned addr, double* v) {
    asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v[0]), "=d"(v[1]) : "r"(addr) : "memory");
}

//   NG 2..4 grids per record; FMODE gfb_force_mode (F32_STORE is served as scalar float stores) or kForceNone;
//   SINGLE one replica and no energy slots; GE per-grid energies wanted.
template <int NG, int FMODE, bool SINGLE, bool GE>
__global__ void __launch_bounds__(kLinesF64Block, 6) gf_eval_lines_f64_kernel(const __grid_constant__ EvalParams p) {
    constexpr int kBlock = kLinesF64Block;
    constexpr unsigned kWarpSlice16 = 512;   // 8 KB per warp: first the warp's 32 positions, then its 32 records of 256 bytes
    __shared__ __align__(128) double2 s_buf[(kBlock / 32) * kWarpSlice16];

    const unsigned tid = threadIdx.x;
    const unsigned lane = tid & 31u;
    const unsigned t = blockIdx.x * kBlock + tid;
    const unsigned total = (unsigned) p.total;
    const bool active = t < total;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // see gf_eval_lines_kernel

    const unsigned a = (p.order != nullptr && active) ? (unsigned) p.order[t] : t;
    unsigned rep = 0, ia = a;
    if (!SINGLE) {
        rep = __umulhi(a, p.div_magic);
        ia = a - rep * (unsigned) p.n_atoms;
        if (ia >= (unsigned) p.n_atoms) {
            ia -= (unsigned) p.n_atoms;
            rep++;
        }
    }
    if (!active) ia = 0;
    const bool plain = p.particles == nullptr && p.n_particles == p.n_atoms && p.order == nullptr;   // uniform
    unsigned gidx = t;
    if (!plain) gidx = rep * (unsigned) p.n_particles + (p.particles ? (unsigned) p.particles[ia] : ia);
    int key = -1;
    if (active) key = p.slots ? (int) rep * p.n_slots + p.slots[ia] : (int) rep;

    // ---- positions: 768 contiguous bytes per warp through the warp's own slice (as gf_eval_lines_kernel) ------------
    double x = 0.0, y = 0.0, z = 0.0;
    double2* const s_warp = s_buf + (tid >> 5) * kWarpSlice16;
    const bool staged = plain && (reinterpret_cast<uintptr_t>(p.pos) & 15) == 0;   // uniform
    if (staged) {
        const unsigned w0 = t - lane;
        if (w0 < total) {
            const double2* src = reinterpret_cast<const double2*>(p.pos + 3 * (size_t) w0);
            const unsigned left = 3u * (total - w0);
            double2 va = make_double2(0.0, 0.0), vb = make_double2(0.0, 0.0);
            if (2 * lane + 1 < left) asm volatile("ld.global.cs.v2.f64 {%0,%1}, [%2];" : "=d"(va.x), "=d"(va.y) : "l"(src + lane));
            else if (2 * lane < left) va.x = load_stream(reinterpret_cast<const double*>(src + lane));
            if (lane < 16) {
                if (2 * (32 + lane) + 1 < left) asm volatile("ld.global.cs.v2.f64 {%0,%1}, [%2];" : "=d"(vb.x), "=d"(vb.y) : "l"(src + 32 + lane));
                else if (2 * (32 + lane) < left) vb.x = load_stream(reinterpret_cast<const double*>(src + 32 + lane));
            }
            s_warp[lane] = va;
            if (lane < 16) s_warp[32 + lane] = vb;
        }
        __syncwarp();
        const double* mine = reinterpret_cast<const double*>(s_warp) + 3 * lane;
        x = mine[0];
        y = mine[1];
        z = mine[2];
        __syncwarp();
    } else if (active) {
        const double* mine = p.pos + 3 * (size_t) gidx;
        x = load_stream(mine);
        y = load_stream(mine + 1);
        z = load_stream(mine + 2);
    }

    // ---- classification: exact FP64 division, the reference's expressions (:687-715) ---------------------------------
    const GridView& G = p.grid[0];
    AtomCell c = classify<true>(G, x, y, z);
    c.inside = c.inside && active;
    unsigned cell = 0xffffffffu;
    if (c.inside) cell = ((unsigned) c.ix * (unsigned) G.nc[1] + (unsigned) c.iy) * (unsigned) G.nc[2] + (unsigned) c.iz;

    // ---- records: round i brings the records of the atoms of lanes 2i and 2i+1, sixteen lanes per record -------------
    const unsigned warp_base = (unsigned) __cvta_generic_to_shared(s_warp);
    const unsigned gran = lane & 15u, half = lane >> 4;
    const char* lane_base = static_cast<const char*>(p.lines) + 16u * gran;
#pragma unroll
    for (int i = 0; i < 16; i++) {
        const unsigned A = 2u * i + half;
        const unsigned cc = __shfl_sync(kFull, cell, (int) A);
        if (cc != 0xffffffffu && gran < 4u * NG)
            cp_async16(warp_base + A * 256u + ((((gran & 7u) ^ (A & 7u)) | (gran & 8u)) << 4), lane_base + 256ull * cc);
    }
    cp_async_wait_all();
    __syncwarp();

    double e_g[GE ? NG : 1];
    double e_total = 0.0;
    double Fx = 0.0, Fy = 0.0, Fz = 0.0;
    if (GE) {
#pragma unroll
        for (int g = 0; g < (GE ? NG : 1); g++) e_g[g] = 0.0;
    }
    const unsigned rbase = warp_base + lane * 256u;
    const unsigned sw = lane & 7u;
    // As in gf_eval_lines_kernel: trilinear interpolation is linear in the corner values and the grids share cell and
    // fractions, so the scaled corners are summed over the grids and value and gradient are formed once per atom — one
    // interpolation and three divisions by the spacing (:1072) instead of NG of each (an FP64 division is ~30
    // instructions). Sums of products in FP64: the result differs from the per-grid evaluation by rounding (1e-16).
    if (c.inside) {
        double C[8];
#pragma unroll
        for (int k = 0; k < 8; k++) C[k] = 0.0;
#pragma unroll
        for (int g = 0; g < NG; g++) {
            const double s = p.grid[g].scaling[ia];
            if (s != 0.0) {   // :706
                double v[8];
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const unsigned gr = 4u * g + q;   // granule of the record
                    lds128d(rbase + ((((gr & 7u) ^ sw) | (gr & 8u)) << 4), v + 2 * q);
                }
                if (GE) {   // per-grid energies wanted: this grid's value on its own as well
                    double val, dx, dy, dz;
                    trilinear<double>(v, c.fx, c.fy, c.fz, val, dx, dy, dz);
                    e_g[GE ? g : 0] = s * val;
                }
#pragma unroll
                for (int k = 0; k < 8; k++) C[k] = fma(s, v[k], C[k]);
            }
        }
        double val, dx, dy, dz;
        trilinear<double>(C, c.fx, c.fy, c.fz, val, dx, dy, dz);   // :1039-1071 on the summed corners
        e_total = val;                                              // :1061 summed over the grids
        if (FMODE != kForceNone) {
            Fx = -(dx / G.spacing[0]);                              // :1072, :1082
            Fy = -(dy / G.spacing[1]);
            Fz = -(dz / G.spacing[2]);
        }
    } else if (active) {          // :1093-1117, every force adds its own wall
#pragma unroll
        for (int g = 0; g < NG; g++) {
            double e = 0.0;
            accumulate_restraint(p.grid[g], x, y, z, e, Fx, Fy, Fz);
            e_total += e;
            if (GE) e_g[GE ? g : 0] = e;
        }
    }

    // ---- writes start here (programmatic dependent launch: wait for the previous grid) ---------------------------------
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (p.energies_clear)   // grid-stride: with energy slots the next accumulator can have more entries than the launch has threads
        for (unsigned c = t; c < (unsigned) (p.n_replicas * p.n_slots); c += gridDim.x * blockDim.x) p.energies_clear[c] = 0.0;
    if (p.atom_energies && active) p.atom_energies[a] = e_total;
    auto write_forces = [&]() {   // deferred behind the gather ticket in a gather launch (see gf_eval_lines_kernel)
        const bool stage_f = FMODE == GFB_FORCE_F64_STORE && p.forces != nullptr && plain && (t - lane) + 32u <= total &&
                             (reinterpret_cast<uintptr_t>(p.forces) & 15) == 0;   // warp-uniform
        if (FMODE == GFB_FORCE_F64_STORE && stage_f) {
            __syncwarp();   // every lane has consumed its record from this slice
            double* const s_f = reinterpret_cast<double*>(s_warp);
            s_f[3 * lane] = Fx;
            s_f[3 * lane + 1] = Fy;
            s_f[3 * lane + 2] = Fz;
            __syncwarp();
            double2* const dst = reinterpret_cast<double2*>(static_cast<double*>(p.forces) + 3 * (size_t) (t - lane));
            dst[lane] = s_warp[lane];
            if (lane < 16) dst[32 + lane] = s_warp[32 + lane];
        }
        if (FMODE != kForceNone && active && p.forces) {
            if (FMODE == GFB_FORCE_FIXED_ADD) {   // OpenMM's 2^32 fixed point, gridForce.cu:487-499
                unsigned long long* f = static_cast<unsigned long long*>(p.forces);
                const double scale = 4294967296.0;
                red_add_u64(f + gidx, (unsigned long long) (long long) (Fx * scale));
                red_add_u64(f + p.force_stride + gidx, (unsigned long long) (long long) (Fy * scale));
                red_add_u64(f + 2 * p.force_stride + gidx, (unsigned long long) (long long) (Fz * scale));
            } else if (FMODE == GFB_FORCE_F32_STORE) {
                float* f = static_cast<float*>(p.forces) + 3 * (size_t) gidx;
                f[0] = (float) Fx;
                f[1] = (float) Fy;
                f[2] = (float) Fz;
            } else {
                double* f = static_cast<double*>(p.forces) + 3 * (size_t) gidx;
                if (FMODE == GFB_FORCE_F64_STORE) {
                    if (!stage_f) {
                        f[0] = Fx;
                        f[1] = Fy;
                        f[2] = Fz;
                    }
                } else {
                    red_add_f64(f, Fx);
                    red_add_f64(f + 1, Fy);
                    red_add_f64(f + 2, Fz);
                }
            }
        }
    };
    if (p.gather == nullptr) write_forces();

    // ---- energies (as gf_eval_lines_kernel) ------------------------------------------------------------------------------
    if (SINGLE) {
        __shared__ double warp_sum[kBlock / 32];
        if (GE) {
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
            if (tid == 0) {
                double b = 0.0;
#pragma unroll
                for (int w = 0; w < kBlock / 32; w++) b += warp_sum[w];
                if (p.energy_store) *p.energies = b;
                else red_add_f64(p.energies, b);
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
            if (head) red_add_f64(p.energies + key, e_total);
        }
    }
    if (p.gather) {
        const int copier = gather_ticket<kBlock>(p);
        write_forces();
        if (copier >= 0) gather_copy<kBlock>(p, (unsigned) copier);
    }
}

}  // namespace gfb
#endif
