// Cubic B-spline evaluation kernel for MIXED-precision grids in the BSPLINE brick layout that share one geometry
// (GridForce::setInterpolationMethod(1); reference platforms/reference/src/ReferenceGridForceKernels.cpp:727-795), and,
// with METHOD = 2, the tricubic Hermite evaluation (setInterpolationMethod(2), :796-893) on HERMITE records.
// Everything else B-spline (DOUBLE precision, grids of different geometry, an evaluation order) runs
// gf_eval_kernel<S, BSPLINE, ...> in gf_kernels.cuh, which holds the layout's description and the reference arithmetic.
//
// Why a second kernel. The general kernel reads a stencil with 8 LDG.E.256 per lane and grid. An SM retires about one
// gather LANE per clock whatever the load width (DESIGN.md §3), so the L1 pipeline bounds it. Here a stencil's two
// 128-byte records are fetched as two full LINES: eight lanes copy the eight 16-byte rows of one record with cp.async
// (LDGSTS.128), so ONE warp instruction brings the 4 records of two atoms (4 L2 requests of one line each) instead of
// 8 x 32 B from one lane. The records land in an XOR-swizzled slice of shared memory (8 KB per warp, no bank conflicts on
// either side); the owning lane then reads its 64 values with 16 LDS.128. Per warp and grid: 16 LDGSTS + 16 x 32 LDS.128.
#ifndef GF_EVAL_BSPLINE_CUH_
#define GF_EVAL_BSPLINE_CUH_

#include "gf_eval_lines.cuh"

namespace gfb {

#ifndef GFB_BS_MINBLOCKS
#define GFB_BS_MINBLOCKS 4
#endif
constexpr int kBsBlock = 128;                // 4 warps x 8 KB of bricks: 6 blocks (24 warps, 192 KB of smem) per SM
constexpr unsigned kBsWarpBytes = 32 * 256;  // 32 atoms x 2 records x 128 bytes

// Per-atom interpolation weights, computed once and used for every grid (all grids share the geometry).
struct BsWeights {
    double bx[4], by[4], bz[4];            // value path, FP64
    float dbx[4], dby[4], dbz[4];          // gradient path, FP32
};
__device__ __forceinline__ void bspline_weights(double fx, double fy, double fz, BsWeights& w) {
    double d[4];
    bspline_basis(fx, w.bx, d);   // :741-748
#pragma unroll
    for (int k = 0; k < 4; k++) w.dbx[k] = (float) d[k];
    bspline_basis(fy, w.by, d);
#pragma unroll
    for (int k = 0; k < 4; k++) w.dby[k] = (float) d[k];
    bspline_basis(fz, w.bz, d);
#pragma unroll
    for (int k = 0; k < 4; k++) w.dbz[k] = (float) d[k];
}

// One lane's stencil out of its 256-byte smem region: 16 granules of 16 bytes, granule 4*i + r = row r of x-plane i,
// stored at position (4*i + r) ^ (lane & 7). Value FP64 from the FP32 points, gradient FP32 over the points minus the
// stencil's first point (see bspline_interpolate: the error then scales with |grad V|, not with |V|).
__device__ __forceinline__ void bspline_from_smem(unsigned rbase, unsigned sw, const BsWeights& w, double& val, float& gx,
                                                  float& gy, float& gz) {
    val = 0.0;
    gx = gy = gz = 0.f;
    float ref = 0.f;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        double pv = 0.0;
        float pdy = 0.f, pdz = 0.f;
#pragma unroll
        for (int r = 0; r < 4; r++) {
            float v[4];
            lds128(rbase + (((4u * i + r) << 4) ^ sw), v);
            if (i == 0 && r == 0) ref = v[0];
            double rz = 0.0;
            float rzs = 0.f, drz = 0.f;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const float d = v[k] - ref;
                rz = fma(w.bz[k], (double) v[k], rz);
                rzs = fmaf((float) w.bz[k], d, rzs);
                drz = fmaf(w.dbz[k], d, drz);
            }
            pv = fma(w.by[r], rz, pv);
            pdy = fmaf(w.dby[r], rzs, pdy);
            pdz = fmaf((float) w.by[r], drz, pdz);
        }
        val = fma(w.bx[i], pv, val);
        gx = fmaf(w.dbx[i], (float) (pv - (double) ref), gx);
        gy = fmaf((float) w.bx[i], pdy, gy);
        gz = fmaf((float) w.bx[i], pdz, gz);
    }
}

// Tricubic Hermite (interpolation method 2) out of the same 256-byte smem region, for HERMITE records (filled by flat
// index, gf_repack_bspline_kernel<float, true>): the point at offsets (i-1, r-1, k-1) is element k of granule 4*i + r.
// 12 of the 16 granules are read (rows 1-2 of every x-plane, rows 0 and 3 of planes 1-2); arithmetic FP64 (tricubic_eval).
// volatile: ptxas otherwise narrows the 16-byte loads of which only elements 1-2 are used (planes 0 and 3, rows 0 and 3) to
// pairs of 4-byte loads, and 4-byte loads of this swizzle are 4-way bank conflicts (lanes l, l+8, l+16, l+24 share a
// bank; a 16-byte load is served a quarter-warp at a time and has none): ncu counted 14.2 M conflicts per launch against
// 0.13 M for the B-spline arithmetic on the same slice.
__device__ __forceinline__ void lds128_whole(unsigned addr, float* v) {
    asm volatile("ld.volatile.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(addr) : "memory");
}
struct TricubicSmem {
    float g[4][4][4];      // [i][r][k]; entries of the four granules never read stay unset
    __device__ __forceinline__ double operator()(int i, int r, int k) const { return (double) g[i][r][k]; }
};
__device__ __forceinline__ void tricubic_from_smem(unsigned rbase, unsigned sw, bool xin, bool yin, bool zin, const TricubicWeights& w,
                                                   double& val, double& gx, double& gy, double& gz) {
    TricubicSmem V;
    // in the order tricubic_eval consumes them: rows 1 and 2 of the four x-planes (x stage), then rows 0 and 3 of planes 1-2
#pragma unroll
    for (int r = 1; r <= 2; r++) {
#pragma unroll
        for (int i = 0; i < 4; i++) lds128_whole(rbase + (((4u * i + r) << 4) ^ sw), V.g[i][r]);
    }
#pragma unroll
    for (int r = 0; r <= 3; r += 3) {
#pragma unroll
        for (int i = 1; i <= 2; i++) lds128_whole(rbase + (((4u * i + r) << 4) ^ sw), V.g[i][r]);
    }
    tricubic_eval(V, xin, yin, zin, w, val, gx, gy, gz);
}

//   SINGLE  one replica and no energy slots (block-level energy reduction); the force mode is p.force_mode (launch-uniform)
//   METHOD  1 cubic B-spline on BSPLINE records, 2 tricubic Hermite on HERMITE records (same fetch, other arithmetic)
template <bool SINGLE, int METHOD>
__global__ void __launch_bounds__(kBsBlock, GFB_BS_MINBLOCKS) gf_eval_bspline_kernel(const __grid_constant__ EvalParams p) {
    __shared__ __align__(128) unsigned char s_tiles[(kBsBlock / 32) * kBsWarpBytes];

    const unsigned tid = threadIdx.x;
    const unsigned lane = tid & 31u;
    const unsigned t = blockIdx.x * kBsBlock + tid;
    const unsigned total = (unsigned) p.total;
    const bool active = t < total;
    if (p.energies_clear)   // grid-stride: with energy slots the next accumulator can have more entries than the launch has threads
        for (unsigned c = t; c < (unsigned) (p.n_replicas * p.n_slots); c += gridDim.x * blockDim.x) p.energies_clear[c] = 0.0;

    // ---- who am I (as gf_eval_lines_kernel) ----------------------------------------------------------------------
    unsigned rep = 0, ia = t;
    if (!SINGLE) {
        rep = __umulhi(t, p.div_magic);
        ia = t - rep * (unsigned) p.n_atoms;
        if (ia >= (unsigned) p.n_atoms) {
            ia -= (unsigned) p.n_atoms;
            rep++;
        }
    }
    if (!active) ia = 0;
    const bool plain = p.particles == nullptr && p.n_particles == p.n_atoms;   // uniform
    unsigned gidx = t;
    if (!plain) gidx = rep * (unsigned) p.n_particles + (p.particles ? (unsigned) p.particles[ia] : ia);
    int key = -1;
    if (active) key = p.slots ? (int) rep * p.n_slots + p.slots[ia] : (int) rep;

    // ---- position (three streaming loads; a warp's positions are 768 contiguous bytes when no indirection is in play)
    double x = 0.0, y = 0.0, z = 0.0;
    if (active) {
        const double* mine = p.pos + 3 * (size_t) gidx;
        x = load_stream(mine);
        y = load_stream(mine + 1);
        z = load_stream(mine + 2);
    }

    // ---- classification (:687-715), bit-exact; all grids share grid 0's geometry ------------------------------------
    const GridView& G = p.grid[0];
    const FastCell fc = classify_fast(G, p.near_int, x, y, z, active);
    const bool inside = fc.inside;
    const unsigned brick0 = inside ? (unsigned) ((fc.ix * G.nc[1] + fc.iy) * G.nc[2] + fc.iz) : 0xffffffffu;   // record (ix,iy,iz)
    const unsigned plane_recs = (unsigned) (G.nc[1] * G.nc[2]);   // records from one x-plane to the next

    const unsigned warp_base = (unsigned) __cvta_generic_to_shared(s_tiles) + (tid >> 5) * kBsWarpBytes;
    const unsigned sub = lane & 15u, half = lane >> 4;   // sub = 4*plane + row: which 16 bytes of an atom's 256 this lane copies
    const unsigned rbase = warp_base + lane * 256u;
    const unsigned sw = (lane & 7u) << 4;

    BsWeights wts;
    TricubicWeights tw;
    if constexpr (METHOD == 1) bspline_weights(fc.fx, fc.fy, fc.fz, wts);
    else tricubic_weights(fc.fx, fc.fy, fc.fz, tw);
    const bool xin = fc.ix > 0 && fc.ix < G.nc[0], yin = fc.iy > 0 && fc.iy < G.nc[1], zin = fc.iz > 0 && fc.iz < G.nc[2];   // :817, :849, :866

    double e_total = 0.0;
    double Fx = 0.0, Fy = 0.0, Fz = 0.0;
    unsigned heads = 0;
    unsigned span = 0;
    bool head = false;
    if (!SINGLE) {
        span = run_span(key, lane, heads);
        head = key >= 0 && ((heads >> lane) & 1u);
    }

    for (int g = 0; g < p.n_grids; g++) {
        const GridView& Gg = p.grid[g];
        const double s = active ? Gg.scaling[ia] : 0.0;
        const bool interp = inside && s != 0.0;   // :706
        // ---- fetch: round i brings the four bricks of the atoms of lanes 2i and 2i+1, sixteen lanes per atom --------
        const unsigned mybrick = interp ? brick0 : 0xffffffffu;
        // sub = 8*(which record: a = ix | ix+2) + 4*(which plane of it) + row: 16 bytes of a 128-byte record
        const char* lane_base = static_cast<const char*>(Gg.cells) + 16u * (sub & 7u) + 128ull * (unsigned long long) (2u * (sub >> 3)) * plane_recs;
        __syncwarp();   // the previous grid's bricks have been consumed
#pragma unroll 8
        for (int i = 0; i < 16; i++) {
            const unsigned A = 2u * (unsigned) i + half;
            const unsigned bk = __shfl_sync(kFull, mybrick, (int) A);
            if (bk != 0xffffffffu) cp_async16(warp_base + A * 256u + ((sub ^ (A & 7u)) << 4), lane_base + 128ull * bk);
        }
        cp_async_wait_all();
        __syncwarp();
        // ---- evaluate -----------------------------------------------------------------------------------------------
        double e_g = 0.0;
        if (METHOD == 2 && interp) {
            double val, gx, gy, gz;
            tricubic_from_smem(rbase, sw, xin, yin, zin, tw, val, gx, gy, gz);
            tricubic_epilogue(Gg, s, val, gx, gy, gz, e_g, Fx, Fy, Fz);      // :879-893
        } else if (interp) {
            double val;
            float dx, dy, dz;
            bspline_from_smem(rbase, sw, wts, val, dx, dy, dz);
            double gx = (double) (dx * (float) Gg.inv_spacing[0]);   // :790
            double gy = (double) (dy * (float) Gg.inv_spacing[1]);
            double gz = (double) (dz * (float) Gg.inv_spacing[2]);
            if (Gg.inv_power > 0.0) {   // :778-787
                const double base = val;
                val = pow(base, Gg.inv_power);
                const double pf = Gg.inv_power * pow(base, Gg.inv_power - 1.0);
                gx *= pf;
                gy *= pf;
                gz *= pf;
            }
            e_g = s * val;   // :793
            Fx -= s * gx;    // :794
            Fy -= s * gy;
            Fz -= s * gz;
        } else if (active) {   // :1093-1117
            accumulate_restraint(Gg, x, y, z, e_g, Fx, Fy, Fz);
        }
        e_total += e_g;
        if (p.grid_energies) {   // uniform branch
            double eg = e_g;
            if (SINGLE) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) eg += __shfl_xor_sync(kFull, eg, o);
                if (lane == 0) red_add_f64(p.grid_energies + g, eg);
            } else {
                run_sum(eg, span);
                if (head) red_add_f64(p.grid_energies + (size_t) key * p.n_grids + g, eg);
            }
        }
    }

    if (p.atom_energies && active) p.atom_energies[t] = e_total;   // uniform branch

    // ---- forces --------------------------------------------------------------------------------------------------------
    if (active && p.forces) {
        const int fmode = p.force_mode;   // launch-uniform
        if (fmode == GFB_FORCE_FIXED_ADD) {   // OpenMM's 2^32 fixed point, gridForce.cu:487-499
            unsigned long long* f = static_cast<unsigned long long*>(p.forces);
            const double scale = 4294967296.0;
            red_add_u64(f + gidx, (unsigned long long) (long long) (Fx * scale));
            red_add_u64(f + p.force_stride + gidx, (unsigned long long) (long long) (Fy * scale));
            red_add_u64(f + 2 * p.force_stride + gidx, (unsigned long long) (long long) (Fz * scale));
        } else if (fmode == GFB_FORCE_F32_STORE) {
            float* f = static_cast<float*>(p.forces) + 3 * (size_t) gidx;
            f[0] = (float) Fx;
            f[1] = (float) Fy;
            f[2] = (float) Fz;
        } else {
            double* f = static_cast<double*>(p.forces) + 3 * (size_t) gidx;
            if (fmode == GFB_FORCE_F64_STORE) {
                f[0] = Fx;
                f[1] = Fy;
                f[2] = Fz;
            } else {
                red_add_f64(f, Fx);
                red_add_f64(f + 1, Fy);
                red_add_f64(f + 2, Fz);
            }
        }
    }

    // ---- energies ------------------------------------------------------------------------------------------------------
    if (p.energies) {   // uniform branch
        if (SINGLE) {
            __shared__ double warp_sum[kBsBlock / 32];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) e_total += __shfl_xor_sync(kFull, e_total, o);
            if (lane == 0) warp_sum[tid >> 5] = e_total;
            __syncthreads();
            if (tid == 0) {
                double b = 0.0;
#pragma unroll
                for (int w = 0; w < kBsBlock / 32; w++) b += warp_sum[w];
                if (p.energy_store) *p.energies = b;
                else red_add_f64(p.energies, b);
            }
        } else {
            run_sum(e_total, span);
            if (head) red_add_f64(p.energies + key, e_total);
        }
    }
}

}  // namespace gfb
#endif
