// DOUBLE-precision twin of gf_eval_bspline_kernel (gf_eval_bspline.cuh): cubic B-spline grids in the BSPLINE record layout
// (METHOD 1) or tricubic Hermite grids in the HERMITE record layout (METHOD 2, :796-893, arithmetic tricubic_eval)
// that share one geometry, no evaluation order (GridForce::setInterpolationMethod(1) on a "double" platform; reference
// platforms/reference/src/ReferenceGridForceKernels.cpp:727-795, whose arithmetic is FP64 throughout).
//
// The general kernel (gf_eval_kernel<double, BSPLINE>) reads the 64 doubles of a stencil with 16 LDG.E.256 per lane and
// grid and needs 255 registers (one block per SM): 2.5 ms on the C5 shape. Here a stencil's two 256-byte records are
// fetched as four full LINES: the 32 lanes of a warp copy the 32 granules of 16 bytes of ONE atom's stencil with cp.async
// (LDGSTS.128), 32 rounds per grid, into an XOR-swizzled 16 KB slice of shared memory per warp; the owning lane then reads
// its 64 values with 32 conflict-free LDS.128. The arithmetic is bspline_interpolate<double>'s (gf_kernels.cuh),
// operation for operation, so the two kernels agree bit for bit; index math divides exactly as the reference does.
// 64-thread blocks (2 warps x 16 KB of static shared memory), 6 per SM.
#ifndef GF_EVAL_BSPLINE_F64_CUH_
#define GF_EVAL_BSPLINE_F64_CUH_

#include "gf_eval_lines.cuh"

namespace gfb {

constexpr int kBsF64Block = 64;
constexpr unsigned kBsF64WarpBytes = 32 * 512;   // 32 atoms x 2 records x 256 bytes

__device__ __forceinline__ void lds128_f64(unsigned addr, double* v) {
    asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v[0]), "=d"(v[1]) : "r"(addr) : "memory");
}

// whole 16-byte loads whatever part of them the arithmetic uses (see lds128_whole in gf_eval_bspline.cuh)
__device__ __forceinline__ void lds128_f64_whole(unsigned addr, double* v) {
    asm volatile("ld.volatile.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v[0]), "=d"(v[1]) : "r"(addr) : "memory");
}
// Tricubic Hermite (METHOD 2, HERMITE records filled by flat index) out of a lane's 512-byte region: the point at offsets
// (i-1, r-1, k-1) is element k & 1 of granule 8*i + 2*r + (k >> 1). 24 of the 32 granules are read.
struct TricubicSmemF64 {
    double g[4][4][4];     // [i][r][k]; the four (x,y) corner rows stay unset
    __device__ __forceinline__ double operator()(int i, int r, int k) const { return g[i][r][k]; }
};
__device__ __forceinline__ void tricubic_from_smem_f64(unsigned rbase, unsigned sw, bool xin, bool yin, bool zin, const TricubicWeights& w,
                                                       double& val, double& gx, double& gy, double& gz) {
    TricubicSmemF64 V;
#pragma unroll
    for (int r = 1; r <= 2; r++) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            lds128_f64_whole(rbase + (((8u * i + 2u * r) << 4) ^ sw), V.g[i][r]);
            lds128_f64_whole(rbase + (((8u * i + 2u * r + 1u) << 4) ^ sw), V.g[i][r] + 2);
        }
    }
#pragma unroll
    for (int r = 0; r <= 3; r += 3) {
#pragma unroll
        for (int i = 1; i <= 2; i++) {
            lds128_f64_whole(rbase + (((8u * i + 2u * r) << 4) ^ sw), V.g[i][r]);
            lds128_f64_whole(rbase + (((8u * i + 2u * r + 1u) << 4) ^ sw), V.g[i][r] + 2);
        }
    }
    tricubic_eval(V, xin, yin, zin, w, val, gx, gy, gz);
}

//   SINGLE  one replica and no energy slots (block-level energy reduction); the force mode is p.force_mode (launch-uniform)
//   METHOD  1 cubic B-spline on BSPLINE records, 2 tricubic Hermite on HERMITE records (same fetch, other arithmetic)
template <bool SINGLE, int METHOD>
__global__ void __launch_bounds__(kBsF64Block, 6) gf_eval_bspline_f64_kernel(const __grid_constant__ EvalParams p) {
    __shared__ __align__(128) unsigned char s_tiles[(kBsF64Block / 32) * kBsF64WarpBytes];

    const unsigned tid = threadIdx.x;
    const unsigned lane = tid & 31u;
    const unsigned t = blockIdx.x * kBsF64Block + tid;
    const unsigned total = (unsigned) p.total;
    const bool active = t < total;
    if (p.energies_clear)   // grid-stride: with energy slots the next accumulator can have more entries than the launch has threads
        for (unsigned c = t; c < (unsigned) (p.n_replicas * p.n_slots); c += gridDim.x * blockDim.x) p.energies_clear[c] = 0.0;

    // ---- who am I (as gf_eval_bspline_kernel) --------------------------------------------------------------------
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

    double x = 0.0, y = 0.0, z = 0.0;
    if (active) {
        const double* mine = p.pos + 3 * (size_t) gidx;
        x = load_stream(mine);
        y = load_stream(mine + 1);
        z = load_stream(mine + 2);
    }

    // ---- classification: exact FP64 division, the reference's expressions (:687-715); all grids share grid 0's geometry
    const GridView& G = p.grid[0];
    AtomCell c = classify<true>(G, x, y, z);
    const bool inside = c.inside && active;
    const unsigned brick0 = inside ? (unsigned) ((c.ix * G.nc[1] + c.iy) * G.nc[2] + c.iz) : 0xffffffffu;   // record (ix,iy,iz)
    const unsigned plane_recs = (unsigned) (G.nc[1] * G.nc[2]);   // records from one x-plane to the next

    const unsigned warp_base = (unsigned) __cvta_generic_to_shared(s_tiles) + (tid >> 5) * kBsF64WarpBytes;
    const unsigned rbase = warp_base + lane * 512u;
    const unsigned sw = (lane & 7u) << 4;

    // per-atom weights, used for every grid (:741-748)
    double bx[4], dbx[4], by[4], dby[4], bz[4], dbz[4];
    TricubicWeights tw;
    if constexpr (METHOD == 1) {
        bspline_basis(c.fx, bx, dbx);
        bspline_basis(c.fy, by, dby);
        bspline_basis(c.fz, bz, dbz);
    } else {
        tricubic_weights(c.fx, c.fy, c.fz, tw);
    }
    const bool xin = c.ix > 0 && c.ix < G.nc[0], yin = c.iy > 0 && c.iy < G.nc[1], zin = c.iz > 0 && c.iz < G.nc[2];   // :817, :849, :866

    double e_total = 0.0;
    double Fx = 0.0, Fy = 0.0, Fz = 0.0;
    double Sx = 0.0, Sy = 0.0, Sz = 0.0;   // sum over grids of scaling * index-space gradient
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
        // ---- fetch: round A brings the stencil of the atom of lane A; lane l copies granule l of its 512 bytes:
        //      granule = 16*(which record: a = ix | ix + 2) + 8*(which plane of it) + 2*row + half
        const unsigned mybrick = interp ? brick0 : 0xffffffffu;
        const char* lane_base = static_cast<const char*>(Gg.cells) + 16u * (lane & 15u) +
                                256ull * (unsigned long long) (2u * (lane >> 4)) * plane_recs;
        __syncwarp();   // the previous grid's records have been consumed
#pragma unroll 8
        for (int A = 0; A < 32; A++) {
            const unsigned bk = __shfl_sync(kFull, mybrick, A);
            if (bk != 0xffffffffu) cp_async16(warp_base + (unsigned) A * 512u + ((lane ^ ((unsigned) A & 7u)) << 4), lane_base + 256ull * bk);
        }
        cp_async_wait_all();
        __syncwarp();
        // ---- evaluate: bspline_interpolate<double>, operation for operation ---------------------------------------------
        double e_g = 0.0;
        if (METHOD == 2 && interp) {
            double val, gx, gy, gz;
            tricubic_from_smem_f64(rbase, sw, xin, yin, zin, tw, val, gx, gy, gz);
            tricubic_epilogue(Gg, s, val, gx, gy, gz, e_g, Fx, Fy, Fz);      // :879-893
        } else if (interp) {
            double val = 0.0, gx = 0.0, gy = 0.0, gz = 0.0;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                double pv = 0.0, pdy = 0.0, pdz = 0.0;
#pragma unroll
                for (int r = 0; r < 4; r++) {
                    double v[4];
                    lds128_f64(rbase + (((8u * i + 2u * r) << 4) ^ sw), v);
                    lds128_f64(rbase + (((8u * i + 2u * r + 1u) << 4) ^ sw), v + 2);
                    double rz = 0.0, drz = 0.0;
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        rz = fma(bz[k], v[k], rz);
                        drz = fma(dbz[k], v[k], drz);
                    }
                    pv = fma(by[r], rz, pv);
                    pdy = fma(dby[r], rz, pdy);
                    pdz = fma(by[r], drz, pdz);
                }
                val = fma(bx[i], pv, val);
                gx = fma(dbx[i], pv, gx);
                gy = fma(bx[i], pdy, gy);
                gz = fma(bx[i], pdz, gz);
            }
            if (Gg.inv_power > 0.0) {   // :778-787
                const double base = val;
                val = pow(base, Gg.inv_power);
                const double pf = Gg.inv_power * pow(base, Gg.inv_power - 1.0);
                gx *= pf;
                gy *= pf;
                gz *= pf;
            }
            e_g = s * val;   // :793
            Sx = fma(s, gx, Sx);   // :794; the division by the spacing (:790) is common to all grids (one geometry) and is
            Sy = fma(s, gy, Sy);   // done once per atom after the loop instead of once per grid (an FP64 division is ~30
            Sz = fma(s, gz, Sz);   // instructions)
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

    if (inside) {
        Fx -= Sx / G.spacing[0];
        Fy -= Sy / G.spacing[1];
        Fz -= Sz / G.spacing[2];
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
            __shared__ double warp_sum[kBsF64Block / 32];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) e_total += __shfl_xor_sync(kFull, e_total, o);
            if (lane == 0) warp_sum[tid >> 5] = e_total;
            __syncthreads();
            if (tid == 0) {
                double b = 0.0;
#pragma unroll
                for (int w = 0; w < kBsF64Block / 32; w++) b += warp_sum[w];
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
