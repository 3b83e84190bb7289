// Fused forward of the tensor-core mode: K_xz tiles are generated on the fly INSIDE the contraction kernel.
//
//   per 128-row tile:   k(x_n, z_j)  --CUDA cores-->  swizzled smem A stages (TF32 hi/lo planes)
//                       [L^-1 ; C] planes  --TMA-->   swizzled smem B stages
//                       tcgen05.mma (3xTF32)  -->  TMEM  --tcgen05.ld-->  FP32 register accumulation
//                       epilogue: [A | B] row (saved for the backward)  +  mu = a.m, ||a||^2, ||b||^2  ->  mu, v
//
// K_xz never exists in global memory (not even as a staging tile) and the row statistics never re-read [A | B].
// 16 warps, register budget redistributed with setmaxnreg:
//   warpgroup 0: warp 0 = TMA producer of the B planes, warp 1 = TMEM allocation + MMA issue   (64 regs)
//   warpgroups 1-2: 8 epilogue warps (TMEM lane quarter = warp % 4, column half = warpgroup - 1)  (176 regs)
//   warpgroup 3: 4 K-generator warps, thread <-> tile row, FP64 argument + FP32 exponential      (96 regs)
// For every 256-column chunk of the stacked output the K tile is regenerated (8x at M = 1024): ~0.7 of the MMA time on
// the FP64/FP32 pipes, concurrent with the tensor pipe.
#pragma once
#include "gemm_tc.cuh"
#include "tc_path.cuh"

namespace tgp {
namespace tc {

constexpr int FUSED_THREADS = 512;
constexpr int FUSED_MAX_D = 16;
constexpr int ZBUF_DOUBLES = BK * (FUSED_MAX_D + 1);                 // one k-block of pre-scaled inducing points + their norms
constexpr int FUSED_SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + STAGES * ZBUF_DOUBLES * 8 + BM * 3 * 8 + 256;

struct FusedFwdParams {
    const double *X, *Zs, *ls, *os, *mvec;
    const double* u;                 // L^-T m (FP64): mu = K_xz u is accumulated by the K generator (NULL: mu from the FP32 rows a)
    int R, M, D;
    float* AB; long ldab;            // (R x ldab) FP32, [A | B]
    double *mu, *v;
};

__device__ __forceinline__ void named_bar_sync(int id, int count) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}

template <int MAXD>
__global__ void __launch_bounds__(FUSED_THREADS, 1)
fwd_fused_kernel(const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapBlo, const FusedFwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    double* zbuf = reinterpret_cast<double*>(smem + STAGES * STAGE_BYTES);              // [STAGES][BK][D]
    double* xch = zbuf + STAGES * ZBUF_DOUBLES;                                         // [BM][3] half-1 -> half-0 exchange
    uint64_t* full_a = reinterpret_cast<uint64_t*>(xch + BM * 3);
    uint64_t* full_b = full_a + STAGES;
    uint64_t* empty = full_b + STAGES;
    uint64_t* tfull = empty + STAGES;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wg = warp >> 2;
    const int M = p.M, D = p.D, N2 = 2 * p.M;
    const int tiles_m = (p.R + BM - 1) / BM, n_chunks = (N2 + BN - 1) / BN;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full_a[s], 4); mbar_init(&full_b[s], 1); mbar_init(&empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // k-range of output chunk nc: rows n < M of [L^-1; C] are lower triangular (nonzero k <= n)
    auto k_end = [&](int n0) { return n0 < M ? min(M, n0 + BN) : M; };

    if (wg == 0) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
        if (warp == 0 && lane == 0) {
            // ===== TMA producer: B planes =====
            int stage = 0; uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < tiles_m; tile += gridDim.x)
                for (int nc = 0; nc < n_chunks; ++nc) {
                    const int n0 = nc * BN, ke = k_end(n0);
                    for (int k = 0; k < ke; k += BK) {
                        mbar_wait(&empty[stage], phase ^ 1);
                        uint8_t* st = smem + stage * STAGE_BYTES;
                        mbar_expect_tx(&full_b[stage], 2 * B_BYTES);
                        tma_load_2d(st + 2 * A_BYTES, &mapB, &full_b[stage], k, n0);
                        tma_load_2d(st + 2 * A_BYTES + B_BYTES, &mapBlo, &full_b[stage], k, n0);
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    }
                }
        } else if (warp == 1 && lane == 0) {
            // ===== MMA issuer =====
            const uint32_t idesc = make_idesc();
            int stage = 0; uint32_t phase = 0;
            int buf = 0; uint32_t bphase = 0;
            for (int tile = blockIdx.x; tile < tiles_m; tile += gridDim.x)
                for (int nc = 0; nc < n_chunks; ++nc) {
                    const int ke = k_end(nc * BN);
                    int kbi = 0;
                    uint32_t tmem_d = 0, accum = 0;
                    for (int k = 0; k < ke; k += BK) {
                        if (kbi == 0) {
                            mbar_wait(&tempty[buf], bphase ^ 1);
                            tc_fence_after();
                            tmem_d = tmem_base + (uint32_t)buf * BN;
                            accum = 0;
                        }
                        mbar_wait(&full_a[stage], phase);
                        mbar_wait(&full_b[stage], phase);
                        tc_fence_after();
                        uint8_t* st = smem + stage * STAGE_BYTES;
                        const uint64_t dA = make_desc(st), dAl = make_desc(st + A_BYTES);
                        const uint64_t dB = make_desc(st + 2 * A_BYTES), dBl = make_desc(st + 2 * A_BYTES + B_BYTES);
#pragma unroll
                        for (int kk = 0; kk < BK / UMMA_K; ++kk) {
                            const uint64_t adv = (uint64_t)((kk * UMMA_K * 4) >> 4);
                            umma_tf32(tmem_d, dA + adv, dB + adv, idesc, accum);
                            accum = 1;
                            umma_tf32(tmem_d, dAl + adv, dB + adv, idesc, 1);
                            umma_tf32(tmem_d, dA + adv, dBl + adv, idesc, 1);
                        }
                        umma_commit(&empty[stage]);
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                        if (++kbi == KB_PER_CHUNK || k + BK >= ke) {
                            umma_commit(&tfull[buf]);
                            if (++buf == 2) { buf = 0; bphase ^= 1; }
                            kbi = 0;
                        }
                    }
                }
        }
    } else if (wg == 3) {
        // ===== K generator: thread t <-> row m0 + t of the tile =====
        asm volatile("setmaxnreg.dec.sync.aligned.u32 96;");
        const int t = threadIdx.x - 384;
        const float sf = (float)p.os[0];
        int stage = 0; uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < tiles_m; tile += gridDim.x) {
            const long row = (long)tile * BM + t;
            // squared distance by expansion in FP64: |x|^2 + |z|^2 - 2 x.z (absolute error ~1e-15, the formula gpytorch uses);
            // eight inducing points at a time give eight independent FMA chains per thread
            double x2[MAXD], xn = 0.0;
#pragma unroll
            for (int d = 0; d < MAXD; ++d) {
                const double xd = (d < D && row < p.R) ? p.X[row * D + d] / p.ls[d] : 0.0;
                xn = fma(xd, xd, xn);
                x2[d] = -2.0 * xd;
            }
            double mu_acc = 0.0;                      // mu = sum_j K[row, j] u[j] in FP64, taken from the last chunk (it spans all of K)
            for (int nc = 0; nc < n_chunks; ++nc) {
                const int ke = k_end(nc * BN);
                const bool take_mu = p.u != nullptr && nc == n_chunks - 1;
                for (int k = 0; k < ke; k += BK) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    double* zb = zbuf + stage * ZBUF_DOUBLES;          // [BK][MAXD] then [BK] norms
                    double* zn = zb + BK * MAXD;
                    for (int i = t; i < BK * MAXD; i += 128) {
                        const int c = i / MAXD, d = i - c * MAXD;
                        zb[i] = (k + c < M && d < D) ? p.Zs[(long)(k + c) * D + d] : 0.0;
                    }
                    named_bar_sync(2, 128);
                    if (t < BK) {
                        double nz = 0.0;
#pragma unroll
                        for (int d = 0; d < MAXD; ++d) nz = fma(zb[t * MAXD + d], zb[t * MAXD + d], nz);
                        zn[t] = nz;
                    }
                    named_bar_sync(2, 128);
                    uint8_t* st = smem + stage * STAGE_BYTES;
                    uint8_t* rowp_hi = st + t * 128;
                    uint8_t* rowp_lo = st + A_BYTES + t * 128;
#pragma unroll 1
                    for (int c0 = 0; c0 < BK; c0 += 8) {             // two 16-byte chunks of the 128-byte swizzle row
                        double acc[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) acc[e] = xn + zn[c0 + e];
#pragma unroll
                        for (int d = 0; d < MAXD; ++d)
#pragma unroll
                            for (int e = 0; e < 8; ++e) acc[e] = fma(x2[d], zb[(c0 + e) * MAXD + d], acc[e]);
                        float hi[8], lo[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            float val = 0.f;
                            if (row < p.R && k + c0 + e < M) {
                                val = Cov<TGP_KERNEL_RBF>::kf(fmax(acc[e], 0.0), sf);
                                if (take_mu) mu_acc = fma((double)val, __ldg(p.u + k + c0 + e), mu_acc);
                            }
                            hi[e] = tf32_hi(val);
                            lo[e] = val - hi[e];
                        }
#pragma unroll
                        for (int h2 = 0; h2 < 2; ++h2) {
                            const int phys = (((c0 >> 2) + h2) ^ (t & 7)) << 4;   // Swizzle<3,4,3>: chunk index XOR (row mod 8)
                            *reinterpret_cast<float4*>(rowp_hi + phys) = make_float4(hi[4 * h2], hi[4 * h2 + 1], hi[4 * h2 + 2], hi[4 * h2 + 3]);
                            *reinterpret_cast<float4*>(rowp_lo + phys) = make_float4(lo[4 * h2], lo[4 * h2 + 1], lo[4 * h2 + 2], lo[4 * h2 + 3]);
                        }
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> tensor-core reads
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&full_a[stage]);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
            if (p.u != nullptr && row < p.R) p.mu[row] = mu_acc;
        }
    } else {
        // ===== epilogue warps (warpgroups 1, 2) =====
        asm volatile("setmaxnreg.inc.sync.aligned.u32 176;");
        const int q = warp & 3, half = wg - 1;
        int buf = 0; uint32_t bphase = 0;
        for (int tile = blockIdx.x; tile < tiles_m; tile += gridDim.x) {
            const long row = (long)tile * BM + q * 32 + lane;
            double smu = 0.0, ssa = 0.0, ssb = 0.0;
            for (int nc = 0; nc < n_chunks; ++nc) {
                const int n0 = nc * BN, ke = k_end(n0);
                const int nchunks = ((ke + BK - 1) / BK + KB_PER_CHUNK - 1) / KB_PER_CHUNK;
                float acc[128];
#pragma unroll
                for (int i = 0; i < 128; ++i) acc[i] = 0.f;
                for (int chn = 0; chn < nchunks; ++chn) {
                    mbar_wait(&tfull[buf], bphase);
                    tc_fence_after();
                    const uint32_t taddr = tmem_base + (uint32_t)buf * BN + (uint32_t)(half * 128) + ((uint32_t)(q * 32) << 16);
#pragma unroll
                    for (int c = 0; c < 128; c += 32) {
                        uint32_t r[32];
                        asm volatile(
                            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                              "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                              "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                              "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                            : "r"(taddr + (uint32_t)c));
                        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                        for (int i = 0; i < 32; ++i) acc[c + i] += __uint_as_float(r[i]);
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&tempty[buf]);
                    if (++buf == 2) { buf = 0; bphase ^= 1; }
                }
                // chunk finished: save [A | B] and fold it into the row statistics
                if (row < p.R) {
                    const int nbase = n0 + half * 128;
                    float* dst = p.AB + row * p.ldab + nbase;
                    if (nbase + 128 <= N2 && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
#pragma unroll
                        for (int i = 0; i < 128; i += 4)
                            *reinterpret_cast<float4*>(dst + i) = make_float4(acc[i], acc[i + 1], acc[i + 2], acc[i + 3]);
                    } else {
#pragma unroll
                        for (int i = 0; i < 128; ++i) if (nbase + i < N2) dst[i] = acc[i];
                    }
#pragma unroll
                    for (int i = 0; i < 128; ++i) {
                        const int col = nbase + i;
                        const double a = (double)acc[i];
                        if (col < M) { smu = fma(a, __ldg(p.mvec + col), smu); ssa = fma(a, a, ssa); }
                        else if (col < N2) ssb = fma(a, a, ssb);
                    }
                }
            }
            // combine the two column halves of each row: half 1 -> shared -> half 0 writes mu, v
            if (half == 1) { xch[(q * 32 + lane) * 3 + 0] = smu; xch[(q * 32 + lane) * 3 + 1] = ssa; xch[(q * 32 + lane) * 3 + 2] = ssb; }
            named_bar_sync(1, 256);
            if (half == 0 && row < p.R) {
                const int rr = (q * 32 + lane) * 3;
                if (p.u == nullptr) p.mu[row] = smu + xch[rr];
                p.v[row] = p.os[0] - (ssa + xch[rr + 1]) + (ssb + xch[rr + 2]);
            }
            named_bar_sync(1, 256);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512));
    }
}

inline int fwd_fused(const Operand& W, const FusedFwdParams& p, cudaStream_t st) {
    if (p.R <= 0) return 0;
    if (p.D > FUSED_MAX_D) return set_error(-2, "fused forward supports D <= 16");
    CUtensorMap mB, mBl;
    TGP_TRY(make_map(&mB, W.hi, W.rows, W.cols, W.ld, BN));
    TGP_TRY(make_map(&mBl, W.lo, W.rows, W.cols, W.ld, BN));
    static PerDeviceOnce attr_once;
    if (attr_once.first()) {
        cudaFuncSetAttribute(fwd_fused_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, FUSED_SMEM_BYTES);
        cudaFuncSetAttribute(fwd_fused_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, FUSED_SMEM_BYTES);
        cudaFuncSetAttribute(fwd_fused_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, FUSED_SMEM_BYTES);
    }
    const int tiles = (p.R + BM - 1) / BM;
    const int grid = tiles < 148 ? tiles : 148;
    const bool timed = g_gemm_timer.enabled;
    if (timed) g_gemm_timer.begin(2, st);
    if (p.D <= 4) fwd_fused_kernel<4><<<grid, FUSED_THREADS, FUSED_SMEM_BYTES, st>>>(mB, mBl, p);
    else if (p.D <= 8) fwd_fused_kernel<8><<<grid, FUSED_THREADS, FUSED_SMEM_BYTES, st>>>(mB, mBl, p);
    else fwd_fused_kernel<16><<<grid, FUSED_THREADS, FUSED_SMEM_BYTES, st>>>(mB, mBl, p);
    if (timed) g_gemm_timer.end(st);
    return check_launch("fwd_fused_kernel");
}

}  // namespace tc
}  // namespace tgp
