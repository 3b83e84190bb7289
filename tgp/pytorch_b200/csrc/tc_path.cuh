// FP32 / tensor-core mode of the batch contractions (TgpModel.dtype == TGP_F32).
//
// Per-step work (K_zz, Cholesky, L^-1, C, KL, the backward chain) and the row epilogue stay in FP64; only the three
// O(rows * M^2) contractions run on tcgen05 as 3xTF32 products with FP32 accumulation in TMEM (gemm_tc.cuh).
// Operands are staged as (value, value - tf32_trunc(value)) plane pairs, K-major:
//   K      (rows x M)   generated per row chunk, kept for all rows for the backward        forward  A-operand
//   W      (2M x M)   = [L^-1 ; C]                                                        forward  B-operand
//   ABbar  (rows x 2M) = [g_mu m - 2 g_v A | 2 g_v B]                                     backward-data A-operand
//   Wt     (M x 2M)   = [L^-T | C^T]                                                      backward-data B-operand
//   ABbar^T (2M x rows), K^T (M x rows)                                                   backward-weight operands
#pragma once
#include "common.cuh"
#include "gemm_tc.cuh"

namespace tgp {
namespace tc {

// hi = x rounded to nearest TF32 (so that the tensor core's truncation of the plane is exact), lo = x - hi (exact in
// FP32, symmetric around 0: the residual's own truncation to TF32 then leaves an unbiased 2^-23 relative error)
__device__ __forceinline__ float tf32_hi(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
__device__ __forceinline__ void put_planes(float* __restrict__ hi, float* __restrict__ lo, long idx, float x) {
    const float h = tf32_hi(x);
    hi[idx] = h;
    lo[idx] = x - h;
}

inline long pad4(long x) { return (x + 3) / 4 * 4; }

// K tile (distance in FP64, as k_rbf_tile; exponential in FP32: Cov<KIND>::kf, common.cuh), written as FP32 planes: row-major (rows x ldk) and
// transposed (M x ldt).  32 x 64 tile per CTA staged through shared memory so that both writes are coalesced.
constexpr int RP_TR = 32, RP_TC = 64, RP_THREADS = 256;
template <int KIND>
// The marginal mean is accumulated here as well (u = L^-T m, FP64, one per step): mu[n] += sum_j K[n,j] u[j] in FP64 —
// the reference's own evaluation order mu = K_xz (L^-T m) (sparse_MF_SP.py:354-355).  Taking mu from the FP32 rows a = L^-1 k
// instead lets the conditioning of L^-1 amplify the FP32 rounding of a (measured at cfg4: max |dmu| 3.3e-4 against 2.3e-5, ELBO
// 3.6e-5 against 2.4e-6 from FP64; scripts/tf32_error_terms.py).
__global__ void __launch_bounds__(RP_THREADS) k_rbf_planes(const double* __restrict__ X, const double* __restrict__ Zs,
                                                           const double* __restrict__ ls, const double* __restrict__ os,
                                                           int R, int M, int D, float* __restrict__ Khi, float* __restrict__ Klo,
                                                           long ldk, float* __restrict__ KThi, float* __restrict__ KTlo, long ldt,
                                                           const double* __restrict__ u, double* __restrict__ mu) {
    extern __shared__ double sm_rp[];
    const int DP = D + 1;
    double* xs = sm_rp;
    double* zs = sm_rp + RP_TR * DP;
    float* tile = reinterpret_cast<float*>(zs + RP_TC * DP);            // [RP_TR][RP_TC + 1]
    const int r0 = blockIdx.y * RP_TR, c0 = blockIdx.x * RP_TC, tid = threadIdx.x;
    for (int i = tid; i < RP_TR * D; i += RP_THREADS) {
        const int r = i / D, d = i % D, n = r0 + r;
        xs[r * DP + d] = n < R ? X[(long)n * D + d] / ls[d] : 0.0;
    }
    for (int i = tid; i < RP_TC * D; i += RP_THREADS) {
        const int c = i / D, d = i % D, j = c0 + c;
        zs[c * DP + d] = j < M ? Zs[(long)j * D + d] : 0.0;
    }
    __syncthreads();
    const double s = os[0];
    const int c = tid % RP_TC, j = c0 + c;
    const double uj = j < M ? u[j] : 0.0;
    for (int r = tid / RP_TC; r < RP_TR; r += RP_THREADS / RP_TC) {
        const int n = r0 + r;
        float val = 0.f;
        if (n < R && j < M) {
            double acc = 0.0;
            for (int d = 0; d < D; ++d) { const double df = xs[r * DP + d] - zs[c * DP + d]; acc = fma(df, df, acc); }
            // argument in FP64 (exact to ~1e-16), exponential in FP32: exp(a) = expf(a_hi) * (1 + a_lo)
            val = Cov<KIND>::kf(acc, (float)s);
        }
        tile[r * (RP_TC + 1) + c] = val;
        if (n < R && j < M) put_planes(Khi, Klo, (long)n * ldk + j, val);
        // the 32 lanes of a warp hold 32 columns of the SAME row (RP_TC = 64)
        const double part = warp_sum((double)val * uj);
        if ((tid & 31) == 0 && n < R) atomicAdd(mu + n, part);
    }
    __syncthreads();
    const int rr = tid % RP_TR;
    for (int cc = tid / RP_TR; cc < RP_TC; cc += RP_THREADS / RP_TR) {
        const int n = r0 + rr, jj = c0 + cc;
        if (n < R && jj < M) {
            const float val = tile[rr * (RP_TC + 1) + cc];
            put_planes(KThi, KTlo, (long)jj * ldt + n, val);
        }
    }
}

template <int KIND>
inline int launch_rbf_planes(const double* X, const double* Zs, const double* ls, const double* os, int R, int M, int D,
                             float* Khi, float* Klo, long ldk, float* KThi, float* KTlo, long ldt, cudaStream_t st,
                             const double* u, double* mu) {
    const size_t smem = (size_t)(RP_TR + RP_TC) * (D + 1) * sizeof(double) + (size_t)RP_TR * (RP_TC + 1) * sizeof(float);
    if (smem > 200 * 1024) return set_error(-2, "input dimension too large for the plane-generating RBF kernel");
    // above 48 KiB (D >= 53) the kernel needs the opt-in to large dynamic shared memory, set once per device to the bound above
    if (smem > 48 * 1024) {
        static PerDeviceOnce once;
        if (once.first()) cudaFuncSetAttribute(k_rbf_planes<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    }
    dim3 grid((unsigned)cdiv(M, RP_TC), (unsigned)cdiv(R, RP_TR));
    k_rbf_planes<KIND><<<grid, RP_THREADS, smem, st>>>(X, Zs, ls, os, R, M, D, Khi, Klo, ldk, KThi, KTlo, ldt, u, mu);
    return check_launch("k_rbf_planes");
}

// W = [Linv ; C] (2M x ldw) and Wt = [Linv^T | C^T] (M x ldwt) as FP32 plane pairs from the FP64 step matrices (ld = Mp)
__global__ void k_make_w_planes(const double* __restrict__ Linv, const double* __restrict__ Cm, long ld, int M,
                                float* __restrict__ Whi, float* __restrict__ Wlo, long ldw, float* __restrict__ Wthi,
                                float* __restrict__ Wtlo, long ldwt) {
    __shared__ float ta[32][33], tb[32][33];
    const int j0 = blockIdx.y * 32, i0 = blockIdx.x * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
    for (int r = ty; r < 32; r += 8) {
        const int j = j0 + r, i = i0 + tx;
        float a = 0.f, b = 0.f;
        if (j < M && i < M) { a = (float)Linv[(long)j * ld + i]; b = (float)Cm[(long)j * ld + i]; }
        ta[r][tx] = a; tb[r][tx] = b;
        if (j < M && i < M) {
            put_planes(Whi, Wlo, (long)j * ldw + i, a);
            put_planes(Whi, Wlo, (long)(M + j) * ldw + i, b);
        }
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int i = i0 + r, j = j0 + tx;
        if (i < M && j < M) {
            const float a = ta[tx][r], b = tb[tx][r];
            put_planes(Wthi, Wtlo, (long)i * ldwt + j, a);
            put_planes(Wthi, Wtlo, (long)i * ldwt + M + j, b);
        }
    }
}

// v from the FP32 [A | B] rows (sums accumulated in FP64); mu is accumulated by k_rbf_planes
__global__ void __launch_bounds__(128) k_row_stats_f32(const float* __restrict__ AB, long ldab, const double* __restrict__ os, int R,
                                                       int M, double* __restrict__ v) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    for (long n = (long)blockIdx.x * wpb + wid; n < R; n += (long)gridDim.x * wpb) {
        const float* a = AB + n * ldab;
        const float* b = a + M;
        double sa = 0.0, sb = 0.0;
        for (int j = lane; j < M; j += 32) {
            const double aj = a[j], bj = b[j];
            sa = fma(aj, aj, sa);
            sb = fma(bj, bj, sb);
        }
        sa = warp_sum(sa); sb = warp_sum(sb);
        if (lane == 0) v[n] = os[0] - sa + sb;
    }
}

// u = L^-T m (FP64): u[j] = sum_{i >= j} Linv[i][j] m[i].  32 columns x 8 row phases per CTA.
__global__ void __launch_bounds__(256) k_linvT_m(const double* __restrict__ Linv, long ld, const double* __restrict__ m, int M,
                                                 double* __restrict__ u) {
    __shared__ double part[8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5, j = blockIdx.x * 32 + tx;
    double s = 0.0;
    if (j < M) for (int i = (j / 8) * 8 + ty; i < M; i += 8) if (i >= j) s = fma(Linv[(long)i * ld + j], m[i], s);
    part[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && j < M) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += part[k][tx];
        u[j] = t;
    }
}

// [A | B] (FP32) + upstream row gradients -> ABbar planes (rows x 2M) and their transposes (2M x rows);
// accumulates dm[j] += sum_n g_mu A, dos += sum_n g_v (FP64 atomics).  32 rows x 64 columns per CTA.
__global__ void __launch_bounds__(256) k_make_abbar_planes(const float* __restrict__ AB, long ldab, const double* __restrict__ g_mu,
                                                           const double* __restrict__ g_v, const double* __restrict__ m,
                                                           int R, int M, float* __restrict__ Phi, float* __restrict__ Plo, long ldp,
                                                           float* __restrict__ PThi, float* __restrict__ PTlo, long ldpt,
                                                           double* __restrict__ dm, double* __restrict__ dos) {
    __shared__ float ta[32][65], tb[32][65];
    __shared__ double cs[4][64];
    const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 64, tid = threadIdx.x, c = tid & 63, ry = tid >> 6;   // 64 x 4
    const int j = c0 + c;
    const double mj = j < M ? m[j] : 0.0;
    double acc = 0.0, accv = 0.0;
    for (int r = ry; r < 32; r += 4) {
        const int n = r0 + r;
        float abar = 0.f, bbar = 0.f;
        if (n < R) {
            const double gm = g_mu[n], gv = g_v[n];
            accv += gv;
            if (j < M) {
                const double a = AB[(long)n * ldab + j], b = AB[(long)n * ldab + M + j];
                acc = fma(gm, a, acc);
                abar = (float)(gm * mj - 2.0 * gv * a);
                bbar = (float)(2.0 * gv * b);
                put_planes(Phi, Plo, (long)n * ldp + j, abar);
                put_planes(Phi, Plo, (long)n * ldp + M + j, bbar);
            }
        }
        ta[r][c] = abar; tb[r][c] = bbar;
    }
    cs[ry][c] = acc;
    __syncthreads();
    if (ry == 0 && j < M) atomicAdd(dm + j, cs[0][c] + cs[1][c] + cs[2][c] + cs[3][c]);
    if (blockIdx.x == 0 && c == 0) atomicAdd(dos, accv);      // one thread per row-lane: its rows' g_v
    const int rr = tid & 31;
    for (int cc = tid >> 5; cc < 64; cc += 8) {
        const int n = r0 + rr, jj = c0 + cc;
        if (n < R && jj < M) {
            const float a = ta[rr][cc], b = tb[rr][cc];
            put_planes(PThi, PTlo, (long)jj * ldpt + n, a);
            put_planes(PThi, PTlo, (long)(M + jj) * ldpt + n, b);
        }
    }
}

}  // namespace tc
}  // namespace tgp
