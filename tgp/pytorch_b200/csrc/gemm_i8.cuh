// FP64-accurate contraction on the tcgen05 INTEGER tensor path (kind::i8, u8 x u8 -> 32-bit in TMEM): the batch contractions
// of compute mode TGP_F64_I8.
//
// tcgen05 has no f64 kind, and a floating-point split (3xTF32, gemm_tc.cuh) is limited by the FP32 accumulator.  Integer
// MMAs accumulate EXACTLY, so the product can be rebuilt exactly from residues (Chinese remainder theorem; "Ozaki scheme
// II" in the literature):
//   1. integerise  A'[i,:] = rint(A[i,:] 2^(b - eA_i)),  2^eA_i > max_j |A_ij|   (|A'| < 2^b, b <= 53; likewise B per row)
//   2. residues    A_t = A' mod p_t  in [0, p_t), u8,  for T pairwise coprime moduli p_t <= 256           [k_to_residues]
//   3. T independent u8 GEMMs with exact 32-bit accumulation, reduced mod p_t in the epilogue: R_t = A_t B_t^T mod p_t
//      (u8 again)                                                                                        [gemm_i8_mod_kernel]
//   4. CRT         C' = sum_t R_t w_t - m P   in 40-bit words whose partial sums are exact in FP64,  m = rint(sum_t R_t w_t/P)
//   5. scale       C = C' 2^(eA_i + eB_j - 2b)                                                            [k_crt_combine]
// The integer product is exact; the only error is the b-bit truncation of the operands below their row maximum
// (b = 53 with T = 15 moduli for reductions up to 1024, T = 16 up to 2^17) — at or below FP64 GEMM rounding.
// oracle/crt_gemm.py restates steps 1-5 in numpy / exact Python integers (tests/test_crt_oracle.py).
//
// gemm_i8_mod_kernel: persistent, warp-specialised, one CTA per SM (TMA producer warp, single-thread MMA issuer, eight
// epilogue warps); tile 128 x 256 x 128 (one 128-byte swizzle row of int8 per k-block), 4-stage mbarrier ring (192 KiB),
// two 256-column TMEM accumulators so that the mod-p epilogue of one (tile, modulus) overlaps the MMAs of the next.
// N = 256 per MMA is what reaches the integer peak (scripts/microbench/mma_rate.cu: 4556 Tops/s at N = 256, 1991 at N = 64).
#pragma once
#include <cuda.h>
#include "common.cuh"
#include "gemm_f64.cuh"      // GemmTimer
#include "gemm_tc.cuh"       // PTX wrappers (mbarrier, TMA, tcgen05 fences / commit), encode_fn

namespace tgp {
namespace i8 {

constexpr int MAX_T = 16;
constexpr int WORD_BITS = 40, N_WORDS = 4;            // CRT reconstruction: 40-bit words (five weight bytes each)
constexpr int BM = 128, BN = 256, BK = 128;          // BK in bytes == int8 elements
constexpr int STAGES = 4;
constexpr int A_BYTES = BM * BK, B_BYTES = BN * BK, STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 256;
constexpr int EPI_WARPS = 8;                          // 4 TMEM lane quadrants x (EPI_WARPS / 4) column parts (16 warps measured no faster)
constexpr int EPI_COLS = BN / (EPI_WARPS / 4);        // accumulator columns per epilogue thread
constexpr int THREADS = 64 + 32 * EPI_WARPS;
constexpr int UMMA_K = 32;                            // kind::i8: 32 bytes of K per MMA

static const int MODULI[MAX_T] = {256, 255, 253, 251, 247, 241, 239, 233, 229, 227, 223, 217, 211, 199, 197, 193};

struct CrtTable {                 // passed by value to the kernels (< 1 KiB)
    int T;
    int p[MAX_T];
    // CRT weights w_t = (P/p_t) * ((P/p_t)^-1 mod p_t) < P < 256^16 by BYTES, packed for dp4a: byte j of wb[g][k] is byte k of
    // w_{4g+j}, so that sum_t r_t byte_k(w_t) = sum_g dp4a(residues 4g..4g+3 of an element, wb[g][k])
    uint32_t wb[MAX_T / 4][16];
    double Pw[N_WORDS];           // 40-bit words of P
    double log2P;
    double invP;                  // 1 / P
    // residues of a 56-bit magnitude by byte limbs: u = sum_k a_k 256^k  =>  u mod p = (sum_k a_k (256^k mod p)) mod p;
    // clo / chi pack (256^k mod p) for k = 0..3 / 4..7 (dp4a operands), magic = ceil(2^32 / p) (exact floor division of
    // the < 2^19 limb sum by a multiply-high)
    uint32_t clo[MAX_T], chi[MAX_T], magic[MAX_T];
    uint32_t init[MAX_T];         // (p - 2^54 mod p) mod p: signed integers are shifted by 2^54 before the limbs are taken
};

inline const CrtTable& crt_table(int T) {
    static CrtTable tabs[MAX_T + 1];
    static bool have[MAX_T + 1] = {};
    if (T < 1) T = 1;
    if (T > MAX_T) T = MAX_T;
    if (!have[T]) {
        typedef unsigned __int128 u128;
        CrtTable& c = tabs[T];
        c.T = T;
        u128 P = 1;
        for (int t = 0; t < T; ++t) P *= (u128)MODULI[t];
        const u128 mask = (((u128)1) << WORD_BITS) - 1;
        auto to_ld = [](u128 x) { return (long double)(unsigned long long)(x >> 64) * 18446744073709551616.0L + (long double)(unsigned long long)x; };
        for (int t = 0; t < T; ++t) {
            const int p = MODULI[t];
            c.p[t] = p;
            const u128 q = P / (u128)p;
            const int qm = (int)(q % (u128)p);
            int inv = 1;
            while ((qm * inv) % p != 1) ++inv;
            const u128 w = q * (u128)inv;
            for (int k = 0; k < 16; ++k)
                c.wb[t / 4][k] |= (uint32_t)((unsigned)((w >> (8 * k)) & 0xff)) << (8 * (t % 4));
            uint32_t pw = 1 % (uint32_t)p, lo = 0, hi = 0;
            for (int k = 0; k < 8; ++k) {
                if (k < 4) lo |= pw << (8 * k); else hi |= pw << (8 * (k - 4));
                pw = (pw * 256u) % (uint32_t)p;
            }
            c.clo[t] = lo; c.chi[t] = hi;
            c.magic[t] = (uint32_t)((4294967296ull + (unsigned long long)p - 1ull) / (unsigned long long)p);
            c.init[t] = (uint32_t)(((unsigned long long)p - (18014398509481984ull % (unsigned long long)p)) % (unsigned long long)p);
        }
        for (int k = 0; k < N_WORDS; ++k) c.Pw[k] = (double)(unsigned long long)((P >> (WORD_BITS * k)) & mask);
        c.log2P = (double)log2l(to_ld(P));
        c.invP = (double)(1.0L / to_ld(P));
        have[T] = true;
    }
    return tabs[T];
}

// largest b (bits per operand) with 2 * k_red * 2^(2b) < P (and a 2^-30 margin for the rounding of m)
inline int crt_bits(int T, long k_red) {
    const double room = crt_table(T).log2P - 1.0 - log2((double)(k_red > 1 ? k_red : 1)) - 1e-6;
    int b = (int)floor(room / 2.0);
    return b > 53 ? 53 : (b < 1 ? 1 : b);
}

// x * 2^n, exact: one multiply by a constructed power of two when n is an ordinary exponent
__device__ __forceinline__ double mul_pow2(double x, int n) {
    if (n > -1000 && n < 1000) return x * __hiloint2double((1023 + n) << 20, 0);
    return scalbn(x, n);
}

// ---- step 1 + 2: FP64 -> residue planes -----------------------------------------------------------------------------
// exponent e with 2^e > |x| (e = 0 for x = 0)
__device__ __forceinline__ int exp_above(double x) {
    int e;
    frexp(x, &e);
    return x == 0.0 ? 0 : e;
}

// row_exp[r] = max over the row, col_exp[c] = max over the column (atomicMax; both optional, pre-set to a very small value)
__global__ void __launch_bounds__(256) k_exponents(const double* __restrict__ src, long ld, long rows, int cols,
                                                   int* __restrict__ row_exp, int* __restrict__ col_exp) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c0 = blockIdx.x * 256;
    const long r0 = (long)blockIdx.y * 64;
    int cmax[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) cmax[i] = -100000;
    for (long r = r0 + warp; r < min(r0 + 64, rows); r += 8) {
        int rmax = -100000;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int c = c0 + lane + 32 * i;
            if (c < cols) {
                const int e = exp_above(src[r * ld + c]);
                rmax = max(rmax, e);
                cmax[i] = max(cmax[i], e);
            }
        }
        if (row_exp) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) rmax = max(rmax, __shfl_xor_sync(0xffffffffu, rmax, o));
            if (lane == 0) atomicMax(row_exp + r, rmax);
        }
    }
    if (col_exp) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int c = c0 + lane + 32 * i;
            if (c < cols && cmax[i] > -100000) atomicMax(col_exp + c, cmax[i]);
        }
    }
}

__global__ void k_fill_int(int* __restrict__ p, long n, int v) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// residue in [0, p) of the signed integer x (|x| <= 2^53) handed over as u = x + 2^54 (lo / hi words): two dp4a over the byte
// limbs of u (u = sum_k a_k 256^k  =>  u mod p = sum_k a_k (256^k mod p) mod p) started from init = -2^54 mod p, then an exact
// multiply-high division of the < 2^19 limb sum.  Residues are UNSIGNED bytes: the tensor core takes u8 operands
// (K * 255^2 < 2^31 for reductions up to 33025), and no centring is needed anywhere.
__device__ __forceinline__ uint32_t residue_of(uint32_t lo, uint32_t hi, uint32_t clo, uint32_t chi, uint32_t init, uint32_t magic, uint32_t p) {
    const uint32_t s = __dp4a(lo, clo, __dp4a(hi, chi, init));
    return s - __umulhi(s, magic) * p;
}
// the low bytes of four words as one word
__device__ __forceinline__ uint32_t pack4(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    return __byte_perm(__byte_perm(a, b, 0x0040), __byte_perm(c, d, 0x0040), 0x5410);
}

// residues of 16 scaled integers (thread-private, consecutive columns of one row) for the first T moduli -> planes[t][r][c..c+15]
// (one 16-byte store per modulus).  Tile: RS_TR rows x RS_TC columns per CTA of 256 threads; thread (tr = tid / 8,
// tcb = 16 * (tid % 8)).  T is a compile-time constant: the table entries become immediate constant-bank operands.
constexpr int RS_TR = 32, RS_TC = 128;
template <int T>
__device__ __forceinline__ void emit_residues(const long long (&xi)[16], const CrtTable& tab, long r, long rows, int c, int cols,
                                              uint8_t* __restrict__ planes, long ldp, long plane_stride) {
    uint32_t lo[16], hi[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const unsigned long long u = (unsigned long long)(xi[i] + 18014398509481984ll);       // + 2^54 > 0
        lo[i] = (uint32_t)u; hi[i] = (uint32_t)(u >> 32);
    }
    if (!(r < rows && c < cols)) return;
    uint8_t* dst0 = planes + r * ldp + c;
    const bool vec = c + 16 <= ldp;                  // zero residues pad the row up to ldp
#pragma unroll
    for (int t = 0; t < T; ++t) {
        const uint32_t clo = tab.clo[t], chi = tab.chi[t], magic = tab.magic[t], init = tab.init[t], p = (uint32_t)tab.p[t];
        uint32_t w[4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
            w[j] = pack4(residue_of(lo[4 * j], hi[4 * j], clo, chi, init, magic, p), residue_of(lo[4 * j + 1], hi[4 * j + 1], clo, chi, init, magic, p),
                         residue_of(lo[4 * j + 2], hi[4 * j + 2], clo, chi, init, magic, p), residue_of(lo[4 * j + 3], hi[4 * j + 3], clo, chi, init, magic, p));
        uint8_t* dst = dst0 + (long)t * plane_stride;
        if (vec) *reinterpret_cast<uint4*>(dst) = make_uint4(w[0], w[1], w[2], w[3]);
        else for (int i = 0; i < 16 && c + i < ldp; ++i) dst[i] = (uint8_t)((w[i >> 2] >> (8 * (i & 3))) & 0xff);
    }
}
template <int DUMMY = 0>
__device__ __forceinline__ void emit_residues_rt(int T, const long long (&xi)[16], const CrtTable& tab, long r, long rows, int c, int cols,
                                                 uint8_t* __restrict__ planes, long ldp, long plane_stride) {
    if (T == 15) emit_residues<15>(xi, tab, r, rows, c, cols, planes, ldp, plane_stride);
    else if (T == 16) emit_residues<16>(xi, tab, r, rows, c, cols, planes, ldp, plane_stride);
    else {                                           // any other count (tests): emit in two compile-time chunks
        if (T >= 8) emit_residues<8>(xi, tab, r, rows, c, cols, planes, ldp, plane_stride);
        CrtTable rest = tab;
        const int base = T >= 8 ? 8 : 0;
        for (int t = base; t < T; ++t) {
            rest.clo[0] = tab.clo[t]; rest.chi[0] = tab.chi[t]; rest.magic[0] = tab.magic[t]; rest.init[0] = tab.init[t]; rest.p[0] = tab.p[t];
            emit_residues<1>(xi, rest, r, rows, c, cols, planes + (long)t * plane_stride, ldp, plane_stride);
        }
    }
}

// src (rows x cols, ld) -> planes[t][r][c] (ldp bytes per row, plane_stride bytes per plane), scaled by 2^(bits - e) with
// e = exps[r] (scale_mode 0: per row), exps[c] (1: per column) or exps[0] (2).  A second integerisation of the same
// elements (planes2 != NULL: its own scale mode / exponents / bits / moduli) is produced in the same pass — [Abar | Bbar]
// feeds one contraction scaled per row and one scaled per column, and is read once.
__global__ void __launch_bounds__(256) k_to_residues(const double* __restrict__ src, long ld, long rows, int cols,
                                                     int scale_mode, const int* __restrict__ exps, int bits, CrtTable tab,
                                                     uint8_t* __restrict__ planes, long ldp, long plane_stride,
                                                     int scale_mode2, const int* __restrict__ exps2, int bits2, int T2,
                                                     uint8_t* __restrict__ planes2, long ldp2, long plane_stride2) {
    const long r = (long)blockIdx.y * RS_TR + (threadIdx.x >> 3);
    const int c = blockIdx.x * RS_TC + (threadIdx.x & 7) * 16;
    double x[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) x[i] = (r < rows && c + i < cols) ? src[r * ld + c + i] : 0.0;
    long long xi[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const int e = scale_mode == 0 ? (r < rows ? exps[r] : 0) : (scale_mode == 1 ? (c + i < cols ? exps[c + i] : 0) : exps[0]);
        xi[i] = __double2ll_rn(mul_pow2(x[i], bits - e));
    }
    emit_residues_rt(tab.T, xi, tab, r, rows, c, cols, planes, ldp, plane_stride);
    if (planes2) {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int e = scale_mode2 == 0 ? (r < rows ? exps2[r] : 0) : (scale_mode2 == 1 ? (c + i < cols ? exps2[c + i] : 0) : exps2[0]);
            xi[i] = __double2ll_rn(mul_pow2(x[i], bits2 - e));
        }
        emit_residues_rt(T2, xi, tab, r, rows, c, cols, planes2, ldp2, plane_stride2);      // moduli of a shorter table: a prefix
    }
}

// ARD K tile generated in registers (same arithmetic as k_rbf_tile_reg: x / ls differences, FMA chain, Cov<KIND>::phi) and
// converted on the spot to residue planes; K itself is never stored (the backward recomputes its tiles).  The same planes serve
// the forward (reduction over the inducing index: K-major) and the weight contraction (reduction over the rows: MN-major).
// One scale for the whole matrix, for every kind: 0 <= k <= outputscale < 2^kexp, kexp derived from the outputscale in-kernel (the kernel
// depends on nothing the factorisation produces, so it can run on a side stream under it).
template <int MAXD, int KIND>
__global__ void __launch_bounds__(256) k_rbf_residues(const double* __restrict__ X, const double* __restrict__ Zs,
                                                      const double* __restrict__ ls, const double* __restrict__ os, long R, int M, int D,
                                                      int bits, CrtTable tab, uint8_t* __restrict__ planes, long ldp, long plane_stride) {
    // inducing rows of the tile, dimension-major with a skew of one column per 16: the eight column groups of a warp (stride 16
    // columns) read eight different bank pairs (a [column][dimension] layout puts them all on one: an 8-way conflict per load)
    __shared__ __align__(16) double zs[MAXD][RS_TC + RS_TC / 16];
    const int tid = threadIdx.x;
    const int tr = tid >> 3, tcb = (tid & 7) * 16;
    const double s = os[0];
    const int sh = bits - exp_above(s);            // the same exponent tgp_prepare stores for the reconstruction (k_exp)
    // The launcher starts one CTA per tile: when this kernel runs on the side stream under the factorisation, its short CTAs
    // free slots often enough that the factorisation's small kernels do not queue behind thousands of tiles.  A CTA given
    // several tiles walks them column-block-major, so that it reloads its inducing rows rarely.
    const long row_tiles = cdiv(R, RS_TR);
    const long n_tiles = row_tiles * cdiv(M, RS_TC);
    int c0_loaded = -1;
    for (long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int c0 = (int)(tile / row_tiles) * RS_TC;
        const long r0 = (tile % row_tiles) * RS_TR;
        if (c0 != c0_loaded) {
            __syncthreads();
            for (int i = tid; i < RS_TC * MAXD; i += 256) {
                const int c = i / MAXD, d = i % MAXD, j = c0 + c;
                zs[d][c + (c >> 4)] = (j < M && d < D) ? Zs[(long)j * D + d] : 0.0;
            }
            __syncthreads();
            c0_loaded = c0;
        }
        const long r = r0 + tr;
        double xr[MAXD];
#pragma unroll
        for (int d = 0; d < MAXD; ++d) xr[d] = (r < R && d < D) ? X[r * D + d] / ls[d] : 0.0;
        long long xi[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int c = c0 + tcb + i;
            double val = 0.0;
            if (r < R && c < M) {
                double acc = 0.0;
#pragma unroll
                for (int d = 0; d < MAXD; ++d) { const double df = xr[d] - zs[d][tcb + i + (tid & 7)]; acc = fma(df, df, acc); }
                val = s * Cov<KIND>::phi(acc);
            }
            xi[i] = __double2ll_rn(mul_pow2(val, sh));
        }
        emit_residues_rt(tab.T, xi, tab, r, R, c0 + tcb, M, planes, ldp, plane_stride);
    }
}

// ---- step 3: the int8 GEMMs ------------------------------------------------------------------------------------------
struct Params {
    int Mrows, Ncols, K, T;
    int tri_mode, tri_rows;          // as gemm_tc.cuh: 1: B rows n < tri_rows are lower triangular (k <= n);  2: k < tri_rows needs k >= n
    int lower_rows;                  // > 0: for output rows m < lower_rows tiles strictly above the diagonal are skipped
    int mn_major;                    // bit 0: A planes, bit 1: B planes are stored [t][k][m] (MN-major) instead of [t][m][k] (K-major):
                                     // the tensor core reads the transposed tile straight from shared memory, so a contraction
                                     // over the ROWS of row-major planes needs no transposed copy
    uint8_t* C; long ldc, plane_stride_c;       // residue planes of the result [t][m][n]
    int p[MAX_T]; uint32_t magic[MAX_T];
};

__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}
// kind::i8: UNSIGNED 8-bit A and B (format 0), S32 accumulate, M = 128, N = BN; bits 15 / 16: A / B operand is MN-major
__device__ __forceinline__ uint32_t make_idesc_i8(int mn_major) {
    return (2u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24) |
           ((mn_major & 1) ? (1u << 15) : 0u) | ((mn_major & 2) ? (1u << 16) : 0u);
}
// MN-major, 128-byte swizzle: a tile is BK k-rows of 128 bytes (128 consecutive m); 8 k-rows = 1024 B apart (SBO); for the
// 256-wide B operand the second 128-column atom sits one A-sized tile further (LBO = BK * 128 B)
__device__ __forceinline__ uint64_t make_desc_mn(const void* smem_tile) {
    const uint64_t addr = (uint64_t)((tc::smem_u32(smem_tile) & 0x3FFFF) >> 4);
    return addr | ((uint64_t)((BK * 128) >> 4) << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(tc::smem_u32(dst)), "l"(map), "r"(tc::smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

// multicast variants: the tile lands at the same shared-memory offset of every CTA in `mask`, and completes tx bytes on the
// mbarrier at the same offset of each of them
__device__ __forceinline__ void tma_load_3d_mc(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, uint16_t mask) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4, %5}], [%2], %6;"
        ::"r"(tc::smem_u32(dst)), "l"(map), "r"(tc::smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "h"(mask) : "memory");
}
// tcgen05.commit arriving on the mbarrier at this offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(tc::smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// acc mod p in [0, p) for a non-negative accumulator (u8 x u8 products): Barrett with magic = ceil(2^32 / p) = (2^32 + d) / p,
// 0 <= d < p.  umulhi floors acc / p + acc d / (p 2^32), whose second term is in [0, 1/2) for acc < 2^31: the quotient is exact or
// one too large, r = acc - q p lands in [-p, p), one conditional addition fixes it.
__device__ __forceinline__ uint32_t mod_p(uint32_t acc, uint32_t p, uint32_t magic) {
    const int r = (int)(acc - __umulhi(acc, magic) * p);
    return (uint32_t)(r < 0 ? r + (int)p : r);
}

// 32 lanes x 32 consecutive 32-bit TMEM columns -> 32 registers per thread (asynchronous: complete after tcgen05.wait::ld)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}

// waits for the outstanding TMEM loads; the registers of the load being consumed are passed through as in/out operands so that the
// compiler cannot move their uses above the wait
__device__ __forceinline__ void tmem_wait_ld(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                   "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                   "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :: "memory");
}

// Launched as clusters of TWO CTAs that own vertically adjacent 128-row tiles of the same (modulus, n-tile): the B tile is the
// same for both, so each CTA fetches one 128-row half of it and MULTICASTS it into both shared memories (L2 -> SM traffic per
// CTA and k-block: 16 KiB of A + 16 KiB of B instead of 16 + 32; the single-CTA version was L2-bound at ~10 TB/s).  A stage
// may be refilled only when BOTH consumers have released it: the MMA issuer's tcgen05.commit arrives on the `empty` barrier of
// both CTAs (count 2).
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
gemm_i8_mod_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const Params p) {
    using namespace tc;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
    uint64_t* empty = full + STAGES;
    uint64_t* tfull = empty + STAGES;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rank = (int)cluster_ctarank();
    const int n_clusters = gridDim.x >> 1, cluster_id = blockIdx.x >> 1;
    const int tiles_m = (p.Mrows + BM - 1) / BM, tiles_n = (p.Ncols + BN - 1) / BN;
    const int pairs_m = (tiles_m + 1) >> 1;
    const long n_work = (long)p.T * pairs_m * tiles_n;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 2); }
        for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();              // the peer's barriers are initialised before anything is multicast into this CTA
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // work item (cluster-wide) -> (modulus t, pair of m-tiles, n-tile, k-range); this CTA's m-tile is 2 * pair + rank.  n fastest
    // (the A row blocks are shared by consecutive clusters), modulus slowest (one modulus' planes of both operands fit the L2).
    // Both CTAs of a cluster run the same sequence with the same k-range, so their pipelines stay in step.
    auto decode = [&](long w, int& t, int& m0, int& n0, int& kb, int& ke) -> bool {
        n0 = (int)(w % tiles_n) * BN;
        const long r = w / tiles_n;
        const int mp = (int)(r % pairs_m);
        m0 = (2 * mp + rank) * BM;
        t = (int)(r / pairs_m);
        const int m_hi = (2 * mp + 1) * BM;                    // the lower tile of the pair
        if (p.lower_rows > 0 && m_hi < p.lower_rows && n0 > m_hi + BM - 1) return false;       // both tiles strictly above the diagonal
        kb = 0; ke = p.K;
        if (p.tri_mode == 1 && n0 < p.tri_rows) ke = min(p.K, n0 + BN);
        if (p.tri_mode == 2 && n0 < p.tri_rows) kb = (n0 / BK) * BK;
        return ke > kb;
    };

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            uint8_t* const bhalf_off = reinterpret_cast<uint8_t*>((uintptr_t)(A_BYTES + rank * (B_BYTES / 2)));
            for (long w = cluster_id; w < n_work; w += n_clusters) {
                int t, m0, n0, kb, ke;
                if (!decode(w, t, m0, n0, kb, ke)) continue;
                for (int k = kb; k < ke; k += BK) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    uint8_t* st = smem + stage * STAGE_BYTES;
                    mbar_expect_tx(&full[stage], STAGE_BYTES);          // own A + both halves of B
                    // MN-major planes [t][k][m]: boxes of 128 m-bytes x BK k-rows; K-major [t][m][k]: BK k-bytes x rows
                    if (p.mn_major & 1) tma_load_3d(st, &mapA, &full[stage], m0, k, t);
                    else tma_load_3d(st, &mapA, &full[stage], k, m0, t);
                    uint8_t* bdst = st + (uintptr_t)bhalf_off;           // this CTA's 128-row half of the B tile, for both CTAs
                    if (p.mn_major & 2) tma_load_3d_mc(bdst, &mapB, &full[stage], n0 + 128 * rank, k, t, (uint16_t)3);
                    else tma_load_3d_mc(bdst, &mapB, &full[stage], k, n0 + 128 * rank, t, (uint16_t)3);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = make_idesc_i8(p.mn_major);
            int stage = 0; uint32_t phase = 0;
            int buf = 0; uint32_t bphase = 0;
            for (long w = cluster_id; w < n_work; w += n_clusters) {
                int t, m0, n0, kb, ke;
                if (!decode(w, t, m0, n0, kb, ke)) continue;
                mbar_wait(&tempty[buf], bphase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)buf * BN;
                uint32_t accum = 0;
                for (int k = kb; k < ke; k += BK) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    uint8_t* st = smem + stage * STAGE_BYTES;
                    // per 32-deep MMA the descriptor advances 32 B inside the swizzle row (K-major) or 32 k-rows of 128 B (MN-major)
                    const uint64_t dA = (p.mn_major & 1) ? make_desc_mn(st) : make_desc(st);
                    const uint64_t dB = (p.mn_major & 2) ? make_desc_mn(st + A_BYTES) : make_desc(st + A_BYTES);
                    const uint64_t sA = (uint64_t)(((p.mn_major & 1) ? UMMA_K * 128 : UMMA_K) >> 4);
                    const uint64_t sB = (uint64_t)(((p.mn_major & 2) ? UMMA_K * 128 : UMMA_K) >> 4);
#pragma unroll
                    for (int kk = 0; kk < BK / UMMA_K; ++kk) {
                        umma_i8(tmem_d, dA + kk * sA, dB + kk * sB, idesc, accum);
                        accum = 1;
                    }
                    umma_commit_mc(&empty[stage], (uint16_t)3);       // releases the stage in BOTH CTAs when these MMAs retire
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit(&tfull[buf]);
                if (++buf == 2) { buf = 0; bphase ^= 1; }
            }
        }
    } else {
        const int q = warp & 3;
        const int half = (warp - 2) >> 2;              // column part of this warp
        int buf = 0; uint32_t bphase = 0;
        for (long w = cluster_id; w < n_work; w += n_clusters) {
            int t, m0, n0, kb, ke;
            if (!decode(w, t, m0, n0, kb, ke)) continue;
            const uint32_t pm = (uint32_t)p.p[t], ip = p.magic[t];
            mbar_wait(&tfull[buf], bphase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + (uint32_t)buf * BN + (uint32_t)(half * EPI_COLS) + ((uint32_t)(q * 32) << 16);
            const int row = m0 + q * 32 + lane;
            const int nbase = n0 + half * EPI_COLS;
            // this CTA's tile may lie strictly above the diagonal (its pair partner does not) or below the last row: nothing to store
            const bool store = row < p.Mrows && !(p.lower_rows > 0 && m0 < p.lower_rows && n0 > m0 + BM - 1);
            uint8_t* dst = p.C + (long)t * p.plane_stride_c + (long)row * p.ldc + nbase;
            // EPI_COLS accumulator columns per thread in 32-column TMEM loads, software-pipelined: the load of chunk c + 1 is in
            // flight while chunk c is reduced mod p, packed and stored (tcgen05.wait::ld waits for every outstanding load, so the
            // next one is issued right after the wait)
            uint32_t ra[32], rb[32];
            tmem_ld32(taddr, ra);
#pragma unroll
            for (int ci = 0; ci < EPI_COLS / 32; ++ci) {
                const int c = ci * 32;
                uint32_t (&r)[32] = (ci & 1) ? rb : ra;
                tmem_wait_ld(r);
                if (ci + 1 < EPI_COLS / 32) tmem_ld32(taddr + (uint32_t)(c + 32), (ci & 1) ? ra : rb);
                if (store) {
                    uint32_t packed[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        packed[i] = pack4(mod_p(r[4 * i], pm, ip), mod_p(r[4 * i + 1], pm, ip), mod_p(r[4 * i + 2], pm, ip), mod_p(r[4 * i + 3], pm, ip));
                    if (nbase + c + 32 <= p.ldc) {
                        *reinterpret_cast<uint4*>(dst + c) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
                        *reinterpret_cast<uint4*>(dst + c + 16) = make_uint4(packed[4], packed[5], packed[6], packed[7]);
                    } else {
                        for (int i = 0; i < 32 && nbase + c + i < p.ldc; ++i) dst[c + i] = (uint8_t)((packed[i >> 2] >> (8 * (i & 3))) & 0xff);
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[buf]);
            if (++buf == 2) { buf = 0; bphase ^= 1; }
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();              // no CTA leaves while its peer may still multicast into it or arrive on its barriers
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512));
    }
}

// 3D map over residue planes: (cols = K bytes, rows, T); box = 128 bytes x box_rows x 1, 128B swizzle
struct PlaneMapKey { const void* base; long rows, cols, ld, plane_stride; int T, box_rows; };
struct PlaneMapCache {
    static constexpr int N = 32;
    PlaneMapKey key[N]; CUtensorMap map[N]; int used = 0, next = 0;
};
inline int make_plane_map(CUtensorMap* map, const uint8_t* base, long rows, long cols, long ld, long plane_stride, int T, int box_rows,
                          int box_cols = BK) {
    static PlaneMapCache cache;
    for (int i = 0; i < cache.used; ++i) {
        const PlaneMapKey& k = cache.key[i];
        if (k.base == base && k.rows == rows && k.cols == cols && k.ld == ld && k.plane_stride == plane_stride && k.T == T &&
            k.box_rows == box_rows + 1000 * box_cols) {
            *map = cache.map[i];
            return 0;
        }
    }
    tc::EncodeTiledFn fn = tc::encode_fn();
    if (!fn) return set_error(-101, "cuTensorMapEncodeTiled not available from the driver");
    if ((ld & 15) != 0 || (plane_stride & 15) != 0 || (reinterpret_cast<uintptr_t>(base) & 15) != 0)
        return set_error(-2, "residue planes must be 16-byte aligned with 16-byte multiples as strides");
    cuuint64_t gdim[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)T};
    cuuint64_t gstr[2] = {(cuuint64_t)ld, (cuuint64_t)plane_stride};
    cuuint32_t box[3] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t*>(base), gdim, gstr, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(-102, "cuTensorMapEncodeTiled (residue planes) failed");
    const int i = cache.used < PlaneMapCache::N ? cache.used++ : (cache.next = (cache.next + 1) % PlaneMapCache::N);
    cache.key[i] = PlaneMapKey{base, rows, cols, ld, plane_stride, T, box_rows + 1000 * box_cols};
    cache.map[i] = *map;
    return 0;
}

// K-major: rows = operand rows (m or n), cols = reduction length.  MN-major (Params.mn_major): the planes are stored
// [t][k][m]: rows = reduction length, cols = operand rows.
struct Planes { const uint8_t* base; long rows, cols, ld, plane_stride; };

inline int gemm_i8_mod(const Planes& A, const Planes& B, Params p, cudaStream_t st) {
    if (p.Mrows <= 0 || p.Ncols <= 0 || p.K <= 0) return 0;
    if ((long)p.K * 65025 >= 2147483648L) return set_error(-3, "u8 reduction too long for exact s32 accumulation (K <= 33025)");
    CUtensorMap mA, mB;
    // MN-major boxes: 128 operand rows (contiguous bytes) x BK reduction rows
    if (p.mn_major & 1) TGP_TRY(make_plane_map(&mA, A.base, A.rows, A.cols, A.ld, A.plane_stride, p.T, BK, 128));
    else TGP_TRY(make_plane_map(&mA, A.base, A.rows, A.cols, A.ld, A.plane_stride, p.T, BM));
    if (p.mn_major & 2) TGP_TRY(make_plane_map(&mB, B.base, B.rows, B.cols, B.ld, B.plane_stride, p.T, BK, 128));
    else TGP_TRY(make_plane_map(&mB, B.base, B.rows, B.cols, B.ld, B.plane_stride, p.T, BN / 2));      // each CTA loads one half
    const CrtTable& tab = crt_table(p.T);
    for (int t = 0; t < p.T; ++t) { p.p[t] = tab.p[t]; p.magic[t] = tab.magic[t]; }
    static PerDeviceOnce attr_once;
    if (attr_once.first()) cudaFuncSetAttribute(gemm_i8_mod_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    const long pairs = (long)((cdiv(p.Mrows, BM) + 1) / 2) * cdiv(p.Ncols, BN) * p.T;        // cluster-wide work items
    const int grid = 2 * (int)(pairs < 74 ? pairs : 74);
    const bool timed = g_gemm_timer.enabled;
    if (timed) g_gemm_timer.begin(2, st);
    gemm_i8_mod_kernel<<<grid, THREADS, SMEM_BYTES, st>>>(mA, mB, p);
    if (timed) g_gemm_timer.end(st);
    return check_launch("gemm_i8_mod_kernel");
}

// ---- step 4 + 5: CRT reconstruction -----------------------------------------------------------------------------------
// Values of sum_t r_t w_t mod P (centred) for the FOUR elements whose residues sit in the bytes of w[t], as doubles (relative
// error <= 3 * 2^-53).  Integer first: the residues of one element are gathered into dp4a operands (a 4 x 4 byte transpose per
// group of four moduli), and for every byte position k of the weights  S_k = sum_t r_t byte_k(w_t)  (< 16 * 255 * 255 < 2^20) is
// a handful of dp4a with constant-bank operands; total = sum_k S_k 256^k exactly.  Four 40-bit-spaced words
// W_j = sum_{i<5} S_{5j+i} 256^i (< 2^53: exact in FP64) are formed from the S_k; the multiple of P is m = rint(total / P) with
// total evaluated in FP64 (m <= 2^12: its rounding error is ~2^-41, far inside the margin the bit budget leaves between |C'| / P
// and 1/2); W_j - m P_j is exact, carries are propagated, and only the final FMAs round.
__device__ __forceinline__ double u32_to_double(uint32_t x) {          // (2^52 + x) - 2^52: no conversion instruction
    return __hiloint2double(0x43300000, (int)x) - 4503599627370496.0;
}
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
    return r;
}

template <int T>
__device__ __forceinline__ void crt_value4(const uint32_t (&w)[T], const CrtTable& tab, double (&out)[4]) {
    constexpr int NG = (T + 3) / 4;
    constexpr int NB = T;                     // bytes of P for the instantiated counts (9, 12, 15, 16 moduli: P < 256^T)
    uint32_t q[4][NG];                        // q[i][g]: residues 4g..4g+3 of element i
#pragma unroll
    for (int g = 0; g < NG; ++g) {
        const uint32_t a = w[4 * g], b = 4 * g + 1 < T ? w[4 * g + 1] : 0u, c = 4 * g + 2 < T ? w[4 * g + 2] : 0u,
                       d = 4 * g + 3 < T ? w[4 * g + 3] : 0u;
        const uint32_t t0 = prmt(a, b, 0x5140u), t1 = prmt(a, b, 0x7362u);      // a0 b0 a1 b1 | a2 b2 a3 b3
        const uint32_t t2 = prmt(c, d, 0x5140u), t3 = prmt(c, d, 0x7362u);
        q[0][g] = prmt(t0, t2, 0x5410u); q[1][g] = prmt(t0, t2, 0x7632u);
        q[2][g] = prmt(t1, t3, 0x5410u); q[3][g] = prmt(t1, t3, 0x7632u);
    }
    const double two = 1099511627776.0, inv = 9.094947017729282e-13;       // 2^40, 2^-40
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        uint32_t S[20];
#pragma unroll
        for (int k = 0; k < 20; ++k) {
            uint32_t s = 0u;
            if (k < NB) {
#pragma unroll
                for (int g = 0; g < NG; ++g) s = __dp4a(q[i][g], tab.wb[g][k], s);
            }
            S[k] = s;
        }
        double W[4];
#pragma unroll
        for (int j = 0; j < 4; ++j)           // (S_5j + S_5j+1 2^8) + (S_5j+2 + S_5j+3 2^8) 2^16 + S_5j+4 2^32: < 2^53, exact
            W[j] = fma(u32_to_double(S[5 * j + 4]), 4294967296.0,
                       fma(u32_to_double(S[5 * j + 2] + (S[5 * j + 3] << 8)), 65536.0, u32_to_double(S[5 * j] + (S[5 * j + 1] << 8))));
        const double m = rint(fma(fma(fma(W[3], two, W[2]), two, W[1]), two, W[0]) * tab.invP);
        double D0 = fma(-m, tab.Pw[0], W[0]), D1 = fma(-m, tab.Pw[1], W[1]), D2 = fma(-m, tab.Pw[2], W[2]), D3 = fma(-m, tab.Pw[3], W[3]);
        double c = rint(D0 * inv); D0 = fma(-c, two, D0); D1 += c;
        c = rint(D1 * inv); D1 = fma(-c, two, D1); D2 += c;
        c = rint(D2 * inv); D2 = fma(-c, two, D2); D3 += c;
        out[i] = fma(fma(fma(D3, two, D2), two, D1), two, D0);
    }
}

// stats (forward only; cols = 2 * stat_M, row = [a | b]): mu[r] = sum_{c < M} out * m[c], v[r] = os - sum_{c<M} out^2 +
// sum_{c>=M} out^2 — the q(f) marginals come out of the reconstruction pass, [A | B] is not re-read for them
struct RowStats { const double* m; const double* os; double* mu; double* v; int M; };

// R planes [t][rows][ldr] -> out[r * ldo + c] = (or +=) crt * 2^(ea + eb - bits2)
//   ea: row exponents (ea_mode 0) / one exponent ea[0] (ea_mode 2);  eb: per-column exponents (eb_mode 1) / eb[0] (2)
//   accumulate = 1: FP64 atomicAdd (weight gradients summed over row chunks); lower_rows > 0: rows r < lower_rows only c <= r
// one warp per row, four consecutive columns per lane per step
template <int T>
__global__ void __launch_bounds__(256) k_crt_combine(const uint8_t* __restrict__ R, long ldr, long plane_stride, long rows, int cols,
                                                     const __grid_constant__ CrtTable tab, int bits2, const int* __restrict__ ea, int ea_mode,
                                                     const int* __restrict__ eb, int eb_mode, double* __restrict__ out, long ldo,
                                                     int accumulate, int lower_rows, RowStats st) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    for (long r = (long)blockIdx.x * wpb + wid; r < rows; r += (long)gridDim.x * wpb) {
        const int era = (ea_mode == 0 ? ea[r] : ea[0]) - bits2;
        const int climit = (lower_rows > 0 && r < lower_rows) ? (int)min((long)cols, r + 1) : cols;
        double sm = 0.0, sa = 0.0, sb = 0.0;
        for (int c0 = lane * 4; c0 < climit; c0 += 128) {
            uint32_t w[T];
#pragma unroll
            for (int t = 0; t < T; ++t) w[t] = *reinterpret_cast<const uint32_t*>(R + (long)t * plane_stride + r * ldr + c0);
            int e4[4];
            if (eb_mode == 1) {
                if (c0 + 4 <= cols && ((reinterpret_cast<uintptr_t>(eb + c0) & 15) == 0)) {
                    const int4 e = *reinterpret_cast<const int4*>(eb + c0);
                    e4[0] = e.x; e4[1] = e.y; e4[2] = e.z; e4[3] = e.w;
                } else {
#pragma unroll
                    for (int i = 0; i < 4; ++i) e4[i] = c0 + i < cols ? eb[c0 + i] : 0;
                }
            } else {
                e4[0] = e4[1] = e4[2] = e4[3] = eb[0];
            }
            double v4[4];
            crt_value4<T>(w, tab, v4);
#pragma unroll
            for (int i = 0; i < 4; ++i) v4[i] = mul_pow2(v4[i], era + e4[i]);
            double* o = out + r * ldo + c0;
            if (!accumulate && c0 + 4 <= climit && ((reinterpret_cast<uintptr_t>(o) & 15) == 0)) {
                *reinterpret_cast<double2*>(o) = make_double2(v4[0], v4[1]);
                *reinterpret_cast<double2*>(o + 2) = make_double2(v4[2], v4[3]);
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (c0 + i < climit) { if (accumulate) atomicAdd(o + i, v4[i]); else o[i] = v4[i]; }
            }
            if (st.mu) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int c = c0 + i;
                    if (c < climit) {
                        if (c < st.M) { sm = fma(v4[i], __ldg(st.m + c), sm); sa = fma(v4[i], v4[i], sa); }
                        else sb = fma(v4[i], v4[i], sb);
                    }
                }
            }
        }
        if (st.mu) {
            sm = warp_sum(sm); sa = warp_sum(sa); sb = warp_sum(sb);
            if (lane == 0) { st.mu[r] = sm; st.v[r] = st.os[0] - sa + sb; }
        }
    }
}

inline int crt_grid(long rows) {
    const long blocks = cdiv(rows, 8);
    return (int)(blocks < 148 * 8 ? (blocks < 1 ? 1 : blocks) : 148 * 8);
}

}  // namespace i8
}  // namespace tgp
