// Host-side orchestration of compute mode TGP_F64_I8: FP64-accurate batch contractions on the tcgen05 integer tensor path
// (gemm_i8.cuh).  Same mathematics and reduce-buffer contents as the tensor-core mode of tc_driver.cuh (two independent
// contractions of the K tile with the stacked operand W = [L^-1; C], C = L_S^T L^-1), but every product is exact up to a
// 52/53-bit truncation of the operands, so the results carry the FP64 parity tolerances.
#pragma once
#include "step_kernels.cuh"
#include "backward_kernels.cuh"
#include "row_kernels.cuh"
#include "gemm_i8.cuh"

namespace tgp {
namespace crt {

using i8::Planes;
constexpr long CRT_ROW_CHUNK = 16384;
constexpr int T_ALL = 16;                          // planes generated for operands shared with the weight contraction

inline long pad16(long x) { return (x + 15) / 16 * 16; }
inline long chunk_rows(long R) { return R < CRT_ROW_CHUNK ? R : CRT_ROW_CHUNK; }

// bits left for the second operand when the first one carries `fixed` bits: 2 k 2^(fixed + b) < P
inline int bits_other(int T, long k_red, int fixed) {
    const int b = (int)floor(i8::crt_table(T).log2P - 1.0 - log2((double)(k_red > 1 ? k_red : 1)) - (double)fixed - 1e-6);
    return b > 53 ? 53 : (b < 1 ? 1 : b);
}
// forward  [A | B] = K W^T, reduction M: K carries 53 bits (one scale for the whole matrix); 15 moduli if W keeps >= 52 bits
inline int fwd_T(int M) { return bits_other(15, M, 53) >= 52 ? 15 : 16; }
inline int fwd_bits_w(int M) { return bits_other(fwd_T(M), M, 53); }
// backward-data  Kbar = ABbar W~, reduction 2M: ABbar carries the bits of the weight contraction's planes (one set serves both);
// 15 moduli if W~ keeps >= 52 bits
inline int bwd_T(int M, int bits_x) { return bits_other(15, 2L * M, bits_x) >= 52 ? 15 : 16; }
inline int bwd_bits_w(int M, int bits_x) { return bits_other(bwd_T(M, bits_x), 2L * M, bits_x); }
// weight contraction  [Gbar; Cbar] += ABbar^T K, reduction = rows of the chunk: all 16 moduli, K^T carries 53 bits
inline int wgt_bits(long rc) { return bits_other(T_ALL, rc, 53); }

struct StepPlanes {               // per step: residues of W = [Linv; C] (2M x M), scaled per row and scaled per column
    double* Wst;                  // FP64 stacked operand (2M x M, ld M)
    uint8_t *W;                    // planes [T][2M][ldk], per-row scale: forward operand (reduction over its columns, K-major)
    uint8_t *Wc;                   // planes [T][2M][ldk] of W~ = diag(2^c) W, per-column scale: backward-data operand, rebuilt per row
                                  // chunk (c = column exponents of that chunk's [Abar | Bbar]); reduction over its ROWS: the tensor
                                  // core reads it MN-major, no transposed copy
    int *w_row_exp, *k_exp;
    long ldk;
};

// the residue region of the step workspace, carved after its FP64 region
inline StepPlanes step_planes(Carve& c, int M) {
    StepPlanes s;
    s.ldk = pad16(M);
    s.Wst = c.take<double>(2L * M * M);
    s.W = c.take<uint8_t>(T_ALL * 2L * M * s.ldk);
    s.Wc = c.take<uint8_t>(T_ALL * 2L * M * s.ldk);
    s.w_row_exp = c.take<int>(2L * M);
    s.k_exp = c.take<int>(1);
    return s;
}

struct BatchView {
    double *AB;                   // (R x 2M) FP64, forward -> backward ([A | B], turned into [Abar | Bbar] in place)
    double *Kbuf;                 // (R x M) FP64 K_xz — only for D > 32 (staged generation); otherwise K_xz exists as residue planes
                                  // only and the kernel-gradient pass recomputes its tiles from X and Z
    double *Kbar;                 // (Rc x M)
    uint8_t *Kp;                   // planes [T_ALL][R][ldk]   K_xz residues: forward operand AND weight-contraction operand
    uint8_t *Op;                   // planes [T][Rc][ld2m]     result residues of the forward
    uint8_t *Pc;                   // planes [T_ALL][Rc][ld2m] ABbar scaled per column: K-major operand of Kbar = ABbar W~ and MN-major
                                  // operand of the weight contraction
    uint8_t *Kbp;                  // planes [T][Rc][ldk]      Kbar result residues
    uint8_t *Gp;                   // planes [T_ALL][2M][ldk]  weight-contraction result residues
    int *col_exp, *wc_exp, *zero_exp;   // (2M) column exponents of ABbar, (M) of W~, a zero
    long Rc, ldk, ld2m;
};

// D <= 32: K_xz is generated straight into residue planes (i8::k_rbf_residues) and recomputed by the backward
inline bool keeps_kxz(int D) { return D > 32; }

inline BatchView batch_view(Carve& c, int M, int D, long R) {
    BatchView b;
    b.Rc = chunk_rows(R); b.ldk = pad16(M); b.ld2m = pad16(2L * M);
    b.AB = c.take<double>(R * 2 * M);
    b.Kbuf = keeps_kxz(D) ? c.take<double>(R * M) : nullptr;
    b.Kbar = c.take<double>(b.Rc * M);
    b.Kp = c.take<uint8_t>(T_ALL * R * b.ldk);
    b.Op = c.take<uint8_t>(T_ALL * b.Rc * b.ld2m);
    b.Pc = c.take<uint8_t>(T_ALL * b.Rc * b.ld2m);
    b.Kbp = c.take<uint8_t>(T_ALL * b.Rc * b.ldk);
    b.Gp = c.take<uint8_t>(T_ALL * 2 * M * b.ldk);
    b.col_exp = c.take<int>(2L * M);
    b.wc_exp = c.take<int>(M);
    b.zero_exp = c.take<int>(1);
    return b;
}

// stacked FP64 operand Wst = [Linv; C] (ld M) from the padded step matrices (ld Mp)
__global__ void k_stack_w(const double* __restrict__ Linv, const double* __restrict__ Cm, long ld, int M, double* __restrict__ Wst) {
    const int r = blockIdx.x;
    const double* src = r < M ? Linv + (long)r * ld : Cm + (long)(r - M) * ld;
    for (int c = threadIdx.x; c < M; c += blockDim.x) Wst[(long)r * M + c] = src[c];
}
__global__ void k_exp_of_scalar(const double* __restrict__ x, int* __restrict__ e) { e[0] = i8::exp_above(x[0]); }

inline int fill_int(int* p, long n, int v, cudaStream_t st) {
    i8::k_fill_int<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(p, n, v);
    return check_launch("k_fill_int");
}

inline int exponents(const double* src, long ld, long rows, int cols, int* row_exp, int* col_exp, cudaStream_t st) {
    if (row_exp) TGP_TRY(fill_int(row_exp, rows, -100000, st));
    if (col_exp) TGP_TRY(fill_int(col_exp, cols, -100000, st));
    dim3 grid((unsigned)cdiv(cols, 256), (unsigned)cdiv(rows, 64));
    i8::k_exponents<<<grid, 256, 0, st>>>(src, ld, rows, cols, row_exp, col_exp);
    return check_launch("k_exponents");
}

inline int to_residues(const double* src, long ld, long rows, int cols, int scale_mode, const int* exps, int bits, int T,
                       uint8_t* planes, long ldp, long plane_stride, cudaStream_t st, int scale_mode2 = 0, const int* exps2 = nullptr,
                       int bits2 = 0, int T2 = 0, uint8_t* planes2 = nullptr, long ldp2 = 0, long plane_stride2 = 0) {
    dim3 grid((unsigned)cdiv(cols, i8::RS_TC), (unsigned)cdiv(rows, i8::RS_TR));
    // the second set may use more moduli than the first: pass the longer table, the first set's count travels in tab.T
    i8::CrtTable tab = i8::crt_table(T > T2 ? T : T2);
    tab.T = T;
    i8::k_to_residues<<<grid, 256, 0, st>>>(src, ld, rows, cols, scale_mode, exps, bits, tab, planes, ldp, plane_stride, scale_mode2,
                                           exps2, bits2, T2, planes2, ldp2, plane_stride2);
    return check_launch("k_to_residues");
}

inline int combine(const uint8_t* R, long ldr, long plane_stride, long rows, int cols, int T, int bits2, const int* ea, int ea_mode,
                   const int* eb, int eb_mode, double* out, long ldo, int accumulate, int lower_rows, cudaStream_t st,
                   i8::RowStats stats = i8::RowStats{nullptr, nullptr, nullptr, nullptr, 0}) {
    const i8::CrtTable& tab = i8::crt_table(T);
    const int grid = i8::crt_grid(rows);
#define TGP_CC(TT) i8::k_crt_combine<TT><<<grid, 256, 0, st>>>(R, ldr, plane_stride, rows, cols, tab, bits2, ea, ea_mode, eb, eb_mode, out, \
                                                             ldo, accumulate, lower_rows, stats)
    switch (T) {          // the modulus count is a compile-time constant of the kernel (immediate constant-bank operands)
        case 16: TGP_CC(16); break;
        case 15: TGP_CC(15); break;
        case 12: TGP_CC(12); break;
        case 9: TGP_CC(9); break;
        default: return set_error(-1, "CRT reconstruction is instantiated for 9, 12, 15 and 16 moduli");
    }
#undef TGP_CC
    return check_launch("k_crt_combine");
}

// residue planes of K_xz (i8::k_rbf_residues)
template <int KIND>
inline int rbf_residues(const double* X, const double* Zs, const double* ls, const double* os, long R, int M, int D, int T,
                        uint8_t* planes, long ldp, long plane_stride, cudaStream_t st) {
    // one CTA per tile (short CTAs: a concurrent high-priority stream gets slots every few microseconds)
    const unsigned grid = (unsigned)(cdiv(M, i8::RS_TC) * cdiv(R, i8::RS_TR));
    const i8::CrtTable& tab = i8::crt_table(T);
#define TGP_RR(MD) i8::k_rbf_residues<MD, KIND><<<grid, 256, 0, st>>>(X, Zs, ls, os, R, M, D, 53, tab, planes, ldp, plane_stride)
    if (D <= 4) TGP_RR(4);
    else if (D <= 8) TGP_RR(8);
    else if (D <= 16) TGP_RR(16);
    else if (D <= 32) TGP_RR(32);
    else return -7;              // wider inputs: the caller falls back to launch_rbf + to_residues
#undef TGP_RR
    return check_launch("k_rbf_residues");
}

// per step, after run_prepare: residues of W scaled per row (forward operand; the backward-data operand is built per chunk)
inline int make_step_planes(const StepView& v, const StepPlanes& s, cudaStream_t st) {
    const int M = v.M;
    k_stack_w<<<2 * M, 256, 0, st>>>(v.Linv, v.Cm, v.Mp, M, s.Wst);
    TGP_TRY(check_launch("k_stack_w"));
    k_exp_of_scalar<<<1, 1, 0, st>>>(v.os, s.k_exp);
    TGP_TRY(check_launch("k_exp_of_scalar"));
    TGP_TRY(exponents(s.Wst, M, 2L * M, M, s.w_row_exp, nullptr, st));
    return to_residues(s.Wst, M, 2L * M, M, 0, s.w_row_exp, fwd_bits_w(M), fwd_T(M), s.W, s.ldk, 2L * M * s.ldk, st);
}

// ---- backward operand: [Abar | Bbar] is never materialised ------------------------------------------------------------
// Abar = g_mu m - 2 g_v A, Bbar = 2 g_v B (upstream row gradients applied to the forward's [A | B], which stays untouched).
// Both contractions that consume it — Kbar = [Abar | Bbar] W over its columns and [Gbar; Cbar] += [Abar | Bbar]^T K over its
// rows — read ONE set of residue planes, integerised per COLUMN (exponent c_j above the column maximum of the chunk): the
// row contraction needs a scale that is constant along the reduction, so 2^c_j moves into the other operand, W~ = diag(2^c) W,
// whose planes are rebuilt per chunk (2M x M elements: 6 % of the chunk).  Every consumer of Kbar sums over the rows
// (Kbar o K -> dZ, dlengthscale, doutputscale), so a column-wise fixed point — absolute accuracy 2^-53 of the column maximum —
// is what FP64 accumulation of those sums delivers too.
__device__ __forceinline__ double abbar_value(double gm, double gv, double mj, double ab, bool left) {
    return left ? gm * mj - 2.0 * gv * ab : 2.0 * gv * ab;
}

// pass 1: column exponents of [Abar | Bbar] (pre-set to a very small value), dm[j] += sum_n g_mu A[n,j], dos += sum_n g_v.
// ABS_ROWS rows x 128 columns per CTA (measured: 64 rows 0.077 ms per 16384-row chunk, 256 rows 0.15 ms — it needs the CTAs).  The
// exponent is taken from the running maximum of |.| once per thread: a frexp per element made this kernel 1.5x slower.
constexpr int ABS_ROWS = 64;
__global__ void __launch_bounds__(128) k_abbar_stats(const double* __restrict__ AB, const double* __restrict__ g_mu,
                                                     const double* __restrict__ g_v, const double* __restrict__ m, long R, int M,
                                                     double* __restrict__ dm, double* __restrict__ dos, int* __restrict__ col_exp) {
    const int j = blockIdx.x * 128 + threadIdx.x;
    const long n0 = (long)blockIdx.y * ABS_ROWS, n1 = min(n0 + ABS_ROWS, R);
    const double mj = j < M ? m[j] : 0.0;
    double acc = 0.0, accv = 0.0;
    double amax = 0.0, bmax = 0.0;                      // column maxima of |.|: the exponent is taken once, at the end
    for (long nb = n0; nb < n1; nb += 8) {              // eight rows per iteration: their loads are in flight together
        double a[8], b[8], gm[8], gv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const long n = nb + u;
            const bool ok = n < n1;
            gm[u] = ok ? g_mu[n] : 0.0; gv[u] = ok ? g_v[n] : 0.0;
            a[u] = (ok && j < M) ? AB[n * 2 * M + j] : 0.0;
            b[u] = (ok && j < M) ? AB[n * 2 * M + M + j] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            accv += gv[u];
            acc = fma(gm[u], a[u], acc);
            amax = fmax(amax, fabs(abbar_value(gm[u], gv[u], mj, a[u], true)));
            bmax = fmax(bmax, fabs(abbar_value(gm[u], gv[u], mj, b[u], false)));
        }
    }
    if (j < M) {
        atomicAdd(dm + j, acc);
        atomicMax(col_exp + j, i8::exp_above(amax));
        atomicMax(col_exp + M + j, i8::exp_above(bmax));
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(dos, accv);
}

// pass 2: residue planes[t][n][j] of rint([Abar | Bbar][n,j] 2^(bits - c_j)); tile and thread layout of i8::k_to_residues
__global__ void __launch_bounds__(256) k_abbar_residues(const double* __restrict__ AB, long rows, int M, const double* __restrict__ g_mu,
                                                        const double* __restrict__ g_v, const double* __restrict__ m,
                                                        const int* __restrict__ col_exp, int bits, i8::CrtTable tab,
                                                        uint8_t* __restrict__ planes, long ldp, long plane_stride) {
    const long r = (long)blockIdx.y * i8::RS_TR + (threadIdx.x >> 3);
    const int c = blockIdx.x * i8::RS_TC + (threadIdx.x & 7) * 16;
    const int cols = 2 * M;
    const double gm = r < rows ? g_mu[r] : 0.0, gv = r < rows ? g_v[r] : 0.0;
    double ab[16];
    if (r < rows && c + 16 <= cols && ((reinterpret_cast<uintptr_t>(AB + r * cols + c) & 15) == 0)) {
        const double2* src = reinterpret_cast<const double2*>(AB + r * cols + c);
#pragma unroll
        for (int i = 0; i < 8; ++i) { const double2 t = src[i]; ab[2 * i] = t.x; ab[2 * i + 1] = t.y; }
    } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) ab[i] = (r < rows && c + i < cols) ? AB[r * cols + c + i] : 0.0;
    }
    long long xi[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const int j = c + i;
        double x = 0.0;
        int e = 0;
        if (r < rows && j < cols) {
            x = abbar_value(gm, gv, j < M ? m[j] : 0.0, ab[i], j < M);
            e = col_exp[j];
        }
        xi[i] = __double2ll_rn(i8::mul_pow2(x, bits - e));
    }
    i8::emit_residues_rt(tab.T, xi, tab, r, rows, c, cols, planes, ldp, plane_stride);
}

// W~ = diag(2^c) W (2M x M): exponent above each column maximum (pre-set to a very small value) ...
__global__ void __launch_bounds__(256) k_wt_colexp(const double* __restrict__ W, int rows, int M, const int* __restrict__ row_shift,
                                                   int* __restrict__ wc_exp) {
    const int k = blockIdx.x * 256 + threadIdx.x;
    const int j0 = blockIdx.y * 64, j1 = min(j0 + 64, rows);
    if (k >= M) return;
    int e = -200000;
    for (int j = j0; j < j1; ++j) e = max(e, row_shift[j] + i8::exp_above(W[(long)j * M + k]));
    atomicMax(wc_exp + k, e);
}

// ... and its residue planes[t][j][k] of rint(W[j,k] 2^(c_j + bits - e_k)): the backward-data operand, read MN-major
__global__ void __launch_bounds__(256) k_wt_residues(const double* __restrict__ W, long rows, int M, const int* __restrict__ row_shift,
                                                     const int* __restrict__ wc_exp, int bits, i8::CrtTable tab,
                                                     uint8_t* __restrict__ planes, long ldp, long plane_stride) {
    const long r = (long)blockIdx.y * i8::RS_TR + (threadIdx.x >> 3);
    const int c = blockIdx.x * i8::RS_TC + (threadIdx.x & 7) * 16;
    const int sh = r < rows ? row_shift[r] + bits : 0;
    long long xi[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const bool in = r < rows && c + i < M;
        xi[i] = in ? __double2ll_rn(i8::mul_pow2(W[r * M + c + i], sh - wc_exp[c + i])) : 0ll;
    }
    i8::emit_residues_rt(tab.T, xi, tab, r, rows, c, M, planes, ldp, plane_stride);
}

template <int KIND>
inline int qf_forward_k(const StepView& s, const StepPlanes& sp, const BatchView& b, const double* X, long R, double* mu, double* v,
                        cudaStream_t st) {
    const int M = s.M, D = s.D;
    const int Tf = fwd_T(M), bits = fwd_bits_w(M);
    // K_xz residue planes of all rows in one launch.  It depends on Zs / ls / os only, not on the factorisation:
    // it is enqueued BEFORE the join with the factorisation, which may still be running on the library's high-priority stream
    // (TGP_OPT_OVERLAP_KGEN, common.cuh), and runs under it.  K residues: one scale for the whole matrix (0 <= k <= outputscale),
    // shared by the forward and the weight contraction.
    {
        const int rr = rbf_residues<KIND>(X, s.Zs, s.ls, s.os, R, M, D, T_ALL, b.Kp, b.ldk, R * b.ldk, st);
        if (rr != 0 && rr != -7) return rr;
        if (join_factor(st)) return set_error(-100, "join with the factorisation failed");
        if (rr == -7) {
            TGP_TRY(launch_rbf<KIND>(X, s.Zs, s.ls, s.os, (int)R, M, D, 0, b.Kbuf, M, (int)R, M, 0.0, st));
            TGP_TRY(to_residues(b.Kbuf, M, R, M, 2, sp.k_exp, 53, T_ALL, b.Kp, b.ldk, R * b.ldk, st));
        }
    }
    for (long r0 = 0; r0 < R; r0 += b.Rc) {
        const int rc = (int)((R - r0) < b.Rc ? (R - r0) : b.Rc);
        i8::Params p{};
        p.Mrows = rc; p.Ncols = 2 * M; p.K = M; p.T = Tf; p.tri_mode = 1; p.tri_rows = M; p.lower_rows = 0; p.mn_major = 0;
        p.C = b.Op; p.ldc = b.ld2m; p.plane_stride_c = (long)b.Rc * b.ld2m;
        Planes A{b.Kp + r0 * b.ldk, rc, M, b.ldk, R * b.ldk};
        Planes B{sp.W, 2L * M, M, sp.ldk, 2L * M * sp.ldk};
        TGP_TRY(i8::gemm_i8_mod(A, B, p, st));
        TGP_TRY(combine(b.Op, b.ld2m, (long)b.Rc * b.ld2m, rc, 2 * M, Tf, 53 + bits, sp.k_exp, 2, sp.w_row_exp, 1, b.AB + r0 * 2 * M,
                        2L * M, 0, 0, st, i8::RowStats{s.mvec, s.os, mu + r0, v + r0, M}));
    }
    return 0;
}

inline int qf_forward(const StepView& s, const StepPlanes& sp, const BatchView& b, const double* X, long R, double* mu, double* v,
                      cudaStream_t st) {
    return with_kernel(s.kind, [&](auto k) { return qf_forward_k<decltype(k)::value>(s, sp, b, X, R, mu, v, st); });
}

template <int KIND>
inline int qf_backward_k(const StepView& s, const StepPlanes& sp, const BatchView& b, const double* X, long R, const double* g_mu,
                         const double* g_v, double* dm, double* dos, double* dZ, double* dls, double* Gbar, double* Cbar, double* dX,
                         cudaStream_t st) {
    const int M = s.M, D = s.D;
    TGP_TRY(fill_int(b.zero_exp, 1, 0, st));
    // NULL for D <= 32: k_kernel_grads recomputes the K_xz tile (same arithmetic); only the RBF reads it for D > 32
    const double* const kval = b.Kbuf;
    for (long r0 = 0; r0 < R; r0 += b.Rc) {
        const int rc = (int)((R - r0) < b.Rc ? (R - r0) : b.Rc);
        const double* ABc = b.AB + r0 * 2 * M;
        // [Abar | Bbar] of the chunk: column exponents (+ dm, doutputscale), then ONE set of residue planes scaled per column
        const int Tw = T_ALL, bits_x = wgt_bits(rc);
        const int Tb = bwd_T(M, bits_x), bits_w = bwd_bits_w(M, bits_x);
        {
            TGP_TRY(fill_int(b.col_exp, 2L * M, -100000, st));
            dim3 grid((unsigned)cdiv(M, 128), (unsigned)cdiv(rc, ABS_ROWS));
            k_abbar_stats<<<grid, 128, 0, st>>>(ABc, g_mu + r0, g_v + r0, s.mvec, rc, M, dm, dos, b.col_exp);
            TGP_TRY(check_launch("k_abbar_stats"));
            dim3 rgrid((unsigned)cdiv(2L * M, i8::RS_TC), (unsigned)cdiv(rc, i8::RS_TR));
            k_abbar_residues<<<rgrid, 256, 0, st>>>(ABc, rc, M, g_mu + r0, g_v + r0, s.mvec, b.col_exp, bits_x, i8::crt_table(Tw), b.Pc,
                                                    b.ld2m, (long)b.Rc * b.ld2m);
            TGP_TRY(check_launch("k_abbar_residues"));
        }
        {   // W~ = diag(2^c) W for this chunk's column exponents: per-column scale e_k, planes read MN-major by the tensor core
            TGP_TRY(fill_int(b.wc_exp, M, -200000, st));
            dim3 egrid((unsigned)cdiv(M, 256), (unsigned)cdiv(2L * M, 64));
            k_wt_colexp<<<egrid, 256, 0, st>>>(sp.Wst, 2 * M, M, b.col_exp, b.wc_exp);
            TGP_TRY(check_launch("k_wt_colexp"));
            dim3 rgrid((unsigned)cdiv(M, i8::RS_TC), (unsigned)cdiv(2L * M, i8::RS_TR));
            k_wt_residues<<<rgrid, 256, 0, st>>>(sp.Wst, 2L * M, M, b.col_exp, b.wc_exp, bits_w, i8::crt_table(Tb), sp.Wc, sp.ldk,
                                                 2L * M * sp.ldk);
            TGP_TRY(check_launch("k_wt_residues"));
        }
        {   // Kbar (rc x M) = ABbar (rc x 2M) * W~ (2M x M); for k < M only k >= n contributes.  A is K-major (the first Tb of the
            // Tw planes: the moduli of a shorter table are a prefix); the reduction runs over the ROWS of W~ (mn_major bit 1)
            i8::Params p{};
            p.Mrows = rc; p.Ncols = M; p.K = 2 * M; p.T = Tb; p.tri_mode = 2; p.tri_rows = M; p.lower_rows = 0; p.mn_major = 2;
            p.C = b.Kbp; p.ldc = b.ldk; p.plane_stride_c = (long)b.Rc * b.ldk;
            Planes A{b.Pc, rc, 2L * M, b.ld2m, (long)b.Rc * b.ld2m};
            Planes B{sp.Wc, 2L * M, M, sp.ldk, 2L * M * sp.ldk};
            TGP_TRY(i8::gemm_i8_mod(A, B, p, st));
        }
        // reconstruction of Kbar, then Kbar o K -> dZ, dlengthscale, doutputscale
        TGP_TRY(combine(b.Kbp, b.ldk, (long)b.Rc * b.ldk, rc, M, Tb, bits_x + bits_w, b.zero_exp, 2, b.wc_exp, 1, b.Kbar, M, 0, 0, st));
        TGP_TRY(launch_kernel_grads<KIND>(b.Kbar, M, X + r0 * D, 0, s.Zs, s.ls, s.os, rc, M, D, 0, 1.0, dZ, dls, dos, st, kval ? kval + r0 * M : nullptr, M));
        if (dX) TGP_TRY(launch_input_grads<KIND>(b.Kbar, M, X + r0 * D, s.Zs, s.ls, s.os, rc, M, D, dX + r0 * D, st));
        {   // [Gbar; Cbar] (2M x M) += ABbar^T K: reduction over the chunk rows; both operands are row-major planes read MN-major
            i8::Params p{};
            p.Mrows = 2 * M; p.Ncols = M; p.K = rc; p.T = Tw; p.tri_mode = 0; p.tri_rows = 0; p.lower_rows = M; p.mn_major = 3;
            p.C = b.Gp; p.ldc = b.ldk; p.plane_stride_c = 2L * M * b.ldk;
            Planes A{b.Pc, rc, 2L * M, b.ld2m, (long)b.Rc * b.ld2m};
            Planes B{b.Kp + r0 * b.ldk, rc, M, b.ldk, R * b.ldk};
            TGP_TRY(i8::gemm_i8_mod(A, B, p, st));
            // K residues carry 53 bits, ABbar (per column) bits_x
            TGP_TRY(combine(b.Gp, b.ldk, 2L * M * b.ldk, M, M, Tw, bits_x + 53, b.col_exp, 0, sp.k_exp, 2, Gbar, s.Mp, 1, M, st));
            TGP_TRY(combine(b.Gp + (long)M * b.ldk, b.ldk, 2L * M * b.ldk, M, M, Tw, bits_x + 53, b.col_exp + M, 0, sp.k_exp, 2, Cbar,
                            s.Mp, 1, 0, st));
        }
    }
    return 0;
}

inline int qf_backward(const StepView& s, const StepPlanes& sp, const BatchView& b, const double* X, long R, const double* g_mu,
                       const double* g_v, double* dm, double* dos, double* dZ, double* dls, double* Gbar, double* Cbar, double* dX,
                       cudaStream_t st) {
    return with_kernel(s.kind, [&](auto k) {
        return qf_backward_k<decltype(k)::value>(s, sp, b, X, R, g_mu, g_v, dm, dos, dZ, dls, Gbar, Cbar, dX, st);
    });
}

// ---- test hook: C = A B^T through the residue pipeline ------------------------------------------------------------------
// mn_major bit 0 / 1: A / B is passed TRANSPOSED ((K x Mr) / (K x N), row-major) and contracted over its rows.  The scratch
// holds the operand planes of either orientation: its size does not depend on mn_major.
struct DebugScratch { uint8_t *Ap, *Bp, *Cp; int *ea, *eb; };
inline DebugScratch debug_scratch(Carve& c, long Mr, long N, long K, int T) {
    const long ldk = pad16(K), ldn = pad16(N), ldm = pad16(Mr);
    DebugScratch d;
    d.Ap = c.take<uint8_t>((size_t)T * (K * ldm > Mr * ldk ? K * ldm : Mr * ldk));
    d.Bp = c.take<uint8_t>((size_t)T * (K * ldn > N * ldk ? K * ldn : N * ldk));
    d.Cp = c.take<uint8_t>((size_t)T * Mr * ldn);
    d.ea = c.take<int>(Mr);
    d.eb = c.take<int>(N);
    return d;
}

inline int debug_matmul(long Mr, long N, long K, const double* A, long lda, const double* B, long ldb, double* C, long ldc, int T,
                        int tri_mode, int tri_rows, int lower_rows, int accumulate, int mn_major, void* scratch, cudaStream_t st) {
    const long ldk = pad16(K), ldn = pad16(N), ldm = pad16(Mr);
    const bool at = mn_major & 1, bt = mn_major & 2;
    Carve c(scratch);
    const DebugScratch d = debug_scratch(c, Mr, N, K, T);
    const int bits = i8::crt_bits(T, K);
    if (at) {
        TGP_TRY(exponents(A, lda, K, (int)Mr, nullptr, d.ea, st));
        TGP_TRY(to_residues(A, lda, K, (int)Mr, 1, d.ea, bits, T, d.Ap, ldm, K * ldm, st));
    } else {
        TGP_TRY(exponents(A, lda, Mr, (int)K, d.ea, nullptr, st));
        TGP_TRY(to_residues(A, lda, Mr, (int)K, 0, d.ea, bits, T, d.Ap, ldk, Mr * ldk, st));
    }
    if (bt) {
        TGP_TRY(exponents(B, ldb, K, (int)N, nullptr, d.eb, st));
        TGP_TRY(to_residues(B, ldb, K, (int)N, 1, d.eb, bits, T, d.Bp, ldn, K * ldn, st));
    } else {
        TGP_TRY(exponents(B, ldb, N, (int)K, d.eb, nullptr, st));
        TGP_TRY(to_residues(B, ldb, N, (int)K, 0, d.eb, bits, T, d.Bp, ldk, N * ldk, st));
    }
    i8::Params q{};
    q.Mrows = (int)Mr; q.Ncols = (int)N; q.K = (int)K; q.T = T; q.tri_mode = tri_mode; q.tri_rows = tri_rows; q.lower_rows = lower_rows;
    q.mn_major = mn_major;
    q.C = d.Cp; q.ldc = ldn; q.plane_stride_c = Mr * ldn;
    const Planes PA = at ? Planes{d.Ap, K, Mr, ldm, K * ldm} : Planes{d.Ap, Mr, K, ldk, Mr * ldk};
    const Planes PB = bt ? Planes{d.Bp, K, N, ldn, K * ldn} : Planes{d.Bp, N, K, ldk, N * ldk};
    TGP_TRY(i8::gemm_i8_mod(PA, PB, q, st));
    return combine(d.Cp, ldn, Mr * ldn, Mr, (int)N, T, 2 * bits, d.ea, 0, d.eb, 1, C, ldc, accumulate, lower_rows, st);
}

}  // namespace crt
}  // namespace tgp
