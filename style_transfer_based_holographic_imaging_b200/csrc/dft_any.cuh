// dft_any.cuh -- every field size that is NOT a power of two (the reference accepts any square N unpadded and any even
// square N with zero_padding=True, utils/Angular_Spectrum_Method.py:11-23; its own loader produces 92 x 92 fields,
// utils/Data_loader.py:24).
//
// The propagation is four matrix products with two precomputed matrices that carry the padding, the crop and the fold:
//   analysis  A[xs][u]  (N x M):  forward  sum over the padded positions x that replicate source pixel xs of W_M^{x u}
//                                 adjoint  W_M^{(xs + P) u}                              (zero embedding)
//   synthesis S[u][xo]  (M x N):  forward  conj(W_M)^{u (xo + P)} / M                    (crop)
//                                 adjoint  sum over the padded positions folded onto xo of conj(W_M)^{u x} / M
//   T1 = In A            [N x M]      rows
//   T2 = H . (A^T T1)    [M x M]      columns + transfer function  (H(u, v) evaluated in fp64, no table)
//   T3 = S^T T2          [N x M]      columns back
//   Out = T3 S           [N x N]      rows back + output stage
// (W_M = exp(-2 pi i / M); unpadded: P = 0, A and S are the plain DFT matrices.)  This is a completeness path: O(N^3)
// per sample on the FP32 pipe, meant for the small odd sizes of the MNIST loaders, accepted up to FFT size 2048.
#pragma once

namespace asmb {

constexpr int DFT_MAX_M = 2048;
constexpr int DFT_T = 32, DFT_K = 16;        // output tile 32 x 32, K step 16, 256 threads

struct DftGeom {
    int N, M, P, chunk;
    size_t a_bytes, s_bytes, t1_bytes, t2_bytes, t3_bytes;   // per-call matrices, per-chunk intermediates
};

static bool dft_geometry(int planes, int N, int pad, DftGeom* g) {
    if (planes <= 0 || N < 2 || (N & (N - 1)) == 0) return false;              // powers of two take the FFT kernels
    if ((N & 1) && pad) return false;                                          // the reference's replicate padding needs an even N (ASM.py:12-14)
    const int M = pad ? 2 * N : N;
    if (M > DFT_MAX_M) return false;
    g->N = N; g->M = M; g->P = (M - N) / 2;
    const size_t per = ((size_t)2 * N * M + (size_t)M * M) * sizeof(float2);
    size_t c = ((size_t)96 << 20) / per;
    if (c < 1) c = 1;
    if (c > (size_t)planes) c = planes;
    g->chunk = (int)c;
    auto al = [](size_t x) { return (x + 255) / 256 * 256; };
    g->a_bytes = al((size_t)N * M * sizeof(float2)); g->s_bytes = al((size_t)M * N * sizeof(float2));
    g->t1_bytes = al(c * N * M * sizeof(float2)); g->t2_bytes = al(c * M * M * sizeof(float2)); g->t3_bytes = al(c * N * M * sizeof(float2));
    return true;
}
static size_t dft_workspace(const DftGeom& g) { return g.a_bytes + g.s_bytes + g.t1_bytes + g.t2_bytes + g.t3_bytes; }

// e^{-+ 2 pi i (a b mod M) / M} in double
__device__ __forceinline__ void dft_w(int a, int b, int M, double sign, double* re, double* im) {
    const long long k = ((long long)a * b) % M;
    double s, c;
    sincospi(2.0 * (double)k / (double)M, &s, &c);
    *re = c; *im = sign * s;
}

__global__ void k_dft_setup(float2* A, float2* S, int N, int M, int P, int adj) {
    const int total = N * M;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        {   // A[xs][u]
            const int xs = idx / M, u = idx % M;
            double re = 0.0, im = 0.0;
            int lo = xs + P, hi = xs + P;
            if (!adj && P > 0) { if (xs == 0) lo = 0; if (xs == N - 1) hi = M - 1; }
            for (int x = lo; x <= hi; ++x) { double r, i; dft_w(x, u, M, -1.0, &r, &i); re += r; im += i; }
            A[idx] = make_float2((float)re, (float)im);
        }
        {   // S[u][xo]
            const int u = idx / N, xo = idx % N;
            double re = 0.0, im = 0.0;
            int lo = xo + P, hi = xo + P;
            if (adj && P > 0) { if (xo == 0) lo = 0; if (xo == N - 1) hi = M - 1; }
            for (int x = lo; x <= hi; ++x) { double r, i; dft_w(x, u, M, 1.0, &r, &i); re += r; im += i; }
            S[idx] = make_float2((float)(re / M), (float)(im / M));
        }
    }
}

__device__ __forceinline__ float2 dft_load_any(const Params& p, size_t idx) {
    switch (p.in_mode) {
        case ASM_B200_IN_COMPLEX: return load_one<ASM_B200_IN_COMPLEX>(p, idx);
        case ASM_B200_IN_AMP_PHASE: return load_one<ASM_B200_IN_AMP_PHASE>(p, idx);
        case ASM_B200_IN_CONST_AMP_PHASE: return load_one<ASM_B200_IN_CONST_AMP_PHASE>(p, idx);
        case ASM_B200_IN_SQRT_REAL: return load_one<ASM_B200_IN_SQRT_REAL>(p, idx);
        case ASM_B200_IN_COT_FIELD: return load_one<ASM_B200_IN_COT_FIELD>(p, idx);
        default: return load_one<ASM_B200_IN_REAL>(p, idx);
    }
}
__device__ __forceinline__ float dft_emit_any(const Params& p, int plane, int y, int x, float2 u) {
    switch (p.out_mode) {
        case ASM_B200_OUT_COMPLEX: return emit_one<ASM_B200_OUT_COMPLEX>(p, plane, y, x, u);
        case ASM_B200_OUT_INTENSITY: return emit_one<ASM_B200_OUT_INTENSITY>(p, plane, y, x, u);
        case ASM_B200_OUT_ABS_ANGLE: return emit_one<ASM_B200_OUT_ABS_ANGLE>(p, plane, y, x, u);
        case ASM_B200_OUT_REIM_CAT: return emit_one<ASM_B200_OUT_REIM_CAT>(p, plane, y, x, u);
        case ASM_B200_OUT_ABSANG_CAT: return emit_one<ASM_B200_OUT_ABSANG_CAT>(p, plane, y, x, u);
        case ASM_B200_OUT_GRAD_AP: return emit_one<ASM_B200_OUT_GRAD_AP>(p, plane, y, x, u);
        default: return emit_one<OUT_DOT>(p, plane, y, x, u);
    }
}

// transfer function at bin (u, v), fp64 phase (same arithmetic as the kappa tables: ASM.py:16-29 on unshifted bins)
__device__ __forceinline__ float2 dft_h(const Params& p, int u, int v, int M, double cph) {
    const int ku = u < (M + 1) / 2 ? u : u - M, kv = v < (M + 1) / 2 ? v : v - M;
    const double arg = fma(-p.s2, (double)ku * ku + (double)kv * kv, 1.0);
    const double root = arg > 0.0 ? sqrt(arg) : 0.0;                 // kz lambda; evanescent -> 0 (H = 1)
    double t = root * p.inv_lambda * 0.15915494309189535 * cph;      // turns
    t -= rint(t);
    float sn, cs;
    sincospif((float)(2.0 * t), &sn, &cs);
    if (p.h_mode == H_DERIV) { const float f = (float)(root - p.kshift); return make_float2(-sn * f, cs * f); }
    return make_float2(cs, sn);
}

// Out[b][r][c] = sum_k L(b, r, k) R(b, k, c):  KIND 0: In A;  1: H . A^T T1;  2: S^T T2;  3: T3 S -> output stage
template <int KIND>
__global__ void __launch_bounds__(256) k_dft_mm(const Params p, const float2* __restrict__ A, const float2* __restrict__ S,
                                                 float2* __restrict__ T1, float2* __restrict__ T2, float2* __restrict__ T3,
                                                 int plane0, int N, int M) {
    __shared__ float2 Ls[DFT_T][DFT_K + 1];
    __shared__ float2 Rs[DFT_K][DFT_T + 1];
    __shared__ float red[8];
    const int img = blockIdx.z, plane = plane0 + img;
    const int R_ = (KIND == 1) ? M : N, C_ = (KIND == 3) ? N : M, K_ = (KIND == 0 || KIND == 1) ? N : M;
    const int r0 = blockIdx.y * DFT_T, c0 = blockIdx.x * DFT_T;
    const int t = threadIdx.x, tx = t % DFT_T, ty = t / DFT_T;      // outputs (r0 + ty + 8 i, c0 + tx), i < 4
    float2 acc[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[i] = make_float2(0.f, 0.f);
    for (int k0 = 0; k0 < K_; k0 += DFT_K) {
        for (int e = t; e < DFT_T * DFT_K; e += 256) {               // left tile [r][k]
            const int rr = e / DFT_K, kk = e % DFT_K, r = r0 + rr, k = k0 + kk;
            float2 val = make_float2(0.f, 0.f);
            if (r < R_ && k < K_) {
                if (KIND == 0) val = dft_load_any(p, ((size_t)(p.kst ? plane / p.kst : plane) * N + r) * N + k);
                else if (KIND == 1) val = A[(size_t)k * M + r];
                else if (KIND == 2) val = S[(size_t)k * N + r];
                else val = T3[((size_t)img * N + r) * M + k];
            }
            Ls[rr][kk] = val;
        }
        for (int e = t; e < DFT_K * DFT_T; e += 256) {               // right tile [k][c]
            const int kk = e / DFT_T, cc = e % DFT_T, k = k0 + kk, c = c0 + cc;
            float2 val = make_float2(0.f, 0.f);
            if (k < K_ && c < C_) {
                if (KIND == 0) val = A[(size_t)k * M + c];
                else if (KIND == 1) val = T1[((size_t)img * N + k) * M + c];
                else if (KIND == 2) val = T2[((size_t)img * M + k) * M + c];
                else val = S[(size_t)k * N + c];
            }
            Rs[kk][cc] = val;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < DFT_K; ++kk) {
            const float2 b = Rs[kk][tx];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float2 a = Ls[ty + 8 * i][kk];
                acc[i].x = fmaf(a.x, b.x, fmaf(-a.y, b.y, acc[i].x));
                acc[i].y = fmaf(a.x, b.y, fmaf(a.y, b.x, acc[i].y));
            }
        }
        __syncthreads();
    }
    float dot = 0.f;
    const int c = c0 + tx;
    double cph = 0.0;
    if (KIND == 1) cph = phase_constant_of(p, plane / p.C);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = r0 + ty + 8 * i;
        if (r >= R_ || c >= C_) continue;
        if (KIND == 0) T1[((size_t)img * N + r) * M + c] = acc[i];
        else if (KIND == 1) {
            const float2 h = dft_h(p, c, r, M, cph);                 // column index = row-pass frequency u, row index = v
            T2[((size_t)img * M + r) * M + c] = make_float2(acc[i].x * h.x - acc[i].y * h.y, acc[i].x * h.y + acc[i].y * h.x);
        } else if (KIND == 2) T3[((size_t)img * N + r) * M + c] = acc[i];
        else if (p.out0) dot += dft_emit_any(p, plane, r, c, acc[i]);
    }
    if (KIND == 3 && p.part) {                                       // focal-stack moments: one partial per tile, fixed order
        float m[3] = {0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (r0 + ty + 8 * i < N && c < N) mom_add(m, acc[i]);
        double d[3];
        mom_reduce<32>(d, m);
        __shared__ double mred[8][3];
        if ((t & 31) == 0) { mred[t >> 5][0] = d[0]; mred[t >> 5][1] = d[1]; mred[t >> 5][2] = d[2]; }
        __syncthreads();
        if (t < 3) {
            double s = 0.0;
            for (int w = 0; w < 8; ++w) s += mred[w][t];
            p.part[(((size_t)img * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 3 + t] = s;
        }
    }
    if (KIND == 3 && p.out_mode == OUT_DOT) {                        // uniform branch: reduce the block, one atomic
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
        if ((t & 31) == 0) red[t >> 5] = dot;
        __syncthreads();
        if (t == 0) {
            float s = 0.f;
            for (int i = 0; i < 8; ++i) s += red[i];
            const double K = p.z_f64 ? 6.283185307179586 : (double)6.2831854820251465f;
            atomicAdd((double*)p.out0 + plane / p.C, (double)s * K * p.inv_lambda);
        }
    }
}

}  // namespace asmb
