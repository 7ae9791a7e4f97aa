// asm_b200.cu -- B200 (sm_100a) angular-spectrum propagator: kernels + C ABI (include/asm_b200.h).
//
// Pipeline per chunk of samples (the chunk's intermediate lives in an L2-resident workspace):
//   rows_fwd : source rows (HBM, read once; input construction + replicate/zero padding fused) -> row FFT -> ws
//   cols     : TMA column slab ws -> smem; column FFT . H(z) (generated on the fly) . column IFFT; TMA -> ws
//   rows_inv : ws -> row IFFT -> crop/fold + output stage fused -> HBM (written once)
// Reference semantics: utils/Angular_Spectrum_Method.py:7-53, utils/Forward_model.py:16-65 (see DESIGN.md).
#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <mutex>

#include "../../include/asm_b200.h"
#include "fft_core.cuh"

namespace asmb {

// internal output mode: reduce Re(conj(g) * D) per sample (grad_z)
constexpr int OUT_DOT = 6;
constexpr int H_FWD = 0, H_CONJ = 1, H_DERIV = 2;

struct Params {
    const void* in0; const void* in1;     // input field (see in_mode)
    const void* aux0; const void* aux1;   // amplitude/phase (OUT_GRAD_AP) or cotangent (OUT_DOT)
    void* out0; void* out1;
    const void* z;
    float2* ws;                           // chunk intermediate: [chunk_imgs][N rows][M] complex64, swizzled/digit-reversed cols
    const float2* tw;                     // twiddle tables (global)
    const float2* tw32;                   // FFT 2048: half twiddle table of the 1024-point transform (k64.cuh)
    const double* kzt;                    // kappa table [M/2+1][M] (global), or nullptr
    double s2;                            // (lambda / (M px))^2
    double inv_lambda;                    // 1 / lambda
    double lambda;
    double kshift;                        // H_DERIV: the filter is i (kz - kshift / lambda) H (see asm_b200_grad_z)
    double S;                             // M px: the window of the FFT grid (band limit)
    float in_scale, out_scale, inv_m2;
    int planes, C, N, M, P;               // planes = B*C
    int in_mode, out_mode, aux_mode, h_mode, adj, z_f64;
    int band_limit;                       // 1: zero the bins outside the band limit of each plane's z (band_limit_of)
    // focal stack (asm_b200_focal_stack): planes are (sample, distance) pairs q = b kst + k.  The column pass reads the
    // spectrum of sample q / kst from src (slot q / kst - s0) and writes plane q to ws; kst = 0 outside a stack.
    const float2* src;
    int kst, s0;
    double* part;                         // per-row moment partials (Sum |U|, |U|^2, |U|^4) of the planes in ws, or nullptr
};

// slot of the column pass's source image: in place outside a focal stack, the sample's spectrum inside one
__device__ __forceinline__ int src_slot(const Params& p, int plane0, int img) { return p.kst ? (plane0 + img) / p.kst - p.s0 : img; }
__device__ __forceinline__ const float2* src_base(const Params& p) { return p.kst ? p.src : p.ws; }

// Sum |u|, |u|^2, |u|^4 of one value (fp32), accumulated per thread before the row reduction in double
__device__ __forceinline__ void mom_add(float (&m)[3], float2 u) {
    const float i2 = fmaf(u.x, u.x, u.y * u.y);
    m[0] += sqrtf(i2); m[1] += i2; m[2] = fmaf(i2, i2, m[2]);
}
// xor-shuffle sum in double over `width` consecutive lanes (a fixed order: repeated calls give identical bits)
template <int W>
__device__ __forceinline__ void mom_reduce(double (&d)[3], const float (&m)[3]) {
#pragma unroll
    for (int j = 0; j < 3; ++j) d[j] = (double)m[j];
#pragma unroll
    for (int o = 1; o < W; o <<= 1) {
#pragma unroll
        for (int j = 0; j < 3; ++j) d[j] += __shfl_xor_sync(0xffffffffu, d[j], o);
    }
}

// moments[plane0 + i] = Sum of the R row partials of plane i, in index order (one warp per plane)
__global__ void k_moments_reduce(const double* __restrict__ part, double* __restrict__ mom, int R, int nimg, int plane0) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= nimg) return;
    double d[3] = {0.0, 0.0, 0.0};
    const double* src = part + (size_t)w * R * 3;
    for (int r = lane; r < R; r += 32) {
#pragma unroll
        for (int j = 0; j < 3; ++j) d[j] += src[(size_t)r * 3 + j];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int j = 0; j < 3; ++j) d[j] += __shfl_xor_sync(0xffffffffu, d[j], o);
    }
    if (lane == 0) {
#pragma unroll
        for (int j = 0; j < 3; ++j) mom[(size_t)(plane0 + w) * 3 + j] = d[j];
    }
}

// phase constant c of a sample (ASM.py:29): fl32(fl32(2 pi) z) for fp32 distances, 2 pi z in double otherwise
__device__ __forceinline__ double phase_constant_of(const Params& p, int b) {
    double cph;
    if (p.z_f64) cph = 6.283185307179586 * __ldg((const double*)p.z + b);
    else cph = (double)__fmul_rn(6.2831854820251465f, __ldg((const float*)p.z + b));
    return p.h_mode == H_CONJ ? -cph : cph;
}

// Band limit of a sample (Matsushima & Shimobaba, Opt. Express 17, 19662, 2009): bin (u, v) is kept iff |k(u)| <= lim
// and |k(v)| <= lim, lim = floor(S / (lambda sqrt(1 + q^2))), q = 2 z / S, S = M px, in double in exactly this order
// (no contraction), clamped to M before the conversion (S / lambda may exceed INT_MAX; a NaN z keeps every bin).
// Without the band limit every bin is kept (lim = M > M / 2).  The only statement of the rule on the device.
__device__ __forceinline__ int band_limit_of(const Params& p, int b) {
    if (!p.band_limit) return p.M;
    const double z = p.z_f64 ? __ldg((const double*)p.z + b) : (double)__ldg((const float*)p.z + b);
    const double q = __ddiv_rn(__dmul_rn(2.0, z), p.S);
    const double t = __ddiv_rn(p.S, __dmul_rn(p.lambda, __dsqrt_rn(__dadd_rn(1.0, __dmul_rn(q, q)))));
    return (int)fmin(floor(t), (double)p.M);
}

// ---------------------------------------------------------------------------------------------------
// small PTX wrappers (mbarrier + TMA tensor copies)
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int x, int y, int z) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(x), "r"(y), "r"(z) : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* src, int x, int y, int z) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"(map), "r"(smem_u32(src)), "r"(x), "r"(y), "r"(z) : "memory");
}
__device__ __forceinline__ void tma_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------------
// tables (rebuilt by every call into the caller's workspace; stream-ordered, a few microseconds)
//   twiddles : entry (e, j) of a segment with stride S is W_{S 2^m}^{Q + S u}, e = 2^{m-1} - 1 + u.
//              forward segments are indexed by the thread's position bits j = hi (Q = fwd_q(hi)),
//              inverse segments by j = Q directly -> consecutive threads read consecutive entries.
//   kz       : kappa[ru][c] = kz(|ku| = ru, kv(c)) / (2 pi) in double, ru = 0..M/2, c = workspace column
//              (digit-reversed row-pass frequency).  theta / 2pi = c_phase * kappa.
// ---------------------------------------------------------------------------------------------------
__global__ void k_setup_tables(float2* tw, double* kzt, int n, double s2, double inv_2pi_lambda) {
    const TwLayout lay = make_layout(n);
    const int a = n % 4, nf = n / 4, r = 1 << a, M = 1 << n;
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    for (int e = gtid; e < lay.total; e += gsz) {
        int off = -1, S = 1, ff = 0;
        bool inv = false;
        for (int f = 0; f < nf; ++f) {
            const int Sf = r * ipow16(nf - 1 - f);
            if (lay.fwd[f] >= 0 && e >= lay.fwd[f] && e < lay.fwd[f] + 15 * Sf) { off = lay.fwd[f]; S = Sf; ff = f; }
            const int Si = ipow16(f);
            if (lay.inv[f] >= 0 && e >= lay.inv[f] && e < lay.inv[f] + 15 * Si) { off = lay.inv[f]; S = Si; inv = true; }
        }
        if (lay.invA >= 0 && e >= lay.invA) { off = lay.invA; S = M / r; inv = true; }
        const int idx = e - off;
        const int ent = idx / S, j = idx % S;
        const int Q = inv ? j : fwd_q_from_hi(n, ff, j);
        int m = 1;
        while ((1 << m) - 1 <= ent) ++m;           // ent in [2^{m-1}-1, 2^m-1)
        const int u = ent - ((1 << (m - 1)) - 1);
        const int D = S << m;
        const int x = Q + S * u;
        float sn, cs;
        sincospif(2.0f * (float)x / (float)D, &sn, &cs);   // x/D exact in fp32 (D is a power of two <= 2^13)
        tw[e] = make_float2(cs, inv ? sn : -sn);
    }
    if (kzt) {
        const int rows = M / 2 + 1;
        for (int idx = gtid; idx < rows * M; idx += gsz) {
            const int ru = idx / M, c = idx % M;
            const int v = freq_of_pos(n, c);
            const int kv = v < M / 2 ? v : v - M;
            const double kk = (double)ru * ru + (double)kv * kv;
            const double arg = fma(-s2, kk, 1.0);                      // 1 - lambda^2 (fx^2 + fy^2)
            kzt[idx] = (arg > 0.0 ? sqrt(arg) : 0.0) * inv_2pi_lambda; // evanescent -> kz = 0 (H = 1)
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// input construction / output stage (mode switch hoisted out of the unrolled loops)
// ---------------------------------------------------------------------------------------------------
__device__ __noinline__ float atan2_full(float y, float x) { return atan2f(y, x); }
// sin / cos of an input phase: three-term Cody-Waite reduction to [-pi, pi] (exact products for |x| < 5e4: the first
// two constants have 11 significant bits), then the MUFU approximations (absolute error < 5e-7 there).  Inputs beyond
// that range (or non-finite) take the library slow path.  Inlined: ~8 instructions instead of a call per pixel.
__device__ __noinline__ void sincos_slow(float x, float* s, float* c) { sincosf(x, s, c); }
__device__ __forceinline__ void sincos_reduced(float x, float* s, float* c) {
    if (fabsf(x) < 5.0e4f) {
        const float k = rintf(x * 0.15915494309189535f);
        float r = fmaf(-k, 6.28125f, x);
        r = fmaf(-k, 0.0019350051879882812f, r);
        r = fmaf(-k, 3.019916050561733e-07f, r);
        __sincosf(r, s, c);
    } else {
        sincos_slow(x, s, c);
    }
}

// Inputs and outputs are touched exactly once: streaming (evict-first) hints keep them from displacing the
// L2-resident intermediate.
template <int MODE>
__device__ __forceinline__ float2 load_one(const Params& p, size_t idx) {
    if constexpr (MODE == ASM_B200_IN_COMPLEX) return __ldcs((const float2*)p.in0 + idx);
    else if constexpr (MODE == ASM_B200_IN_AMP_PHASE) {
        const float a = __ldcs((const float*)p.in0 + idx);
        const float ph = __ldcs((const float*)p.in1 + idx) * p.in_scale;
        float sn, cs;
        sincos_reduced(ph, &sn, &cs);
        return make_float2(a * cs, a * sn);
    } else if constexpr (MODE == ASM_B200_IN_CONST_AMP_PHASE) {
        const float a = __ldg((const float*)p.in0);
        const float ph = __ldcs((const float*)p.in1 + idx) * p.in_scale;
        float sn, cs;
        sincos_reduced(ph, &sn, &cs);
        return make_float2(a * cs, a * sn);
    } else if constexpr (MODE == ASM_B200_IN_SQRT_REAL) return make_float2(sqrtf(__ldcs((const float*)p.in0 + idx)), 0.f);
    else if constexpr (MODE == ASM_B200_IN_COT_FIELD) {
        const float w = 2.f * __ldcs((const float*)p.in0 + idx);
        const float2 u = __ldcs((const float2*)p.in1 + idx);
        return make_float2(w * u.x, w * u.y);
    } else return make_float2(__ldcs((const float*)p.in0 + idx), 0.f);
}

// registers <- window n-4 of padded source row y (positions tl + TPL i), padding fused by index clamp / zero
template <int MODE, int TPL>
__device__ __forceinline__ void load16(float2 (&v)[16], const Params& p, int plane, int y, int tl) {
    const size_t row = ((size_t)plane * p.N + y) * p.N;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        int x = tl + TPL * i - p.P;
        if (p.adj) {
            v[i] = (x >= 0 && x < p.N) ? load_one<MODE>(p, row + x) : make_float2(0.f, 0.f);
        } else {
            x = min(max(x, 0), p.N - 1);
            v[i] = load_one<MODE>(p, row + x);
        }
    }
}

template <int MODE>
__device__ __forceinline__ float emit_one(const Params& p, int plane, int y, int x, float2 u) {
    const size_t idx = ((size_t)plane * p.N + y) * p.N + x;
    if constexpr (MODE == ASM_B200_OUT_COMPLEX) __stcs((float2*)p.out0 + idx, u);
    else if constexpr (MODE == ASM_B200_OUT_INTENSITY) {
        __stcs((float*)p.out0 + idx, fmaf(u.x, u.x, u.y * u.y));
        if (p.out1) __stcs((float2*)p.out1 + idx, u);
    } else if constexpr (MODE == ASM_B200_OUT_ABS_ANGLE) {
        ((float*)p.out0)[idx] = sqrtf(fmaf(u.x, u.x, u.y * u.y));
        ((float*)p.out1)[idx] = atan2_full(u.y, u.x);
    } else if constexpr (MODE == ASM_B200_OUT_REIM_CAT) {
        const size_t b = ((size_t)plane * 2 * p.N + y) * p.N + x;
        ((float*)p.out0)[b] = u.x * p.out_scale;
        ((float*)p.out0)[b + (size_t)p.N * p.N] = u.y * p.out_scale;
    } else if constexpr (MODE == ASM_B200_OUT_ABSANG_CAT) {
        const size_t b = ((size_t)plane * 2 * p.N + y) * p.N + x;
        const float re = u.x * p.out_scale, im = u.y * p.out_scale;
        ((float*)p.out0)[b] = sqrtf(fmaf(re, re, im * im));
        ((float*)p.out0)[b + (size_t)p.N * p.N] = atan2_full(im, re);
    } else if constexpr (MODE == ASM_B200_OUT_GRAD_AP) {
        const float a = __ldg((const float*)p.aux0 + idx);
        const float ph = __ldg((const float*)p.aux1 + idx) * p.in_scale;
        float sn, cs;
        sincos_reduced(ph, &sn, &cs);
        const float re = fmaf(cs, u.x, sn * u.y);    // conj(e) * u
        const float im = fmaf(cs, u.y, -sn * u.x);
        ((float*)p.out0)[idx] = re;
        ((float*)p.out1)[idx] = p.in_scale * a * im;
    } else {  // OUT_DOT
        float2 g;
        if (p.aux_mode == ASM_B200_IN_COT_FIELD) {
            const float w = 2.f * __ldg((const float*)p.aux0 + idx);
            const float2 f = __ldg((const float2*)p.aux1 + idx);
            g = make_float2(w * f.x, w * f.y);
        } else {
            g = __ldg((const float2*)p.aux0 + idx);
        }
        return fmaf(g.x, u.x, g.y * u.y);
    }
    return 0.f;
}

// registers hold window n-4 (positions tl + TPL i) of output row y; crop to [P, P+N) and emit.
// fl / fr: fold contributions added to columns 0 and N-1 (adjoint of replicate padding), zero otherwise.
template <int MODE, int TPL>
__device__ __forceinline__ float emit16(const float2 (&v)[16], const Params& p, int plane, int y, int tl, float2 fl, float2 fr) {
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const int x = tl + TPL * i - p.P;
        if (x >= 0 && x < p.N) {
            float2 u = v[i];
            if (x == 0) { u.x += fl.x; u.y += fl.y; }
            if (x == p.N - 1) { u.x += fr.x; u.y += fr.y; }
            dot += emit_one<MODE>(p, plane, y, x, u);
        }
    }
    return dot;
}

// ---------------------------------------------------------------------------------------------------
// row passes.  256 threads; a line of L points uses L/16 threads; LPC = 4096/L lines per tile;
// persistent CTAs loop over tiles so the twiddle tables are staged once per CTA.
// ---------------------------------------------------------------------------------------------------
#ifndef ASM_ROW_THREADS
#define ASM_ROW_THREADS 256
#endif
#ifndef ASM_CC10
#define ASM_CC10 8
#endif
constexpr int ROW_THREADS = ASM_ROW_THREADS;

template <int n>
__global__ void __launch_bounds__(ROW_THREADS, 1024 / ROW_THREADS) k_rows_fwd(const Params p, int plane0, int nlines, int ntiles) {
    constexpr int L = 1 << n, TPL = L / 16, LPC = ROW_THREADS / TPL, LP = RowLayout::line_elems(L);
    constexpr TwLayout lay = make_layout(n);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* lines = reinterpret_cast<float2*>(smem_raw);        // [LPC][LP]
    float2* tw = lines + LPC * LP;                              // forward tables [0, fwd_end)
    const int t = threadIdx.x, ll = t / TPL, tl = t % TPL;
    for (int i = t; i < lay.fwd_end; i += ROW_THREADS) tw[i] = __ldg(p.tw + i);
    float2* line = lines + ll * LP;
    auto sync = [] { __syncthreads(); };
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int gline = tile * LPC + ll;
        const bool active = gline < nlines;
        const int img = gline / p.N, y = gline % p.N;           // ws holds N rows per plane
        float2 v[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = make_float2(0.f, 0.f);
        if (active) {
            const int plane = plane0 + img;
            switch (p.in_mode) {
                case ASM_B200_IN_COMPLEX: load16<ASM_B200_IN_COMPLEX, TPL>(v, p, plane, y, tl); break;
                case ASM_B200_IN_AMP_PHASE: load16<ASM_B200_IN_AMP_PHASE, TPL>(v, p, plane, y, tl); break;
                case ASM_B200_IN_CONST_AMP_PHASE: load16<ASM_B200_IN_CONST_AMP_PHASE, TPL>(v, p, plane, y, tl); break;
                case ASM_B200_IN_SQRT_REAL: load16<ASM_B200_IN_SQRT_REAL, TPL>(v, p, plane, y, tl); break;
                case ASM_B200_IN_COT_FIELD: load16<ASM_B200_IN_COT_FIELD, TPL>(v, p, plane, y, tl); break;
                default: load16<ASM_B200_IN_REAL, TPL>(v, p, plane, y, tl); break;
            }
        }
        fwd_line<n, RowLayout>(v, line, tw, tl, sync);
        sts16<RowLayout, 0>(v, line + RowLayout::base(thread_part(tl, 0)));
        __syncthreads();
        if (active) {
            // coalesced copy of the digit-reversed line to the workspace (dense, position order)
            float2* dst = p.ws + ((size_t)img * p.N + y) * L;
#pragma unroll
            for (int k = 0; k < 16; ++k) dst[tl + TPL * k] = line[RowLayout::phys(tl) + RowLayout::off(k, n - 4)];
        }
        __syncthreads();
    }
}

// MOM: also write the focal-stack moment partials (p.part) of the cropped rows
template <int n, bool MOM = false>
__global__ void __launch_bounds__(ROW_THREADS, 1024 / ROW_THREADS) k_rows_inv(const Params p, int plane0, int nlines, int ntiles) {
    constexpr int L = 1 << n, TPL = L / 16, LPC = ROW_THREADS / TPL, LP = RowLayout::line_elems(L);
    constexpr TwLayout lay = make_layout(n);
    constexpr int NTW = lay.total - lay.fwd_end;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* lines = reinterpret_cast<float2*>(smem_raw);
    float2* tw_s = lines + LPC * LP;
    float2* fold = tw_s + NTW;                                  // [8 warps][2] fold partials (adjoint, padded)
    const float2* tw = tw_s - lay.fwd_end;                      // so that layout offsets apply directly
    const int t = threadIdx.x, ll = t / TPL, tl = t % TPL;
    for (int i = t; i < NTW; i += ROW_THREADS) tw_s[i] = __ldg(p.tw + lay.fwd_end + i);
    float2* line = lines + ll * LP;
    auto sync = [] { __syncthreads(); };
    const bool folding = p.adj && p.P > 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int gline = tile * LPC + ll;
        const bool active = gline < nlines;
        const int img = gline / p.N, y = gline % p.N;
        if (active) {
            const float2* src = p.ws + ((size_t)img * p.N + y) * L;
#pragma unroll
            for (int k = 0; k < 16; ++k) line[RowLayout::phys(tl) + RowLayout::off(k, n - 4)] = src[tl + TPL * k];
        }
        __syncthreads();
        float2 v[16];
        lds16<RowLayout, 0>(v, line + RowLayout::base(thread_part(tl, 0)));
        inv_line<n, RowLayout>(v, line, tw, tl, sync);
        // v now holds positions tl + TPL*i (window n-4) of the row in natural order
        const int plane = plane0 + img;
        float2 fl = make_float2(0.f, 0.f), fr = make_float2(0.f, 0.f);
        if (folding) {
            // adjoint of replicate padding: fold columns [0,P) onto 0 and [P+N, M) onto N-1.  Deterministic (no floating-
            // point atomics): xor shuffles inside the line's threads of a warp, then, for lines that span several warps,
            // the warps' partials are added in a fixed order.
            if (active) {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int pos = tl + TPL * i;
                    if (pos < p.P) { fl.x += v[i].x; fl.y += v[i].y; }
                    if (pos >= p.P + p.N) { fr.x += v[i].x; fr.y += v[i].y; }
                }
            }
#pragma unroll
            for (int o = 1; o < (TPL < 32 ? TPL : 32); o <<= 1) {
                fl.x += __shfl_xor_sync(0xffffffffu, fl.x, o); fl.y += __shfl_xor_sync(0xffffffffu, fl.y, o);
                fr.x += __shfl_xor_sync(0xffffffffu, fr.x, o); fr.y += __shfl_xor_sync(0xffffffffu, fr.y, o);
            }
            if constexpr (TPL > 32) {
                constexpr int WPL = TPL / 32;                            // warps per line
                if ((t & 31) == 0) { fold[2 * (t >> 5)] = fl; fold[2 * (t >> 5) + 1] = fr; }
                __syncthreads();
                fl = make_float2(0.f, 0.f); fr = make_float2(0.f, 0.f);
#pragma unroll
                for (int w = 0; w < WPL; ++w) {
                    const float2 a = fold[2 * (ll * WPL + w)], b2 = fold[2 * (ll * WPL + w) + 1];
                    fl.x += a.x; fl.y += a.y; fr.x += b2.x; fr.y += b2.y;
                }
            }
        }
        float dot = 0.f;
        if (active && p.out0) {
            switch (p.out_mode) {
                case ASM_B200_OUT_COMPLEX: emit16<ASM_B200_OUT_COMPLEX, TPL>(v, p, plane, y, tl, fl, fr); break;
                case ASM_B200_OUT_INTENSITY: emit16<ASM_B200_OUT_INTENSITY, TPL>(v, p, plane, y, tl, fl, fr); break;
                case ASM_B200_OUT_ABS_ANGLE: emit16<ASM_B200_OUT_ABS_ANGLE, TPL>(v, p, plane, y, tl, fl, fr); break;
                case ASM_B200_OUT_REIM_CAT: emit16<ASM_B200_OUT_REIM_CAT, TPL>(v, p, plane, y, tl, fl, fr); break;
                case ASM_B200_OUT_ABSANG_CAT: emit16<ASM_B200_OUT_ABSANG_CAT, TPL>(v, p, plane, y, tl, fl, fr); break;
                case ASM_B200_OUT_GRAD_AP: emit16<ASM_B200_OUT_GRAD_AP, TPL>(v, p, plane, y, tl, fl, fr); break;
                default: dot = emit16<OUT_DOT, TPL>(v, p, plane, y, tl, fl, fr); break;
            }
        }
        if (p.out_mode == OUT_DOT) {
            // warp reduce, then one double atomic per warp and sample (lines of one warp may belong to 2 planes)
            const int b = active ? plane / p.C : -1;
            const int b0 = __shfl_sync(0xffffffffu, b, 0);
            const bool uniform = __all_sync(0xffffffffu, b == b0);
            const double K = p.z_f64 ? 6.283185307179586 : (double)6.2831854820251465f;
            if (uniform) {
                float s = dot;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                if ((t & 31) == 0 && b0 >= 0) atomicAdd((double*)p.out0 + b0, (double)s * K * p.inv_lambda);
            } else if (b >= 0) {
                atomicAdd((double*)p.out0 + b, (double)dot * K * p.inv_lambda);
            }
        }
        if constexpr (MOM) {
            // moments of the cropped row: one partial per (row, warp of the row), R = N max(1, TPL / 32) per plane
            constexpr int W = TPL < 32 ? TPL : 32, WPL = TPL > 32 ? TPL / 32 : 1;
            float m[3] = {0.f, 0.f, 0.f};
            if (active) {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int x = tl + TPL * i - p.P;
                    if (x >= 0 && x < p.N) mom_add(m, v[i]);
                }
            }
            double d[3];
            mom_reduce<W>(d, m);
            if (active && tl % W == 0) {
                double* dst = p.part + (((size_t)img * p.N + y) * WPL + tl / 32) * 3;
                dst[0] = d[0]; dst[1] = d[1]; dst[2] = d[2];
            }
        }
        __syncthreads();   // the line buffers (and fold) are reused by the next tile
    }
}

// ---------------------------------------------------------------------------------------------------
// column pass: one CTA = one slab of CC columns of one sample, CC * L/16 threads.
// smem: slab [L][CC] float2 | kappa [L/2+1][CC] double (KZTAB) | twiddles | fold accumulators | mbarrier
// ---------------------------------------------------------------------------------------------------
#ifndef ASM_CC11
#define ASM_CC11 4   // FFT 2048: 4 columns x 128 threads = 512-thread CTAs (128 registers per thread; 8 columns would mean 1024 threads capped at 64)
#endif
#ifndef ASM_CC12
#define ASM_CC12 4
#endif
__host__ __device__ constexpr int cols_per_slab(int n) { return n <= 9 ? 16 : n == 10 ? ASM_CC10 : n == 11 ? ASM_CC11 : ASM_CC12; }
__host__ __device__ constexpr bool use_kz_table(int n) { return n <= 11; }      // kappa table exists in the workspace
__host__ __device__ constexpr bool kz_in_smem(int n) { return n <= 10 || (n == 11 && ASM_CC11 <= 4); }   // ... and its slab is staged in shared memory (else read per bin from L2)
#ifndef ASM_MB11
#define ASM_MB11 2
#endif
__host__ __device__ constexpr int cols_min_blocks(int n) { return n <= 8 ? 4 : n <= 10 ? (1024 / (cols_per_slab(n) * (1 << n) / 16)) : n == 11 ? ASM_MB11 : (ASM_CC12 <= 2 ? 2 : 1); }

// BL: band-limited calls (p.band_limit; a template parameter so that the plain instantiations stay the code they were)
template <int n, bool BL = false>
__global__ void __launch_bounds__(cols_per_slab(n) * (1 << n) / 16, cols_min_blocks(n))
k_cols(const Params p, const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_src,
       const __grid_constant__ CUtensorMap tmap_kz, int plane0) {
    constexpr int L = 1 << n, TPL = L / 16, CC = cols_per_slab(n), NT = CC * TPL;
    constexpr bool KZTAB = kz_in_smem(n);            // kappa slab staged in shared memory by TMA
    constexpr bool KZGLOB = use_kz_table(n) && !KZTAB; // kappa read per bin from the global table
    constexpr int KZROWS = KZTAB ? L / 2 + 1 : 0;
    constexpr TwLayout lay = make_layout(n);
    using LAY = ColLayout<CC>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float2* slab = reinterpret_cast<float2*>(smem_raw);              // [L][CC]
    double* kz_s = reinterpret_cast<double*>(slab + L * CC);         // [KZROWS][CC]
    float2* tw = reinterpret_cast<float2*>(kz_s + KZROWS * CC);      // [lay.total]
    float2* fold = tw + lay.total;                                   // [2][warps][CC] fold partials
    uint64_t* bar = reinterpret_cast<uint64_t*>(fold + 2 * CC * (NT / 32 > 0 ? NT / 32 : 1));
    const int t = threadIdx.x, c = t % CC, tl = t / CC;
    const int nslab = L / CC;
    const int img = blockIdx.x / nslab, slab_i = blockIdx.x % nslab;
    const int plane = plane0 + img;
    const int rows = p.N;                                            // rows held by the workspace
    const int boxr = rows < 256 ? rows : 256;
    constexpr int KBOX = (L / 2) < 256 ? (L / 2) : 256;

    if (t == 0) { mbar_init(bar, 1); fence_mbar_init(); }
    __syncthreads();
    if (t == 0) {
        mbar_expect_tx(bar, (uint32_t)(rows * CC * sizeof(float2)) + (KZTAB ? (uint32_t)((L / 2) * CC * sizeof(double)) : 0u));
        for (int r0 = 0; r0 < rows; r0 += boxr)
            tma_load_3d(slab + (size_t)(p.P + r0) * CC, &tmap_src, bar, slab_i * CC * 2, r0, src_slot(p, plane0, img));
        if constexpr (KZTAB) {
            for (int r0 = 0; r0 < L / 2; r0 += KBOX)
                tma_load_3d(kz_s + (size_t)r0 * CC, &tmap_kz, bar, slab_i * CC * 2, r0, 0);
        }
    }
    for (int i = t; i < lay.total; i += NT) tw[i] = __ldg(p.tw + i);
    if constexpr (KZTAB) {
        if (t < CC) kz_s[(size_t)(L / 2) * CC + t] = __ldg(p.kzt + (size_t)(L / 2) * L + slab_i * CC + t);   // Nyquist row
    }

    // per-sample constant of the transfer function (overlaps the TMA)
    const int b = plane / p.C;
    double cph;                                                      // phase constant c
    if (p.z_f64) cph = 6.283185307179586 * __ldg((const double*)p.z + b);
    else cph = (double)__fmul_rn(6.2831854820251465f, __ldg((const float*)p.z + b));
    if (p.h_mode == H_CONJ) cph = -cph;
    // band limit: this column's |k(v)| is within it -> rows |k(u)| <= lim_u are kept; otherwise none (lim_u = -1)
    int lim_u = L;
    if constexpr (BL) {
        const int vpos = freq_of_pos(n, slab_i * CC + c), lim = band_limit_of(p, b);
        lim_u = (vpos <= L / 2 ? vpos : L - vpos) <= lim ? lim : -1;
    }

    mbar_wait(bar, 0);
    if (p.P > 0) {
        // rows [P, P+N) came from the workspace; fill the padding rows (replicate for forward, zero for adjoint)
        const float2 top = slab[(size_t)p.P * CC + c], bot = slab[(size_t)(p.P + p.N - 1) * CC + c];
        const float2 zero = make_float2(0.f, 0.f);
        for (int r = tl; r < p.P; r += TPL) {
            slab[(size_t)r * CC + c] = p.adj ? zero : top;
            slab[(size_t)(p.P + p.N + r) * CC + c] = p.adj ? zero : bot;
        }
    }
    __syncthreads();

    float2* col = slab + c;
    auto sync = [] { __syncthreads(); };
    float2 v[16];
    // ---- forward column FFT ----
    lds16<LAY, n - 4>(v, col + LAY::base(thread_part(tl, n - 4)));
    fwd_line<n, LAY>(v, col, tw, tl, sync);

    // ---- transfer function: register i holds column-frequency u = Q + (L/16) i ----
    {
        const int Q = fwd_q_from_hi(n, 0, tl);
        const double MAGIC = 6755399441055744.0;                     // 1.5 * 2^52: round to nearest integer
        double cs = 0.0; float kv2 = 0.f;
        if constexpr (!KZTAB && !KZGLOB) {
            cs = cph * p.inv_lambda * 0.15915494309189535;           // cycles per unit of (kz * lambda)
            const int vfreq = freq_of_pos(n, slab_i * CC + c);
            const int kv = vfreq < L / 2 ? vfreq : vfreq - L;
            kv2 = (float)(kv * kv);
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int u = Q + TPL * i;
            const int ru = u <= L / 2 ? u : L - u;                   // |k(u)|
            double tt, kzl = 0.0;
            if constexpr (KZTAB || KZGLOB) {
                const double kap = KZTAB ? kz_s[ru * CC + c] : __ldg(p.kzt + (size_t)ru * L + slab_i * CC + c);
                tt = kap * cph;
                if (p.h_mode == H_DERIV) kzl = kap * (6.283185307179586 * p.lambda);
            } else {
                const int ku = u < L / 2 ? u : u - L;
                const float kk = (float)(ku * ku) + kv2;             // exact (< 2^24)
                const double arg = fma(-p.s2, (double)kk, 1.0);      // 1 - lambda^2 (fx^2 + fy^2)
                kzl = arg > 0.0 ? sqrt(arg) : 0.0;                   // kz * lambda, evanescent -> 0 (H = 1)
                tt = kzl * cs;
            }
            const double rr = tt - __dadd_rn(__dadd_rn(tt, MAGIC), -MAGIC);
            float sn, cn;
            __sincosf((float)rr * 6.283185307179586f, &sn, &cn);
            const float sc = (!BL || ru <= lim_u) ? p.inv_m2 : 0.f;  // H = 0 outside the band limit
            if (p.h_mode == H_DERIV) v[i] = cmul_scaled(v[i], -sn, cn, (float)(kzl - p.kshift) * sc);
            else v[i] = cmul_scaled(v[i], cn, sn, sc);
        }
    }

    // ---- inverse column FFT ----
    inv_line<n, LAY>(v, col, tw, tl, sync);
    sts16<LAY, n - 4>(v, col + LAY::base(thread_part(tl, n - 4)));

    if (p.adj && p.P > 0) {
        // adjoint of replicate padding along rows: fold rows [0,P) onto row P and [P+N, M) onto row P+N-1
        float2 fl = make_float2(0.f, 0.f), fr = make_float2(0.f, 0.f);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int pos = thread_part(tl, n - 4) | (i << (n - 4));
            if (pos < p.P) { fl.x += v[i].x; fl.y += v[i].y; }
            if (pos >= p.P + p.N) { fr.x += v[i].x; fr.y += v[i].y; }
        }
        // deterministic column sums (no floating-point atomics): a warp holds 32 / CC rows x CC columns -> xor shuffles over
        // the row bits, then thread (tl = 0, c) adds the warps' partials in a fixed order
        constexpr int NW = NT / 32 > 0 ? NT / 32 : 1;
#pragma unroll
        for (int o = CC; o < 32; o <<= 1) {
            fl.x += __shfl_xor_sync(0xffffffffu, fl.x, o); fl.y += __shfl_xor_sync(0xffffffffu, fl.y, o);
            fr.x += __shfl_xor_sync(0xffffffffu, fr.x, o); fr.y += __shfl_xor_sync(0xffffffffu, fr.y, o);
        }
        if ((t & 31) < CC) { fold[(t >> 5) * CC + c] = fl; fold[NW * CC + (t >> 5) * CC + c] = fr; }
        __syncthreads();
        if (tl == 0) {
            float2& r0 = slab[(size_t)p.P * CC + c];
            float2& r1 = slab[(size_t)(p.P + p.N - 1) * CC + c];
#pragma unroll
            for (int w = 0; w < NW; ++w) {
                const float2 a = fold[w * CC + c], b2 = fold[NW * CC + w * CC + c];
                r0.x += a.x; r0.y += a.y; r1.x += b2.x; r1.y += b2.y;
            }
        }
    }
    fence_proxy_async();
    __syncthreads();
    if (t == 0) {
        for (int r0 = 0; r0 < rows; r0 += boxr)
            tma_store_3d(&tmap, slab + (size_t)(p.P + r0) * CC, slab_i * CC * 2, r0, img);
        tma_commit();
        tma_wait_read0();
    }
}

}  // namespace asmb
#include "k32.cuh"
#include "k32t.cuh"
#include "k64.cuh"
#ifdef ASM_B200_TUNING   /* measured alternatives: tools/ A/B builds only, not in the product library */
#include "k64t.cuh"
#endif
#ifdef ASM_B200_TUNING
#include "resident.cuh"
#include "cluster256.cuh"
#endif
#include "unwrap.cuh"
#include "dft_any.cuh"
namespace asmb {

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(f);
    });
    return fn;
}

// process-wide launch counter (bench.py reports it as gpu_launches) and optional per-pass event timing
static std::atomic<unsigned long long> g_launches{0};
static std::atomic<int> g_profile{0};
static std::mutex g_prof_mu;
static double g_prof_ms[3] = {0.0, 0.0, 0.0};   // rows_fwd, cols, rows_inv

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Tunables.  The product build reads NO environment variables: every knob is its compiled default.  Builds with
// -DASM_B200_TUNING (tools/ A/B runs only) let ASM_B200_<NAME> override a knob, read once per process.
static int knob(const char* name, int def) {
#ifdef ASM_B200_TUNING
    const char* e = getenv(name);
    return e ? atoi(e) : def;
#else
    (void)name;
    return def;
#endif
}
#define ASM_KNOB(fn, name, def) static int fn() { static const int v = knob(name, def); return v; }
ASM_KNOB(knob_chunk_mb, "ASM_B200_CHUNK_MB", 0)    // bytes of L2-resident intermediates in flight, all lanes (0: per-size default)
ASM_KNOB(knob_lanes, "ASM_B200_LANES", 3)          // chunks in flight (internal streams)
ASM_KNOB(knob_cols_cc, "ASM_B200_COLS_CC", 8)      // FFT 1024: columns per slab of the column kernel (8 or 4)
ASM_KNOB(knob_bulk, "ASM_B200_BULK", 3)            // FFT 1024: bit 0 / 1 = TMA bulk-copy forward / inverse row kernels
ASM_KNOB(knob_row_ctas, "ASM_B200_ROW_CTAS", 12 / K32_BULK_WARPS > 0 ? 12 / K32_BULK_WARPS : 1)   // FFT 1024: bulk row CTAs per SM
ASM_KNOB(knob_ldg_row_ctas, "ASM_B200_LDG_ROW_CTAS", K32_ROW_CTAS)   // FFT 1024: register-landing row CTAs per SM
ASM_KNOB(knob_cols_ctas, "ASM_B200_COLS_CTAS", 0)    // FFT 1024: column CTAs per SM (0: as many as fit, 16 / CC)
ASM_KNOB(knob_graphs, "ASM_B200_GRAPHS", 1)          // replay repeated launch sequences as CUDA graphs (launch-bound small transforms)
ASM_KNOB(knob_graph_max_n, "ASM_B200_GRAPH_MAX_N", 9) // ... for FFT sizes up to 2^n
ASM_KNOB(knob_resident, "ASM_B200_RESIDENT", 0)
ASM_KNOB(knob_k32t, "ASM_B200_K32T", 1)            // FFT 1024: transposed-intermediate kernels (k32t.cuh) instead of k32_rows / k32_cols
ASM_KNOB(knob_promo, "ASM_B200_PROMO", 0)          // k32t tile tensor map: L2 promotion of the 64-byte box rows (0 none, 1 64 B, 2 128 B = every tile load fetches twice its bytes)
ASM_KNOB(knob_cluster256, "ASM_B200_CLUSTER256", 0)  // FFT 256: sample resident in a 4-CTA cluster, transposes through DSMEM (cluster256.cuh); measured slower than the L2 pipeline (profiles/r02_cluster256.md), so opt-in
ASM_KNOB(knob_k64t, "ASM_B200_K64T", 0)            // FFT 2048, TMA-capable modes: transposed-intermediate kernels (k64t.cuh); measured +1.5 % unpadded / -11 % padded (profiles/r02_experiments.md section 7), so opt-in
ASM_KNOB(knob_k64, "ASM_B200_K64", 1)              // FFT 2048: 2 x 1024 kernels (k64.cuh) instead of the generic 16-point kernels    // FFT <= 256: one persistent launch per call (resident.cuh)

// default budget (measured on B200): small transforms like a tight ring, FFT sizes >= 1024 prefer fuller waves
// FFT 1024 unpadded (k32t, 8 MB per sample): 2 lanes x 6 samples keeps the intermediates L2 resident; padded 512^2 (4 MB per
// sample) prefers 3 lanes x 18 (measured 76.9 k vs 67.2 k units/s)
static size_t default_budget(int n, bool padded) { return (size_t)(n <= 9 ? 48 : (n == 10 && !padded) ? 120 : 216) << 20; }
static int default_lanes(int n, bool padded) { return (n == 10 && !padded) ? 2 : knob_lanes(); }

// Chunks are issued round-robin on `lanes` internal streams so that the passes of different chunks overlap.  A lane set
// (streams + fork / join events) belongs to one caller stream at a time: calls on different caller streams of a device
// get different sets (up to LANE_SETS; beyond that the least recently used set is shared, which only adds a false
// dependency, never a race).  Host threads enqueueing on the same set serialise on its mutex; nothing waits for the GPU.
constexpr int MAX_LANES = 8, LANE_SETS = 4;
struct LaneSet {
    cudaStream_t st[MAX_LANES]; cudaEvent_t fork, join[MAX_LANES];
    bool ok = false; cudaStream_t owner = nullptr; unsigned long long stamp = 0; std::mutex issue;
};
static LaneSet* lanes_for(cudaStream_t caller) {
    static LaneSet sets[64][LANE_SETS];
    static std::mutex mu;
    static unsigned long long tick = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lk(mu);
    LaneSet* pick = nullptr;
    for (auto& s : sets[dev]) if (s.ok && s.owner == caller) pick = &s;
    if (!pick) for (auto& s : sets[dev]) if (!s.ok) { pick = &s; break; }
    if (!pick) { pick = &sets[dev][0]; for (auto& s : sets[dev]) if (s.stamp < pick->stamp) pick = &s; }
    if (!pick->ok) {
        for (int i = 0; i < MAX_LANES; ++i) {
            if (cudaStreamCreateWithFlags(&pick->st[i], cudaStreamNonBlocking) != cudaSuccess) return nullptr;
            if (cudaEventCreateWithFlags(&pick->join[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
        }
        if (cudaEventCreateWithFlags(&pick->fork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
        pick->ok = true;
    }
    pick->owner = caller;
    pick->stamp = ++tick;
    return pick;
}

static int sm_count() {
    static int sms[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) return 148;
    if (!sms[dev]) cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev);
    return sms[dev] > 0 ? sms[dev] : 148;
}

struct Geometry {
    int n, M, P, chunk, lanes, cc;         // log2 M, FFT size, pad offset, samples per chunk, chunks in flight, FFT 1024: columns per slab
    size_t tw_bytes, kz_bytes, ctl_bytes, img_bytes;  // table regions, group counters (resident), workspace bytes per sample
    bool resident;                         // one persistent launch; chunk = groups (= L2-resident slots), group = CTAs per sample
    int group;
};

static int pow2_floor(int x) { int r = 1; while (2 * r <= x) r *= 2; return r; }

static bool make_geometry(int planes, int N, int pad, Geometry* g) {
    if (planes <= 0 || N <= 0 || (N & (N - 1))) return false;
    const int M = pad ? 2 * N : N;
    int n = 0;
    while ((1 << n) < M) ++n;
    if (n < 5 || n > 12 || N < 16) return false;
    g->n = n; g->M = M; g->P = (M - N) / 2;
    g->tw_bytes = align_up(((size_t)make_layout(n).total + (n == 11 ? K32_TW : 0)) * sizeof(float2), 256);
    g->kz_bytes = use_kz_table(n) ? align_up((size_t)(M / 2 + 1) * M * sizeof(double), 256) : 0;
    g->img_bytes = (size_t)N * M * sizeof(float2);
    g->cc = knob_cols_cc() == 4 ? 4 : 8;
    g->resident = false; g->group = 1; g->ctl_bytes = 0;
#ifdef ASM_B200_TUNING
    if (n <= 9 && knob_resident()) {
        // resident.cuh: G co-resident CTAs per sample, every group owns one L2-resident slot
        const int cap = RES_CTAS_PER_SM * sm_count();
        const size_t budget = (size_t)(knob_chunk_mb() > 0 ? knob_chunk_mb() : 80) << 20;
        int G = 1;
        while (G < 16 && (size_t)(cap / G) * g->img_bytes > budget) G *= 2;
        const int lpc = 4096 / M, ntile = (N + lpc - 1) / lpc, nsi = M * M / 4096 > 0 ? M * M / 4096 : 1;
        const int gmax = pow2_floor(ntile < nsi ? ntile : nsi);
        while (G < gmax && G < 16 && (long long)planes * G * 2 <= cap) G *= 2;    // few samples: more CTAs per sample
        int groups = cap / G;
        if (groups > planes) groups = planes;
        g->resident = true; g->group = G; g->chunk = groups; g->lanes = 1;
        g->ctl_bytes = align_up((size_t)groups * sizeof(int), 256);
        return true;
    }
#endif
    int lanes = knob_lanes() != 3 ? knob_lanes() : default_lanes(n, pad != 0);   // 3 = the knob's default: per-size choice
    lanes = lanes < 1 ? 1 : (lanes > MAX_LANES ? MAX_LANES : lanes);
    const size_t budget = knob_chunk_mb() > 0 ? (size_t)knob_chunk_mb() << 20 : default_budget(n, pad != 0);
    size_t c = budget / g->img_bytes / lanes;
    if (c < 1) c = 1;
    if (c > (size_t)planes) c = planes;
    // wave quantisation: every pass of a chunk is its own launch, so pick the chunk size (within a factor 2 of the
    // budget) whose column pass fills the resident CTA slots best (e.g. 9 x 128 slabs on 296 slots = 97 %)
    if ((n == 10 || n == 11) && c > 1) {
        const int cc = n == 10 ? g->cc : K64_CC;
        const int slots = (n == 10 ? 16 / cc : 2) * sm_count();      // persistent column CTAs
        const int items = M / cc;
        double best = 0.0; size_t best_c = c;
        for (size_t t = c; t >= (c + 1) / 2 && t >= 1; --t) {
            const double waves = (double)t * items / slots;
            const double util = waves / (double)(long long)(waves + 0.999999);
            if (util > best + 1e-9) { best = util; best_c = t; }
        }
        c = best_c;
    }
    while (lanes > 1 && (size_t)(lanes - 1) * c >= (size_t)planes) --lanes;   // no more lanes than chunks
    g->chunk = (int)c;
    g->lanes = lanes;
    return true;
}

static size_t workspace_need(const Geometry& g) { return g.tw_bytes + g.kz_bytes + g.ctl_bytes + g.img_bytes * g.chunk * g.lanes; }

// opt-in shared memory is a per-device function attribute: set once per (device, kernel)
template <class K>
static cudaError_t set_smem(K kernel, size_t bytes) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}
static bool attrs_done(std::atomic<unsigned long long>& mask, int* dev_out) {
    int dev = 0;
    cudaGetDevice(&dev);
    *dev_out = dev;
    return dev >= 0 && dev < 64 && ((mask.load() >> dev) & 1ull);
}
static void attrs_mark(std::atomic<unsigned long long>& mask, int dev) { if (dev >= 0 && dev < 64) mask.fetch_or(1ull << dev); }

template <int n>
static cudaError_t set_attrs(size_t smem_fwd, size_t smem_inv, size_t smem_cols) {
    static std::atomic<unsigned long long> done{0};
    int dev;
    if (attrs_done(done, &dev)) return cudaSuccess;
    cudaError_t e;
    if ((e = set_smem(k_rows_fwd<n>, smem_fwd)) != cudaSuccess) return e;
    if ((e = set_smem(k_rows_inv<n>, smem_inv)) != cudaSuccess) return e;
    if ((e = set_smem(k_rows_inv<n, true>, smem_inv)) != cudaSuccess) return e;
    if ((e = set_smem(k_cols<n>, smem_cols)) != cudaSuccess) return e;
    if ((e = set_smem(k_cols<n, true>, smem_cols)) != cudaSuccess) return e;
    attrs_mark(done, dev);
    return cudaSuccess;
}

static bool encode3d(EncodeTiledFn enc, CUtensorMap* m, void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint32_t b0, uint32_t b1,
                     CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_NONE, CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_128B) {
    const cuuint64_t dims[3] = {d0, d1, d2};
    const cuuint64_t strides[2] = {d0 * 4, d0 * d1 * 4};
    const cuuint32_t box[3] = {b0, b1, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               swz, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// ---------------------------------------------------------------------------------------------------
// Launch-sequence cache.  A call on a small transform is hundreds of kernels of a few microseconds each (256^2, batch
// 4096: 385 launches), and issuing them one by one costs more host time than the GPU needs to run them.  The launch
// sequence of a call is a pure function of its arguments, so the second time a call with the SAME arguments (pointers
// included) is seen its sequence is captured into a CUDA graph (stream capture of exactly the code below), instantiated
// once and replayed with one cudaGraphLaunch from then on.  Only argument VALUES are kept (a few hundred bytes per entry,
// at most GRAPH_CACHE entries per device, least recently used first out); no device memory is retained and nothing is
// touched after the call returns.  Calls made while the caller's stream is itself being captured are simply enqueued.
// ---------------------------------------------------------------------------------------------------
struct CallKey { unsigned char b[320]; int len; };
template <class T>
static void key_add(CallKey& k, const T& v) {
    if (k.len + (int)sizeof(T) <= (int)sizeof(k.b)) { memcpy(k.b + k.len, &v, sizeof(T)); k.len += (int)sizeof(T); }
}
// Focal stack (asm_b200_focal_stack): pass 1 of a chunk of samples writes their spectra to S once; then each group of
// tq planes runs the column pass S -> T and the inverse row pass T -> output (and the moments reduction).  A lane's
// region is [S: chunk samples][T: tq planes][row moment partials of the tq planes].
struct StackPlan {
    int K;                                 // distances per sample
    int tq;                                // planes per group: a multiple of K (several samples), or <= K (one sample)
    int R;                                 // moment partials per plane written by the inverse row kernel
    double* mom;                           // [B][K][3] moments, or nullptr
    size_t s_elems, t_elems, lane_elems;   // float2 elements of S, T and the whole lane region
};

static CallKey make_key(const Params& p, const Geometry& g, int kind, const StackPlan* sp) {
    CallKey k;
    memset(&k, 0, sizeof(k));
    key_add(k, p.in0); key_add(k, p.in1); key_add(k, p.aux0); key_add(k, p.aux1); key_add(k, p.out0); key_add(k, p.out1);
    key_add(k, p.z); key_add(k, p.ws); key_add(k, p.tw); key_add(k, p.tw32); key_add(k, p.kzt);
    key_add(k, p.s2); key_add(k, p.inv_lambda); key_add(k, p.lambda); key_add(k, p.kshift); key_add(k, p.S);
    key_add(k, p.in_scale); key_add(k, p.out_scale); key_add(k, p.inv_m2);
    key_add(k, p.planes); key_add(k, p.C); key_add(k, p.N); key_add(k, p.M); key_add(k, p.P);
    key_add(k, p.in_mode); key_add(k, p.out_mode); key_add(k, p.aux_mode); key_add(k, p.h_mode); key_add(k, p.adj); key_add(k, p.z_f64);
    key_add(k, p.band_limit);
    key_add(k, g.n); key_add(k, g.chunk); key_add(k, g.lanes); key_add(k, g.cc); key_add(k, kind);
    const int stack = sp != nullptr;
    key_add(k, stack);
    if (sp) { key_add(k, sp->K); key_add(k, sp->tq); key_add(k, sp->R); key_add(k, sp->mom); key_add(k, sp->lane_elems); }
    return k;
}
constexpr int GRAPH_CACHE = 8;
struct GraphEntry { CallKey key; cudaGraphExec_t exec = nullptr; unsigned long long launches = 0, stamp = 0; int seen = 0; };
struct GraphCache { GraphEntry e[GRAPH_CACHE]; std::mutex mu; unsigned long long tick = 0; };
static GraphCache* graph_cache() {
    static GraphCache caches[64];
    int dev = 0;
    cudaGetDevice(&dev);
    return (dev >= 0 && dev < 64) ? &caches[dev] : nullptr;
}

// Issues the three passes of every chunk, round-robin over the lane streams (fork/join with events).
// setup(stream) builds the tables; pass(k, lane, stream, params, plane0, nimg) launches pass k of one chunk.
// A launch error stops the issue loop at the chunk that produced it (the lanes are still joined) and is the call's
// return value; an error that was already pending when the call started is not attributed to this library.
// Focal stack (sp != nullptr): a chunk is g.chunk samples; pass 1 writes their spectra to S, then every group of
// sp->tq planes is 2 launches (3 with moments), so a chunk of c samples costs 1 + c K / tq * (2 or 3) launches.
template <class Setup, class Pass>
static int issue_chunks(const Params& p0, const Geometry& g, int L, cudaStream_t st, LaneSet* ls, int lanes, bool prof,
                        Setup& setup, Pass& pass, unsigned long long* launches_out, const StackPlan* sp) {
    const size_t lane_elems = sp ? sp->lane_elems : (size_t)g.chunk * p0.N * L;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    if (prof) for (auto& x : ev) cudaEventCreate(&x);
    const cudaError_t pending = cudaPeekAtLastError();
    cudaError_t err = cudaSuccess;
    setup(st);
    if (lanes > 1) {   // fork: every lane stream waits for the tables (and everything before) on the caller's stream
        cudaEventRecord(ls->fork, st);
        for (int l = 0; l < lanes; ++l) cudaStreamWaitEvent(ls->st[l], ls->fork, 0);
    }
    unsigned long long launches = 1;
    int ci = 0;
    for (int plane0 = 0; plane0 < p0.planes && err == cudaSuccess; plane0 += g.chunk, ++ci) {
        const int nimg = (p0.planes - plane0 < g.chunk) ? p0.planes - plane0 : g.chunk;
        const int l = ci % lanes;
        cudaStream_t s = lanes > 1 ? ls->st[l] : st;
        Params p = p0;
        p.ws = p0.ws + l * lane_elems;
        if (sp) {
            if (prof) cudaEventRecord(ev[0], s);
            pass(0, l, s, p, plane0, nimg);
            if (prof) cudaEventRecord(ev[1], s);
            Params pt = p;
            pt.src = p.ws; pt.ws = p.ws + sp->s_elems; pt.kst = sp->K; pt.s0 = plane0;
            pt.part = sp->mom ? reinterpret_cast<double*>(pt.ws + sp->t_elems) : nullptr;
            const int q_end = (plane0 + nimg) * sp->K;
            for (int q0 = plane0 * sp->K; q0 < q_end; q0 += sp->tq) {
                const int cnt = q_end - q0 < sp->tq ? q_end - q0 : sp->tq;
                pass(1, l, s, pt, q0, cnt);
                pass(2, l, s, pt, q0, cnt);
                if (pt.part) k_moments_reduce<<<(cnt + 7) / 8, 256, 0, s>>>(pt.part, sp->mom, sp->R, cnt, q0);
                launches += pt.part ? 3 : 2;
            }
            launches += 1;
            if (pending == cudaSuccess) err = cudaPeekAtLastError();
            if (prof) {   // the column and inverse row passes of all groups are reported together in the column slot
                cudaEventRecord(ev[3], s);
                cudaEventSynchronize(ev[3]);
                std::lock_guard<std::mutex> lk(g_prof_mu);
                float ms = 0.f;
                cudaEventElapsedTime(&ms, ev[0], ev[1]); g_prof_ms[0] += ms;
                cudaEventElapsedTime(&ms, ev[1], ev[3]); g_prof_ms[1] += ms;
            }
            continue;
        }
        for (int k = 0; k < 3; ++k) {
            if (prof) cudaEventRecord(ev[k], s);
            pass(k, l, s, p, plane0, nimg);
        }
        launches += 3;
        if (pending == cudaSuccess) err = cudaPeekAtLastError();
        if (prof) {   // profiling mode serialises on purpose: it measures per-pass time, not throughput
            cudaEventRecord(ev[3], s);
            cudaEventSynchronize(ev[3]);
            std::lock_guard<std::mutex> lk(g_prof_mu);
            for (int k = 0; k < 3; ++k) { float ms = 0.f; cudaEventElapsedTime(&ms, ev[k], ev[k + 1]); g_prof_ms[k] += ms; }
        }
    }
    if (lanes > 1) {   // join: the caller's stream continues after every lane has drained
        for (int l = 0; l < lanes; ++l) { cudaEventRecord(ls->join[l], ls->st[l]); cudaStreamWaitEvent(st, ls->join[l], 0); }
    }
    if (prof) for (auto& x : ev) cudaEventDestroy(x);
    *launches_out = launches;
    if (err != cudaSuccess) { cudaGetLastError(); return (int)err; }   // ours: report it and clear the (non-sticky) state
    return 0;
}

template <class Setup, class Pass>
static int run_chunks(const Params& p0, const Geometry& g, int L, cudaStream_t st, Setup setup, Pass pass, int kind = 0,
                      const StackPlan* sp = nullptr) {
    const bool prof = g_profile.load() != 0;
    int lanes = prof ? 1 : g.lanes;
    LaneSet* ls = lanes > 1 ? lanes_for(st) : nullptr;
    if (!ls) lanes = 1;
    std::unique_lock<std::mutex> issue_lock;
    if (ls) issue_lock = std::unique_lock<std::mutex>(ls->issue);
    unsigned long long launches = 0;

    // launch-sequence cache: transforms whose calls are launch bound (many short kernels)
    const int nchunks = (p0.planes + g.chunk - 1) / g.chunk;
    GraphCache* gc = (!prof && knob_graphs() && g.n <= knob_graph_max_n() && nchunks >= 8) ? graph_cache() : nullptr;
    if (gc) {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) gc = nullptr;   // part of the caller's own graph
    }
    if (gc) {
        const CallKey key = make_key(p0, g, kind, sp);
        std::unique_lock<std::mutex> lk(gc->mu);
        GraphEntry* hit = nullptr;
        GraphEntry* victim = &gc->e[0];
        for (auto& e : gc->e) {
            if (e.seen > 0 && e.key.len == key.len && memcmp(e.key.b, key.b, key.len) == 0) hit = &e;
            if (e.stamp < victim->stamp) victim = &e;
        }
        if (hit && hit->exec) {                                   // replay
            hit->stamp = ++gc->tick;
            const cudaError_t e = cudaGraphLaunch(hit->exec, st);
            g_launches.fetch_add(hit->launches);
            return e == cudaSuccess ? 0 : (int)e;
        }
        if (hit) {                                                // second sighting: capture, instantiate, replay
            hit->stamp = ++gc->tick;
            cudaGraph_t graph = nullptr;
            if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                const int rc = issue_chunks(p0, g, L, st, ls, lanes, false, setup, pass, &launches, sp);
                const cudaError_t ec = cudaStreamEndCapture(st, &graph);
                if (rc == 0 && ec == cudaSuccess && graph && cudaGraphInstantiate(&hit->exec, graph, 0) == cudaSuccess) {
                    cudaGraphDestroy(graph);
                    hit->launches = launches;
                    const cudaError_t e = cudaGraphLaunch(hit->exec, st);
                    g_launches.fetch_add(launches);
                    return e == cudaSuccess ? 0 : (int)e;
                }
                if (graph) cudaGraphDestroy(graph);
                hit->exec = nullptr;
                cudaGetLastError();
                if (rc != 0) return rc;
            }
            // capture unavailable: fall through to plain issue
        } else {                                                  // first sighting: remember the arguments only
            if (victim->exec) { cudaGraphExecDestroy(victim->exec); victim->exec = nullptr; }
            victim->key = key; victim->seen = 1; victim->launches = 0; victim->stamp = ++gc->tick;
        }
    }
    const int rc = issue_chunks(p0, g, L, st, ls, lanes, prof, setup, pass, &launches, sp);
    g_launches.fetch_add(launches);
    return rc;
}

template <int n>
static int launch_n(const Params& p0, const Geometry& g, cudaStream_t st, const StackPlan* sp = nullptr) {
    constexpr int L = 1 << n, TPL = L / 16, LPC = ROW_THREADS / TPL, CC = cols_per_slab(n);
    constexpr int LP = RowLayout::line_elems(L);
    constexpr TwLayout lay = make_layout(n);
    constexpr int KZROWS = kz_in_smem(n) ? L / 2 + 1 : 0;
    const size_t smem_fwd = (size_t)LPC * LP * 8 + (size_t)lay.fwd_end * 8;
    constexpr int NWC = (CC * TPL) / 32 > 0 ? (CC * TPL) / 32 : 1;   // warps of a column CTA
    const size_t smem_inv = (size_t)LPC * LP * 8 + (size_t)(lay.total - lay.fwd_end) * 8 + (size_t)16 * 8;
    const size_t smem_cols = (size_t)L * CC * 8 + (size_t)KZROWS * CC * 8 + (size_t)lay.total * 8 + (size_t)2 * CC * NWC * 8 + 16;
    cudaError_t e = set_attrs<n>(smem_fwd, smem_inv, smem_cols);
    if (e != cudaSuccess) return (int)e;

    EncodeTiledFn enc = get_encode();
    if (!enc) return ASM_B200_E_DRIVER;
    CUtensorMap tmap[MAX_LANES], tmap_t[MAX_LANES], tmap_kz;   // per lane: pass-1 destination, column-pass destination
    const int rows = p0.N;
    const size_t lane_elems = sp ? sp->lane_elems : (size_t)g.chunk * rows * L;
    for (int l = 0; l < g.lanes; ++l) {
        if (!encode3d(enc, &tmap[l], p0.ws + l * lane_elems, 2 * (uint64_t)L, rows, g.chunk, 2 * CC, rows < 256 ? rows : 256))
            return ASM_B200_E_DRIVER;
        if (!sp) tmap_t[l] = tmap[l];
        else if (!encode3d(enc, &tmap_t[l], p0.ws + l * lane_elems + sp->s_elems, 2 * (uint64_t)L, rows, sp->tq, 2 * CC, rows < 256 ? rows : 256))
            return ASM_B200_E_DRIVER;
    }
    if (kz_in_smem(n)) {
        if (!encode3d(enc, &tmap_kz, const_cast<double*>(p0.kzt), 2 * (uint64_t)L, L / 2, 1, 2 * CC, (L / 2) < 256 ? (L / 2) : 256))
            return ASM_B200_E_DRIVER;
    } else {
        tmap_kz = tmap[0];
    }
    const int row_ctas_max = (1024 / ROW_THREADS) * sm_count();   // resident CTAs per SM (64 registers/thread)
    auto setup = [&](cudaStream_t s) {
        const int work = use_kz_table(n) ? (L / 2 + 1) * L : lay.total;
        int blocks = (work + 255) / 256;
        if (blocks > 2 * sm_count()) blocks = 2 * sm_count();
        k_setup_tables<<<blocks, 256, 0, s>>>(const_cast<float2*>(p0.tw), const_cast<double*>(p0.kzt), n, p0.s2,
                                              p0.inv_lambda * 0.15915494309189535);
    };
    auto pass = [&](int k, int lane, cudaStream_t s, const Params& p, int plane0, int nimg) {
        const int nlines = nimg * p.N;
        const int ntiles = (nlines + LPC - 1) / LPC;
        const int grid_rows = ntiles < row_ctas_max ? ntiles : row_ctas_max;
        if (k == 0) k_rows_fwd<n><<<grid_rows, ROW_THREADS, smem_fwd, s>>>(p, plane0, nlines, ntiles);
        else if (k == 1 && p.band_limit) k_cols<n, true><<<nimg * (L / CC), CC * TPL, smem_cols, s>>>(p, tmap_t[lane], tmap[lane], tmap_kz, plane0);
        else if (k == 1) k_cols<n><<<nimg * (L / CC), CC * TPL, smem_cols, s>>>(p, tmap_t[lane], tmap[lane], tmap_kz, plane0);
        else if (p.part) k_rows_inv<n, true><<<grid_rows, ROW_THREADS, smem_inv, s>>>(p, plane0, nlines, ntiles);
        else k_rows_inv<n><<<grid_rows, ROW_THREADS, smem_inv, s>>>(p, plane0, nlines, ntiles);
    };
    return run_chunks(p0, g, L, st, setup, pass, 0, sp);
}

#ifdef ASM_B200_TUNING
// FFT sizes <= 256: one persistent launch (resident.cuh)
template <int n>
static int launch_resident(const Params& p0, const Geometry& g, cudaStream_t st, int* ctl) {
    constexpr TwLayout lay = make_layout(n);
    constexpr int L = 1 << n;
    const size_t smem = ResidentCfg<n>::SMEM;
    static std::atomic<unsigned long long> done{0};
    static int occ[64] = {0};
    int dev;
    if (!attrs_done(done, &dev)) {
        cudaError_t e = set_smem(k_resident<n>, smem);
        if (e != cudaSuccess) return (int)e;
        int o = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, k_resident<n>, RES_THREADS, smem);
        if (e != cudaSuccess) return (int)e;
        if (dev >= 0 && dev < 64) occ[dev] = o;
        attrs_mark(done, dev);
    }
    const int o = (dev >= 0 && dev < 64 && occ[dev] > 0) ? occ[dev] : 1;
    int groups = g.chunk;
    if ((long long)groups * g.group > (long long)o * sm_count()) groups = o * sm_count() / g.group;   // every CTA of a group must be resident
    if (groups < 1) return ASM_B200_E_SHAPE;
    const bool prof = g_profile.load() != 0;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    const cudaError_t pending = cudaPeekAtLastError();
    {
        const int work = (L / 2 + 1) * L;
        int blocks = (work + 255) / 256;
        if (blocks > 2 * sm_count()) blocks = 2 * sm_count();
        k_setup_tables<<<blocks, 256, 0, st>>>(const_cast<float2*>(p0.tw), const_cast<double*>(p0.kzt), n, p0.s2,
                                               p0.inv_lambda * 0.15915494309189535);
        (void)lay;
    }
    cudaMemsetAsync(ctl, 0, sizeof(int) * (size_t)groups, st);
    if (prof) { for (auto& x : ev) cudaEventCreate(&x); cudaEventRecord(ev[0], st); }
    k_resident<n><<<groups * g.group, RES_THREADS, smem, st>>>(p0, ctl, g.group);
    g_launches.fetch_add(2);
    if (prof) {   // one kernel does all three passes: its time is reported in the column-pass slot
        cudaEventRecord(ev[1], st);
        cudaEventSynchronize(ev[1]);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev[0], ev[1]);
        { std::lock_guard<std::mutex> lk(g_prof_mu); g_prof_ms[1] += ms; }
        for (auto& x : ev) cudaEventDestroy(x);
    }
    if (pending == cudaSuccess) {
        const cudaError_t e = cudaPeekAtLastError();
        if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
    }
    return 0;
}

#endif  // ASM_B200_TUNING

#ifdef ASM_B200_TUNING
// FFT size 256: one launch, the sample lives in the shared memory of a 4-CTA cluster (cluster256.cuh)
static int launch_cluster256(const Params& p0, const Geometry& g, cudaStream_t st) {
    static std::atomic<unsigned long long> done{0};
    static int nclusters[64] = {0};
    int dev;
    if (!attrs_done(done, &dev)) {
        cudaError_t e = set_smem(k_cluster256, C256_SMEM);
        if (e != cudaSuccess) return (int)e;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(C256_CLUSTER * 64); cfg.blockDim = dim3(C256_THREADS); cfg.dynamicSmemBytes = C256_SMEM;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = C256_CLUSTER; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        int nc = 0;
        if (cudaOccupancyMaxActiveClusters(&nc, k_cluster256, &cfg) != cudaSuccess || nc < 1) { cudaGetLastError(); nc = sm_count() / C256_CLUSTER; }
        if (dev >= 0 && dev < 64) nclusters[dev] = nc;
        attrs_mark(done, dev);
    }
    int nc = (dev >= 0 && dev < 64 && nclusters[dev] > 0) ? nclusters[dev] : sm_count() / C256_CLUSTER;
    if (nc > p0.planes) nc = p0.planes;
    const bool prof = g_profile.load() != 0;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    const cudaError_t pending = cudaPeekAtLastError();
    constexpr int n = 8, L = 256;
    {
        const int work = (L / 2 + 1) * L;
        int blocks = (work + 255) / 256;
        if (blocks > 2 * sm_count()) blocks = 2 * sm_count();
        k_setup_tables<<<blocks, 256, 0, st>>>(const_cast<float2*>(p0.tw), const_cast<double*>(p0.kzt), n, p0.s2,
                                               p0.inv_lambda * 0.15915494309189535);
    }
    if (prof) { for (auto& x : ev) cudaEventCreate(&x); cudaEventRecord(ev[0], st); }
    k_cluster256<<<nc * C256_CLUSTER, C256_THREADS, C256_SMEM, st>>>(p0);
    g_launches.fetch_add(2);
    if (prof) {   // one kernel does all three passes: its time is reported in the column-pass slot
        cudaEventRecord(ev[1], st);
        cudaEventSynchronize(ev[1]);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev[0], ev[1]);
        { std::lock_guard<std::mutex> lk(g_prof_mu); g_prof_ms[1] += ms; }
        for (auto& x : ev) cudaEventDestroy(x);
    }
    (void)g;
    if (pending == cudaSuccess) {
        const cudaError_t e = cudaPeekAtLastError();
        if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
    }
    return 0;
}

#endif  // ASM_B200_TUNING

#ifdef ASM_B200_TUNING
// FFT size 1024: the 32-points-per-thread kernels of k32.cuh
template <int CC>
static void launch_k32_cols(const Params& p, int plane0, int nimg, cudaStream_t s) {
    const int per_sm = knob_cols_ctas() > 0 && knob_cols_ctas() < K32Cols<CC>::CTAS_PER_SM ? knob_cols_ctas() : K32Cols<CC>::CTAS_PER_SM;
    const int wk = nimg * (K32_L / CC), cap = per_sm * sm_count();
    const int grid = wk < cap ? wk : cap;
    if (p.P > 0) k32_cols<CC, true><<<grid, K32Cols<CC>::THREADS, K32Cols<CC>::SMEM, s>>>(p, plane0, nimg);
    else k32_cols<CC, false><<<grid, K32Cols<CC>::THREADS, K32Cols<CC>::SMEM, s>>>(p, plane0, nimg);
}

static int launch_32(const Params& p0, const Geometry& g, cudaStream_t st) {
    constexpr int L = K32_L;
    const size_t smem_rows = (size_t)K32_ROW_WARPS * K32_LP * 8 + (size_t)K32_TW * 8;
    const size_t smem_bulk = (size_t)K32_BULK_WARPS * (K32_L * 8 + K32_LP * 8) + (size_t)K32_TW * 8 + K32_BULK_WARPS * 8;
    {
        static std::atomic<unsigned long long> done{0};
        int dev;
        if (!attrs_done(done, &dev)) {
            cudaError_t e;
            if ((e = set_smem(k32_rows_fwd, smem_rows)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_rows_inv, smem_rows)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_rows_fwd_bulk<0, false>, smem_bulk)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_rows_fwd_bulk<0, true>, smem_bulk)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_rows_fwd_bulk<1, false>, smem_bulk)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_rows_fwd_bulk<1, true>, smem_bulk)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_rows_fwd_bulk<2, false>, smem_bulk)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_rows_fwd_bulk<2, true>, smem_bulk)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_rows_inv_bulk<false, false>, smem_bulk)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_rows_inv_bulk<false, true>, smem_bulk)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_rows_inv_bulk<true, false>, smem_bulk)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_rows_inv_bulk<true, true>, smem_bulk)) != cudaSuccess) return (int)e;
#ifdef ASM_B200_TUNING
            if ((e = set_smem(k32_rows_fwd_bulk<0, false, true>, smem_bulk)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_rows_inv_bulk<false, false, true>, smem_bulk)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_rows_inv_bulk<true, false, true>, smem_bulk)) != cudaSuccess) return (int)e;
#endif
            if ((e = set_smem(k32_cols<8, false>, K32Cols<8>::SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_cols<8, true>, K32Cols<8>::SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_cols<4, false>, K32Cols<4>::SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k32_cols<4, true>, K32Cols<4>::SMEM)) != cudaSuccess) return (int)e;
            attrs_mark(done, dev);
        }
    }
    const int bulk = knob_bulk();
    auto setup = [&](cudaStream_t s) {
        k32_setup<<<2 * sm_count(), 256, 0, s>>>(const_cast<float2*>(p0.tw), const_cast<double*>(p0.kzt), p0.s2,
                                                 p0.inv_lambda * 0.15915494309189535);
    };
    auto pass = [&](int k, int, cudaStream_t s, const Params& p, int plane0, int nimg) {
        const int nlines = nimg * p.N;
        const bool padded = p.P > 0;
        const int want = (nlines + K32_ROW_WARPS - 1) / K32_ROW_WARPS;
        const int grid_rows_max = knob_ldg_row_ctas() * sm_count();
        const int grid_rows = want < grid_rows_max ? want : grid_rows_max;
        const int want_bulk = (nlines + K32_BULK_WARPS - 1) / K32_BULK_WARPS;
        const int cap_bulk = sm_count() * knob_row_ctas();
        const int grid_bulk = want_bulk < cap_bulk ? want_bulk : cap_bulk;
        const int bt = 32 * K32_BULK_WARPS;
        // TMA bulk copies need 16-byte aligned rows; everything else takes the register-landing kernels
        const bool in_ok = (p.N % 4 == 0) && (((uintptr_t)p.in0 | (uintptr_t)p.in1) & 15) == 0;
        const bool fwd_bulk = (bulk & 1) && ((p.in_mode == ASM_B200_IN_COMPLEX && in_ok) || (p.in_mode == ASM_B200_IN_AMP_PHASE && in_ok) ||
                                             (p.in_mode == ASM_B200_IN_CONST_AMP_PHASE && (p.N % 4 == 0) && ((uintptr_t)p.in1 & 15) == 0));
        const bool inv_bulk = (bulk & 2) && (p.N % 4 == 0) && ((uintptr_t)p.out0 & 15) == 0 &&
                              (p.out_mode == ASM_B200_OUT_COMPLEX || (p.out_mode == ASM_B200_OUT_INTENSITY && !p.out1));
#ifdef ASM_B200_TUNING
        if ((bulk & 4) && !padded) {   // A/B: register stores instead of staged bulk stores
            if (k == 0 && fwd_bulk && p.in_mode == ASM_B200_IN_COMPLEX) { k32_rows_fwd_bulk<0, false, true><<<grid_bulk, bt, smem_bulk, s>>>(p, plane0, nlines); return; }
            if (k == 2 && inv_bulk) {
                if (p.out_mode == ASM_B200_OUT_INTENSITY) k32_rows_inv_bulk<true, false, true><<<grid_bulk, bt, smem_bulk, s>>>(p, plane0, nlines);
                else k32_rows_inv_bulk<false, false, true><<<grid_bulk, bt, smem_bulk, s>>>(p, plane0, nlines);
                return;
            }
        }
#endif
        if (k == 0 && fwd_bulk) {
            if (p.in_mode == ASM_B200_IN_COMPLEX) {
                if (padded) k32_rows_fwd_bulk<0, true><<<grid_bulk, bt, smem_bulk, s>>>(p, plane0, nlines);
                else k32_rows_fwd_bulk<0, false><<<grid_bulk, bt, smem_bulk, s>>>(p, plane0, nlines);
            } else if (p.in_mode == ASM_B200_IN_AMP_PHASE) {
                if (padded) k32_rows_fwd_bulk<1, true><<<grid_bulk, bt, smem_bulk, s>>>(p, plane0, nlines);
                else k32_rows_fwd_bulk<1, false><<<grid_bulk, bt, smem_bulk, s>>>(p, plane0, nlines);
            } else {
                if (padded) k32_rows_fwd_bulk<2, true><<<grid_bulk, bt, smem_bulk, s>>>(p, plane0, nlines);
                else k32_rows_fwd_bulk<2, false><<<grid_bulk, bt, smem_bulk, s>>>(p, plane0, nlines);
            }
        } else if (k == 0) {
            k32_rows_fwd<<<grid_rows, 32 * K32_ROW_WARPS, smem_rows, s>>>(p, plane0, nlines);
        } else if (k == 1) {
            if (g.cc == 4) launch_k32_cols<4>(p, plane0, nimg, s);
            else launch_k32_cols<8>(p, plane0, nimg, s);
        } else if (inv_bulk) {
            if (p.out_mode == ASM_B200_OUT_INTENSITY) {
                if (padded) k32_rows_inv_bulk<true, true><<<grid_bulk, bt, smem_bulk, s>>>(p, plane0, nlines);
                else k32_rows_inv_bulk<true, false><<<grid_bulk, bt, smem_bulk, s>>>(p, plane0, nlines);
            } else {
                if (padded) k32_rows_inv_bulk<false, true><<<grid_bulk, bt, smem_bulk, s>>>(p, plane0, nlines);
                else k32_rows_inv_bulk<false, false><<<grid_bulk, bt, smem_bulk, s>>>(p, plane0, nlines);
            }
        } else {
            k32_rows_inv<<<grid_rows, 32 * K32_ROW_WARPS, smem_rows, s>>>(p, plane0, nlines);
        }
    };
    return run_chunks(p0, g, L, st, setup, pass);
}
#endif  // ASM_B200_TUNING


// FFT size 1024, transposed intermediate (k32t.cuh): rows -> tile -> TMA tensor store | warp-private lines | TMA tensor
// load -> rows.  The workspace of a lane is [chunk][1024 u][N y] complex64, described by one tensor map per lane.
static int launch_32t(const Params& p0, const Geometry& g, cudaStream_t st, const StackPlan* sp = nullptr) {
    constexpr int L = K32_L;
    {
        static std::atomic<unsigned long long> done{0};
        int dev;
        if (!attrs_done(done, &dev)) {
            cudaError_t e;
#define K32T_SET(kern, bytes) if ((e = set_smem(kern, bytes)) != cudaSuccess) return (int)e;
            K32T_SET((k32t_rows_fwd<0, false>), K32T_FWD_SMEM) K32T_SET((k32t_rows_fwd<0, true>), K32T_FWD_SMEM)
            K32T_SET((k32t_rows_fwd<1, false>), K32T_FWD_SMEM) K32T_SET((k32t_rows_fwd<1, true>), K32T_FWD_SMEM)
            K32T_SET((k32t_rows_fwd<2, false>), K32T_FWD_SMEM) K32T_SET((k32t_rows_fwd<2, true>), K32T_FWD_SMEM)
            K32T_SET((k32t_rows_fwd<3, false>), K32T_FWD_SMEM) K32T_SET((k32t_rows_fwd<3, true>), K32T_FWD_SMEM)
            K32T_SET((k32t_rows_inv<0, false>), K32T_INV_SMEM) K32T_SET((k32t_rows_inv<0, true>), K32T_INV_SMEM)
            K32T_SET((k32t_rows_inv<1, false>), K32T_INV_SMEM) K32T_SET((k32t_rows_inv<1, true>), K32T_INV_SMEM)
            K32T_SET((k32t_rows_inv<2, false>), K32T_INV_SMEM) K32T_SET((k32t_rows_inv<2, true>), K32T_INV_SMEM)
            K32T_SET((k32t_lines<false>), K32T_LINES_SMEM) K32T_SET((k32t_lines<true>), K32T_LINES_SMEM)
            K32T_SET((k32t_lines<false, true>), K32T_LINES_SMEM) K32T_SET((k32t_lines<true, true>), K32T_LINES_SMEM)
#undef K32T_SET
            attrs_mark(done, dev);
        }
    }
    EncodeTiledFn enc = get_encode();
    if (!enc) return ASM_B200_E_DRIVER;
    CUtensorMap tmap[MAX_LANES], tmap_t[MAX_LANES];                 // per lane: pass-1 destination, pass-3 source
    const size_t lane_elems = sp ? sp->lane_elems : (size_t)g.chunk * p0.N * L;
    const CUtensorMapL2promotion promo = knob_promo() == 2 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B : knob_promo() == 1 ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B : CU_TENSOR_MAP_L2_PROMOTION_NONE;
    for (int l = 0; l < g.lanes; ++l) {
        if (!encode3d(enc, &tmap[l], p0.ws + l * lane_elems, 2 * (uint64_t)p0.N, L, g.chunk, 16, 256, CU_TENSOR_MAP_SWIZZLE_64B, promo))
            return ASM_B200_E_DRIVER;
        if (!sp) tmap_t[l] = tmap[l];
        else if (!encode3d(enc, &tmap_t[l], p0.ws + l * lane_elems + sp->s_elems, 2 * (uint64_t)p0.N, L, sp->tq, 16, 256, CU_TENSOR_MAP_SWIZZLE_64B, promo))
            return ASM_B200_E_DRIVER;
    }
    auto setup = [&](cudaStream_t s) {
        k32t_setup<<<2 * sm_count(), 256, 0, s>>>(const_cast<float2*>(p0.tw), reinterpret_cast<float2*>(const_cast<double*>(p0.kzt)),
                                                  p0.s2, p0.inv_lambda * 0.15915494309189535);
    };
    auto pass = [&](int k, int lane, cudaStream_t s, const Params& p, int plane0, int nimg) {
        const bool padded = p.P > 0;
        const int ngroups = nimg * p.N / 8;
        const int cap_rows = K32T_ROW_CTAS * sm_count();
        const int grid_rows = ngroups < cap_rows ? ngroups : cap_rows;
        const int bt = 32 * K32T_ROW_WARPS;
        const bool in_ok = (p.N % 4 == 0) && (((uintptr_t)p.in0 | (uintptr_t)p.in1) & 15) == 0;
        const bool fwd_bulk = (knob_bulk() & 1) &&
                              ((p.in_mode == ASM_B200_IN_COMPLEX && in_ok) || (p.in_mode == ASM_B200_IN_AMP_PHASE && in_ok) ||
                               (p.in_mode == ASM_B200_IN_CONST_AMP_PHASE && (p.N % 4 == 0) && ((uintptr_t)p.in1 & 15) == 0));
        const bool inv_bulk = (knob_bulk() & 2) && (p.N % 4 == 0) && ((uintptr_t)p.out0 & 15) == 0 &&
                              (p.out_mode == ASM_B200_OUT_COMPLEX || (p.out_mode == ASM_B200_OUT_INTENSITY && !p.out1)) &&
                              p.out0 && !p.part;                     // focal-stack moments: the register-store kernel
        if (k == 0) {
            const int in = !fwd_bulk ? 3 : p.in_mode == ASM_B200_IN_COMPLEX ? 0 : p.in_mode == ASM_B200_IN_AMP_PHASE ? 1 : 2;
#define K32T_FWD(IN) { if (padded) k32t_rows_fwd<IN, true><<<grid_rows, bt, K32T_FWD_SMEM, s>>>(p, tmap[lane], plane0, ngroups); \
                       else k32t_rows_fwd<IN, false><<<grid_rows, bt, K32T_FWD_SMEM, s>>>(p, tmap[lane], plane0, ngroups); }
            if (in == 0) K32T_FWD(0) else if (in == 1) K32T_FWD(1) else if (in == 2) K32T_FWD(2) else K32T_FWD(3)
#undef K32T_FWD
        } else if (k == 1) {
            const int nlines = nimg * L;
            const int want = (nlines + K32T_LINE_WARPS - 1) / K32T_LINE_WARPS, cap = K32T_LINE_CTAS * sm_count();
            const int grid = want < cap ? want : cap;
#define K32T_LINES(PAD, BL) k32t_lines<PAD, BL><<<grid, 32 * K32T_LINE_WARPS, K32T_LINES_SMEM, s>>>(p, plane0, nlines);
            if (p.band_limit) { if (padded) K32T_LINES(true, true) else K32T_LINES(false, true) }
            else { if (padded) K32T_LINES(true, false) else K32T_LINES(false, false) }
#undef K32T_LINES
        } else {
            const int out = !inv_bulk ? 2 : p.out_mode == ASM_B200_OUT_INTENSITY ? 1 : 0;
            const int grid_inv = ngroups / 2 < cap_rows ? ngroups / 2 : cap_rows;   // pairs of groups
#define K32T_INV(OUT) { if (padded) k32t_rows_inv<OUT, true><<<grid_inv, bt, K32T_INV_SMEM, s>>>(p, tmap_t[lane], plane0, ngroups); \
                        else k32t_rows_inv<OUT, false><<<grid_inv, bt, K32T_INV_SMEM, s>>>(p, tmap_t[lane], plane0, ngroups); }
            if (out == 0) K32T_INV(0) else if (out == 1) K32T_INV(1) else K32T_INV(2)
#undef K32T_INV
        }
    };
    return run_chunks(p0, g, L, st, setup, pass, 32, sp);
}

#ifdef ASM_B200_TUNING
static int launch_64t(const Params& p0, const Geometry& g, cudaStream_t st);
#endif

// FFT size 2048: k64.cuh.  The warp-pair bulk row kernels run when both row passes qualify (complex64 or
// amplitude / phase in, complex64 or |U|^2 out, 16-byte aligned rows); otherwise the generic row kernels run, with their
// digit-reversed column order and a kappa table in that order.  The column kernel is the same in both cases.
static int launch_64(const Params& p0, const Geometry& g, cudaStream_t st, const StackPlan* sp = nullptr) {
    constexpr int n = 11, L = K64_L, TPL = L / 16, LPC = ROW_THREADS / TPL, LP = RowLayout::line_elems(L);
    constexpr TwLayout lay = make_layout(n);
    const size_t smem_fwd = (size_t)LPC * LP * 8 + (size_t)lay.fwd_end * 8;
    const size_t smem_inv = (size_t)LPC * LP * 8 + (size_t)(lay.total - lay.fwd_end) * 8 + (size_t)16 * 8;
    {
        static std::atomic<unsigned long long> done{0};
        int dev;
        if (!attrs_done(done, &dev)) {
            cudaError_t e;
            if ((e = set_smem(k_rows_fwd<n>, smem_fwd)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k_rows_inv<n>, smem_inv)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k_rows_inv<n, true>, smem_inv)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_rows_fwd_bulk<0, false>, K64_ROWS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_rows_fwd_bulk<0, true>, K64_ROWS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_rows_fwd_bulk<1, false>, K64_ROWS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_rows_fwd_bulk<1, true>, K64_ROWS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_rows_fwd_bulk<2, false>, K64_ROWS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_rows_fwd_bulk<2, true>, K64_ROWS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_rows_inv_bulk<false, false>, K64_ROWS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_rows_inv_bulk<false, true>, K64_ROWS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_rows_inv_bulk<true, false>, K64_ROWS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_rows_inv_bulk<true, true>, K64_ROWS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_cols<false, false>, K64_COLS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_cols<true, false>, K64_COLS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_cols<false, true>, K64_COLS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_cols<true, true>, K64_COLS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_cols<false, false, true>, K64_COLS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_cols<true, false, true>, K64_COLS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_cols<false, true, true>, K64_COLS_SMEM)) != cudaSuccess) return (int)e;
            if ((e = set_smem(k64_cols<true, true, true>, K64_COLS_SMEM)) != cudaSuccess) return (int)e;
            attrs_mark(done, dev);
        }
    }
    const Params& q = p0;
    const bool in_ok = (q.N % 4 == 0) && (((uintptr_t)q.in0 | (uintptr_t)q.in1) & 15) == 0;
    const bool fwd_bulk = (q.in_mode == ASM_B200_IN_COMPLEX && in_ok) || (q.in_mode == ASM_B200_IN_AMP_PHASE && in_ok) ||
                          (q.in_mode == ASM_B200_IN_CONST_AMP_PHASE && (q.N % 4 == 0) && ((uintptr_t)q.in1 & 15) == 0);
    const bool inv_bulk = (q.N % 4 == 0) && ((uintptr_t)q.out0 & 15) == 0 &&
                          (q.out_mode == ASM_B200_OUT_COMPLEX || (q.out_mode == ASM_B200_OUT_INTENSITY && !q.out1)) &&
                          q.out0 && !(sp && sp->mom);                // focal-stack moments: the generic row kernels
    const bool bulk = fwd_bulk && inv_bulk && knob_bulk() != 0;
#ifdef ASM_B200_TUNING
    if (bulk && knob_k64t() && q.N % 16 == 0) return q.band_limit ? ASM_B200_E_MODE : launch_64t(p0, g, st);   // k64t.cuh has no band limit
#endif
    const bool padded = q.P > 0;
    auto setup = [&](cudaStream_t s) {
        if (bulk) {
            k64_setup<<<2 * sm_count(), 256, 0, s>>>(const_cast<float2*>(q.tw32), const_cast<double*>(q.kzt), q.s2, q.inv_lambda * 0.15915494309189535, 1);
        } else {
            k_setup_tables<<<2 * sm_count(), 256, 0, s>>>(const_cast<float2*>(q.tw), const_cast<double*>(q.kzt), n, q.s2, q.inv_lambda * 0.15915494309189535);
            k64_setup<<<2, 256, 0, s>>>(const_cast<float2*>(q.tw32), nullptr, q.s2, 0.0);
        }
    };
    const int row_ctas_max = (1024 / ROW_THREADS) * sm_count();
    auto pass = [&](int k, int, cudaStream_t s, const Params& p, int plane0, int nimg) {
        const int nlines = nimg * p.N;
        if (k == 1) {
            const int wk = nimg * (L / K64_CC), cap = 2 * sm_count();
            const int grid = wk < cap ? wk : cap;
#define K64_COLS(PAD, PAIRS) { if (p.band_limit) k64_cols<PAD, PAIRS, true><<<grid, 64 * K64_CC, K64_COLS_SMEM, s>>>(p, plane0, nimg); \
                                else k64_cols<PAD, PAIRS><<<grid, 64 * K64_CC, K64_COLS_SMEM, s>>>(p, plane0, nimg); }
            if (bulk) {   // the kappa table of the warp-pair row kernels holds (hi, lo) pairs
                if (padded) K64_COLS(true, true) else K64_COLS(false, true)
            } else {
                if (padded) K64_COLS(true, false) else K64_COLS(false, false)
            }
#undef K64_COLS
            return;
        }
        if (!bulk) {
            const int ntiles = (nlines + LPC - 1) / LPC;
            const int grid_rows = ntiles < row_ctas_max ? ntiles : row_ctas_max;
            if (k == 0) k_rows_fwd<n><<<grid_rows, ROW_THREADS, smem_fwd, s>>>(p, plane0, nlines, ntiles);
            else if (p.part) k_rows_inv<n, true><<<grid_rows, ROW_THREADS, smem_inv, s>>>(p, plane0, nlines, ntiles);
            else k_rows_inv<n><<<grid_rows, ROW_THREADS, smem_inv, s>>>(p, plane0, nlines, ntiles);
            return;
        }
        const int want = (nlines + K64_PAIRS - 1) / K64_PAIRS, cap = 2 * sm_count();
        const int grid = want < cap ? want : cap;
        const int bt = 64 * K64_PAIRS;
        if (k == 0) {
            if (p.in_mode == ASM_B200_IN_COMPLEX) {
                if (padded) k64_rows_fwd_bulk<0, true><<<grid, bt, K64_ROWS_SMEM, s>>>(p, plane0, nlines);
                else k64_rows_fwd_bulk<0, false><<<grid, bt, K64_ROWS_SMEM, s>>>(p, plane0, nlines);
            } else if (p.in_mode == ASM_B200_IN_AMP_PHASE) {
                if (padded) k64_rows_fwd_bulk<1, true><<<grid, bt, K64_ROWS_SMEM, s>>>(p, plane0, nlines);
                else k64_rows_fwd_bulk<1, false><<<grid, bt, K64_ROWS_SMEM, s>>>(p, plane0, nlines);
            } else {
                if (padded) k64_rows_fwd_bulk<2, true><<<grid, bt, K64_ROWS_SMEM, s>>>(p, plane0, nlines);
                else k64_rows_fwd_bulk<2, false><<<grid, bt, K64_ROWS_SMEM, s>>>(p, plane0, nlines);
            }
        } else {
            if (p.out_mode == ASM_B200_OUT_INTENSITY) {
                if (padded) k64_rows_inv_bulk<true, true><<<grid, bt, K64_ROWS_SMEM, s>>>(p, plane0, nlines);
                else k64_rows_inv_bulk<true, false><<<grid, bt, K64_ROWS_SMEM, s>>>(p, plane0, nlines);
            } else {
                if (padded) k64_rows_inv_bulk<false, true><<<grid, bt, K64_ROWS_SMEM, s>>>(p, plane0, nlines);
                else k64_rows_inv_bulk<false, false><<<grid, bt, K64_ROWS_SMEM, s>>>(p, plane0, nlines);
            }
        }
    };
    return run_chunks(p0, g, L, st, setup, pass, 0, sp);
}

// every even size that is not a power of two: four matrix products (dft_any.cuh), chunks in sequence on the caller's stream.
// A focal stack (p0.kst = K) runs the whole transform once per plane (sample q / K), with moments reduced into `mom`.
static int launch_dft(const Params& p0, const DftGeom& g, unsigned char* ws, cudaStream_t st, double* mom = nullptr) {
    float2* A = reinterpret_cast<float2*>(ws);
    float2* S = reinterpret_cast<float2*>(ws + g.a_bytes);
    float2* T1 = reinterpret_cast<float2*>(ws + g.a_bytes + g.s_bytes);
    float2* T2 = reinterpret_cast<float2*>(ws + g.a_bytes + g.s_bytes + g.t1_bytes);
    float2* T3 = reinterpret_cast<float2*>(ws + g.a_bytes + g.s_bytes + g.t1_bytes + g.t2_bytes);
    const cudaError_t pending = cudaPeekAtLastError();
    const int N = g.N, M = g.M;
    int blocks = (N * M + 255) / 256;
    if (blocks > 4 * sm_count()) blocks = 4 * sm_count();
    k_dft_setup<<<blocks, 256, 0, st>>>(A, S, N, M, g.P, p0.adj);
    unsigned long long launches = 1;
    auto tiles = [](int x) { return (unsigned)((x + DFT_T - 1) / DFT_T); };
    for (int plane0 = 0; plane0 < p0.planes; plane0 += g.chunk) {
        const int nimg = (p0.planes - plane0 < g.chunk) ? p0.planes - plane0 : g.chunk;
        k_dft_mm<0><<<dim3(tiles(M), tiles(N), nimg), 256, 0, st>>>(p0, A, S, T1, T2, T3, plane0, N, M);
        k_dft_mm<1><<<dim3(tiles(M), tiles(M), nimg), 256, 0, st>>>(p0, A, S, T1, T2, T3, plane0, N, M);
        k_dft_mm<2><<<dim3(tiles(M), tiles(N), nimg), 256, 0, st>>>(p0, A, S, T1, T2, T3, plane0, N, M);
        k_dft_mm<3><<<dim3(tiles(N), tiles(N), nimg), 256, 0, st>>>(p0, A, S, T1, T2, T3, plane0, N, M);
        launches += 4;
        if (p0.part) {
            k_moments_reduce<<<(nimg + 7) / 8, 256, 0, st>>>(p0.part, mom, (int)(tiles(N) * tiles(N)), nimg, plane0);
            launches += 1;
        }
        if (pending == cudaSuccess && cudaPeekAtLastError() != cudaSuccess) break;
    }
    g_launches.fetch_add(launches);
    if (pending == cudaSuccess) {
        const cudaError_t e = cudaPeekAtLastError();
        if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
    }
    return 0;
}

#ifdef ASM_B200_TUNING
// FFT size 2048, transposed intermediate (k64t.cuh); only the modes whose rows move by TMA bulk copies
static int launch_64t(const Params& p0, const Geometry& g, cudaStream_t st) {
    constexpr int L = K64_L;
    {
        static std::atomic<unsigned long long> done{0};
        int dev;
        if (!attrs_done(done, &dev)) {
            cudaError_t e;
#define K64T_SET(kern, bytes) if ((e = set_smem(kern, bytes)) != cudaSuccess) return (int)e;
            K64T_SET((k64t_rows_fwd<0, false>), K64T_ROWS_SMEM) K64T_SET((k64t_rows_fwd<0, true>), K64T_ROWS_SMEM)
            K64T_SET((k64t_rows_fwd<1, false>), K64T_ROWS_SMEM) K64T_SET((k64t_rows_fwd<1, true>), K64T_ROWS_SMEM)
            K64T_SET((k64t_rows_fwd<2, false>), K64T_ROWS_SMEM) K64T_SET((k64t_rows_fwd<2, true>), K64T_ROWS_SMEM)
            K64T_SET((k64t_rows_inv<0, false>), K64T_ROWS_SMEM) K64T_SET((k64t_rows_inv<0, true>), K64T_ROWS_SMEM)
            K64T_SET((k64t_rows_inv<1, false>), K64T_ROWS_SMEM) K64T_SET((k64t_rows_inv<1, true>), K64T_ROWS_SMEM)
            K64T_SET((k64t_lines<false>), K64T_LINES_SMEM) K64T_SET((k64t_lines<true>), K64T_LINES_SMEM)
#undef K64T_SET
            attrs_mark(done, dev);
        }
    }
    EncodeTiledFn enc = get_encode();
    if (!enc) return ASM_B200_E_DRIVER;
    CUtensorMap tmap[MAX_LANES];
    const size_t lane_elems = (size_t)g.chunk * p0.N * L;
    for (int l = 0; l < g.lanes; ++l)
        if (!encode3d(enc, &tmap[l], p0.ws + l * lane_elems, 2 * (uint64_t)p0.N, L, g.chunk, 8, 256, CU_TENSOR_MAP_SWIZZLE_32B,
                      CU_TENSOR_MAP_L2_PROMOTION_NONE))
            return ASM_B200_E_DRIVER;
    auto setup = [&](cudaStream_t s) {
        k64t_setup<<<2 * sm_count(), 256, 0, s>>>(const_cast<float2*>(p0.tw32), reinterpret_cast<float2*>(const_cast<double*>(p0.kzt)),
                                                  p0.s2, p0.inv_lambda * 0.15915494309189535);
    };
    auto pass = [&](int k, int lane, cudaStream_t s, const Params& p, int plane0, int nimg) {
        const bool padded = p.P > 0;
        const int ngroups = nimg * p.N / 4, cap = 2 * sm_count(), bt = 64 * K64T_PAIRS;
        if (k == 0) {
            const int grid = ngroups < cap ? ngroups : cap;
            const int in = p.in_mode == ASM_B200_IN_COMPLEX ? 0 : p.in_mode == ASM_B200_IN_AMP_PHASE ? 1 : 2;
#define K64T_FWD(IN) { if (padded) k64t_rows_fwd<IN, true><<<grid, bt, K64T_ROWS_SMEM, s>>>(p, tmap[lane], plane0, ngroups); \
                       else k64t_rows_fwd<IN, false><<<grid, bt, K64T_ROWS_SMEM, s>>>(p, tmap[lane], plane0, ngroups); }
            if (in == 0) K64T_FWD(0) else if (in == 1) K64T_FWD(1) else K64T_FWD(2)
#undef K64T_FWD
        } else if (k == 1) {
            const int nlines = nimg * L;
            const int want = (nlines + K64T_PAIRS - 1) / K64T_PAIRS;
            const int grid = want < cap ? want : cap;
            if (padded) k64t_lines<true><<<grid, bt, K64T_LINES_SMEM, s>>>(p, plane0, nlines);
            else k64t_lines<false><<<grid, bt, K64T_LINES_SMEM, s>>>(p, plane0, nlines);
        } else {
            const int nquads = ngroups / 4;
            const int grid = nquads < cap ? nquads : cap;
#define K64T_INV(OUT) { if (padded) k64t_rows_inv<OUT, true><<<grid, bt, K64T_ROWS_SMEM, s>>>(p, tmap[lane], plane0, ngroups); \
                        else k64t_rows_inv<OUT, false><<<grid, bt, K64T_ROWS_SMEM, s>>>(p, tmap[lane], plane0, ngroups); }
            if (p.out_mode == ASM_B200_OUT_INTENSITY) K64T_INV(1) else K64T_INV(0)
#undef K64T_INV
        }
    };
    return run_chunks(p0, g, L, st, setup, pass, 64);
}

#endif  // ASM_B200_TUNING

static int check_device() {
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return ASM_B200_E_DEVICE;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return ASM_B200_E_DEVICE;
    return major == 10 ? 0 : ASM_B200_E_DEVICE;
}

static int run(Params p, int B, int C, int N, int pad, double lambda, double px, void* workspace, size_t workspace_bytes,
               void* stream) {
    if (B <= 0 || C <= 0) return ASM_B200_E_SHAPE;
    Geometry g;
    DftGeom dg;
    const bool fft = make_geometry(B * C, N, pad, &g);
    if (!fft && !dft_geometry(B * C, N, pad, &dg)) return ASM_B200_E_SHAPE;
    if (!(lambda > 0.0) || !(px > 0.0) || !isfinite(lambda) || !isfinite(px)) return ASM_B200_E_OPTICS;
    if (!workspace || ((uintptr_t)workspace & 255) || workspace_bytes < (fft ? workspace_need(g) : dft_workspace(dg))) return ASM_B200_E_WORKSPACE;
    if (!p.in0 || !p.out0 || !p.z) return ASM_B200_E_NULL;
    int rc = check_device();
    if (rc) return rc;
    if (!fft) {   // even, not a power of two: matrix-product path
        p.planes = B * C; p.C = C; p.N = N; p.M = dg.M; p.P = dg.P;
        const double sd = lambda / ((double)dg.M * px);
        p.s2 = sd * sd; p.lambda = lambda; p.inv_lambda = 1.0 / lambda;
        p.S = (double)dg.M * px;
        p.inv_m2 = 1.0f / ((float)dg.M * (float)dg.M);
        return launch_dft(p, dg, reinterpret_cast<unsigned char*>(workspace), reinterpret_cast<cudaStream_t>(stream));
    }
    p.planes = B * C; p.C = C; p.N = N; p.M = g.M; p.P = g.P;
    p.tw = reinterpret_cast<const float2*>(workspace);
    p.tw32 = p.tw + (g.n == 11 ? make_layout(11).total : 0);
    p.kzt = g.kz_bytes ? reinterpret_cast<const double*>(reinterpret_cast<unsigned char*>(workspace) + g.tw_bytes) : nullptr;
    int* ctl = reinterpret_cast<int*>(reinterpret_cast<unsigned char*>(workspace) + g.tw_bytes + g.kz_bytes);
    p.ws = reinterpret_cast<float2*>(reinterpret_cast<unsigned char*>(workspace) + g.tw_bytes + g.kz_bytes + g.ctl_bytes);
    const double s = lambda / ((double)g.M * px);
    p.s2 = s * s;
    p.lambda = lambda;
    p.inv_lambda = 1.0 / lambda;
    p.S = (double)g.M * px;
    p.inv_m2 = 1.0f / ((float)g.M * (float)g.M);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
#ifdef ASM_B200_TUNING
    // the measured alternatives of tuning builds (resident.cuh, cluster256.cuh, k32_cols.cuh) have no band limit
    if (p.band_limit && (g.resident || (g.n == 8 && knob_cluster256()) || (g.n == 10 && !knob_k32t()))) return ASM_B200_E_MODE;
#endif
#if defined(ASM_B200_TUNING) && !defined(ASM_B200_ONLY_1024)
    if (g.resident) {
        switch (g.n) {
            case 5: return launch_resident<5>(p, g, st, ctl);
            case 6: return launch_resident<6>(p, g, st, ctl);
            case 7: return launch_resident<7>(p, g, st, ctl);
            case 8: return launch_resident<8>(p, g, st, ctl);
            case 9: return launch_resident<9>(p, g, st, ctl);
        }
    }
#endif
#ifdef ASM_B200_ONLY_1024    /* tools/ A/B builds: compile the FFT-1024 path only (fast rebuilds) */
    if (g.n == 10) return knob_k32t() ? launch_32t(p, g, st) : launch_32(p, g, st);   /* ONLY_1024 implies TUNING */
    return ASM_B200_E_SHAPE;
#else
#ifdef ASM_B200_TUNING
    if (g.n == 8 && knob_cluster256()) return launch_cluster256(p, g, st);
    if (g.n == 10 && !knob_k32t()) return launch_32(p, g, st);
#endif
    switch (g.n) {
        case 5: return launch_n<5>(p, g, st);
        case 6: return launch_n<6>(p, g, st);
        case 7: return launch_n<7>(p, g, st);
        case 8: return launch_n<8>(p, g, st);
        case 9: return launch_n<9>(p, g, st);
        case 10: return launch_32t(p, g, st);
        case 11: return knob_k64() ? launch_64(p, g, st) : launch_n<11>(p, g, st);
        case 12: return launch_n<12>(p, g, st);
    }
#endif
    return ASM_B200_E_SHAPE;
}

}  // namespace asmb

// ---------------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------------
using namespace asmb;

extern "C" int asm_b200_abi_version(void) { return ASM_B200_ABI_VERSION; }

extern "C" const char* asm_b200_strerror(int code) {
    switch (code) {
        case 0: return "ok";
        case ASM_B200_E_NULL: return "asm_b200: a required pointer is NULL";
        case ASM_B200_E_SHAPE: return "asm_b200: unsupported shape (square N: a power of two with 32 <= FFT size <= 4096, or any other even N with FFT size <= 2048; B, C > 0)";
        case ASM_B200_E_MODE: return "asm_b200: unknown or inconsistent in_mode / out_mode, or band_limit not 0 or 1";
        case ASM_B200_E_WORKSPACE: return "asm_b200: workspace too small or not 256-byte aligned";
        case ASM_B200_E_OPTICS: return "asm_b200: wavelength and pixel size must be finite and positive";
        case ASM_B200_E_DRIVER: return "asm_b200: cuTensorMapEncodeTiled unavailable or failed";
        case ASM_B200_E_DEVICE: return "asm_b200: current CUDA device is not compute capability 10.x (B200)";
    }
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "asm_b200: unknown error";
}

extern "C" unsigned long long asm_b200_launch_count(void) { return g_launches.load(); }

extern "C" void asm_b200_profile(int enable, double* ms3) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    if (ms3) for (int k = 0; k < 3; ++k) ms3[k] = g_prof_ms[k];
    if (enable >= 0) { g_profile.store(enable); for (double& x : g_prof_ms) x = 0.0; }
}

extern "C" size_t asm_b200_workspace_bytes(int B, int C, int N, int pad) {
    Geometry g;
    DftGeom dg;
    if (B <= 0 || C <= 0) return 0;
    if (make_geometry(B * C, N, pad, &g)) return workspace_need(g);
    return dft_geometry(B * C, N, pad, &dg) ? dft_workspace(dg) : 0;
}

// ---------------------------------------------------------------------------------------------------
// focal stack
// ---------------------------------------------------------------------------------------------------
// Chunking: S (chunk samples) + T (tq planes) + partials of every lane stay within the in-flight budget of a single call,
// so S is read from L2 by every group of its sample.  The plan depends on (B, K, N, pad) only.
static bool make_stack_plan(int B, int K, int N, int pad, Geometry* g, StackPlan* sp) {
    if (B <= 0 || K <= 0 || !make_geometry(B, N, pad, g)) return false;
    const int n = g->n, M = g->M;
    int lanes = knob_lanes() != 3 ? knob_lanes() : default_lanes(n, pad != 0);
    lanes = lanes < 1 ? 1 : (lanes > MAX_LANES ? MAX_LANES : lanes);
    const size_t budget = knob_chunk_mb() > 0 ? (size_t)knob_chunk_mb() << 20 : default_budget(n, pad != 0);
    const size_t lane_budget = budget / lanes, img = g->img_bytes;
    const int R = n == 10 ? N : N * (M / 512 > 1 ? M / 512 : 1);   // partials per plane: k32t_rows_inv / k_rows_inv
    const size_t per_plane = img + (size_t)R * 3 * sizeof(double);
    int spc = 1, tq;
    if (img + (size_t)K * per_plane <= lane_budget) {              // whole stacks of several samples per chunk
        spc = (int)(lane_budget / (img + (size_t)K * per_plane));
        if (spc > B) spc = B;
        tq = spc * K;
    } else {                                                       // one sample per chunk, its planes in balanced groups
        const long long gmax = lane_budget > img + per_plane ? (long long)((lane_budget - img) / per_plane) : 1;
        const long long ng = (K + gmax - 1) / gmax;
        tq = (int)((K + ng - 1) / ng);
    }
    const int nchunks = (B + spc - 1) / spc;
    if (lanes > nchunks) lanes = nchunks;
    g->chunk = spc; g->lanes = lanes;
    sp->K = K; sp->tq = tq; sp->R = R; sp->mom = nullptr;
    sp->s_elems = (size_t)spc * N * M;
    sp->t_elems = (size_t)tq * N * M;
    sp->lane_elems = sp->s_elems + sp->t_elems + align_up((size_t)tq * R * 3, 32);   // doubles, one float2 element each
    return true;
}
static size_t stack_workspace_need(const Geometry& g, const StackPlan& sp) {
    return g.tw_bytes + g.kz_bytes + sp.lane_elems * sizeof(float2) * g.lanes;
}
static size_t dft_stack_partials(const DftGeom& dg) {
    const size_t t = (size_t)((dg.N + DFT_T - 1) / DFT_T);
    return align_up((size_t)dg.chunk * t * t * 3 * sizeof(double), 256);
}

static bool needs_in1(int in_mode) { return in_mode == ASM_B200_IN_AMP_PHASE || in_mode == ASM_B200_IN_COT_FIELD || in_mode == ASM_B200_IN_CONST_AMP_PHASE; }

extern "C" int asm_b200_forward(const void* in0, const void* in1, const void* z, int z_dtype, void* out0, void* out1,
                                int B, int C, int N, int pad, int in_mode, int out_mode, double lambda, double px,
                                float in_scale, float out_scale, void* workspace, size_t workspace_bytes, void* stream) {
    return asm_b200_forward_bl(in0, in1, z, z_dtype, out0, out1, B, C, N, pad, in_mode, out_mode, lambda, px, in_scale,
                               out_scale, workspace, workspace_bytes, stream, 0);
}

extern "C" int asm_b200_forward_bl(const void* in0, const void* in1, const void* z, int z_dtype, void* out0, void* out1,
                                   int B, int C, int N, int pad, int in_mode, int out_mode, double lambda, double px,
                                   float in_scale, float out_scale, void* workspace, size_t workspace_bytes, void* stream,
                                   int band_limit) {
    if (band_limit != 0 && band_limit != 1) return ASM_B200_E_MODE;
    if (in_mode < 0 || in_mode > ASM_B200_IN_CONST_AMP_PHASE || out_mode < 0 || out_mode > ASM_B200_OUT_ABSANG_CAT) return ASM_B200_E_MODE;
    if (z_dtype != ASM_B200_Z_F32 && z_dtype != ASM_B200_Z_F64) return ASM_B200_E_MODE;
    if ((out_mode == ASM_B200_OUT_REIM_CAT || out_mode == ASM_B200_OUT_ABSANG_CAT) && C != 1) return ASM_B200_E_MODE;
    if (needs_in1(in_mode) && !in1) return ASM_B200_E_NULL;
    if (out_mode == ASM_B200_OUT_ABS_ANGLE && !out1) return ASM_B200_E_NULL;
    Params p{};
    p.in0 = in0; p.in1 = in1; p.out0 = out0; p.out1 = out1; p.z = z; p.z_f64 = z_dtype;
    p.in_mode = in_mode; p.out_mode = out_mode; p.h_mode = H_FWD; p.adj = 0; p.band_limit = band_limit;
    p.in_scale = in_scale; p.out_scale = out_scale;
    return run(p, B, C, N, pad, lambda, px, workspace, workspace_bytes, stream);
}

extern "C" int asm_b200_adjoint(const void* in0, const void* in1, const void* z, int z_dtype, const void* aux0,
                                const void* aux1, void* out0, void* out1, int B, int C, int N, int pad, int in_mode,
                                int out_mode, double lambda, double px, float in_scale, void* workspace,
                                size_t workspace_bytes, void* stream) {
    return asm_b200_adjoint_bl(in0, in1, z, z_dtype, aux0, aux1, out0, out1, B, C, N, pad, in_mode, out_mode, lambda, px,
                               in_scale, workspace, workspace_bytes, stream, 0);
}

extern "C" int asm_b200_adjoint_bl(const void* in0, const void* in1, const void* z, int z_dtype, const void* aux0,
                                   const void* aux1, void* out0, void* out1, int B, int C, int N, int pad, int in_mode,
                                   int out_mode, double lambda, double px, float in_scale, void* workspace,
                                   size_t workspace_bytes, void* stream, int band_limit) {
    if (band_limit != 0 && band_limit != 1) return ASM_B200_E_MODE;
    if (in_mode != ASM_B200_IN_COMPLEX && in_mode != ASM_B200_IN_COT_FIELD) return ASM_B200_E_MODE;
    if (out_mode != ASM_B200_OUT_COMPLEX && out_mode != ASM_B200_OUT_GRAD_AP) return ASM_B200_E_MODE;
    if (z_dtype != ASM_B200_Z_F32 && z_dtype != ASM_B200_Z_F64) return ASM_B200_E_MODE;
    if (needs_in1(in_mode) && !in1) return ASM_B200_E_NULL;
    if (out_mode == ASM_B200_OUT_GRAD_AP && (!aux0 || !aux1 || !out1)) return ASM_B200_E_NULL;
    Params p{};
    p.in0 = in0; p.in1 = in1; p.aux0 = aux0; p.aux1 = aux1; p.out0 = out0; p.out1 = out1; p.z = z; p.z_f64 = z_dtype;
    p.in_mode = in_mode; p.out_mode = out_mode; p.h_mode = H_CONJ; p.adj = 1; p.band_limit = band_limit;
    p.in_scale = in_scale; p.out_scale = 1.f;
    return run(p, B, C, N, pad, lambda, px, workspace, workspace_bytes, stream);
}

extern "C" int asm_b200_grad_z(const void* in0, const void* in1, const void* z, int z_dtype, const void* cot0,
                               const void* cot1, int cot_mode, double* grad_z, int B, int C, int N, int pad, int in_mode,
                               double lambda, double px, float in_scale, void* workspace, size_t workspace_bytes,
                               void* stream) {
    return asm_b200_grad_z_bl(in0, in1, z, z_dtype, cot0, cot1, cot_mode, grad_z, B, C, N, pad, in_mode, lambda, px,
                              in_scale, workspace, workspace_bytes, stream, 0);
}

extern "C" int asm_b200_grad_z_bl(const void* in0, const void* in1, const void* z, int z_dtype, const void* cot0,
                                  const void* cot1, int cot_mode, double* grad_z, int B, int C, int N, int pad, int in_mode,
                                  double lambda, double px, float in_scale, void* workspace, size_t workspace_bytes,
                                  void* stream, int band_limit) {
    if (band_limit != 0 && band_limit != 1) return ASM_B200_E_MODE;
    if (in_mode < 0 || in_mode > ASM_B200_IN_CONST_AMP_PHASE) return ASM_B200_E_MODE;
    if (cot_mode != ASM_B200_IN_COMPLEX && cot_mode != ASM_B200_IN_COT_FIELD) return ASM_B200_E_MODE;
    if (z_dtype != ASM_B200_Z_F32 && z_dtype != ASM_B200_Z_F64) return ASM_B200_E_MODE;
    if (needs_in1(in_mode) && !in1) return ASM_B200_E_NULL;
    if (!cot0 || !grad_z || (cot_mode == ASM_B200_IN_COT_FIELD && !cot1)) return ASM_B200_E_NULL;
    if (B <= 0) return ASM_B200_E_SHAPE;
    cudaError_t e = cudaMemsetAsync(grad_z, 0, sizeof(double) * (size_t)B, reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return (int)e;
    Params p{};
    p.in0 = in0; p.in1 = in1; p.aux0 = cot0; p.aux1 = cot1; p.aux_mode = cot_mode; p.out0 = grad_z; p.z = z; p.z_f64 = z_dtype;
    p.in_mode = in_mode; p.out_mode = OUT_DOT; p.h_mode = H_DERIV; p.adj = 0; p.band_limit = band_limit;
    // Intensity cotangent g = 2 w U: the constant part of kz contributes Re(conj(g) i k0 U) = 0 exactly, but in fp32 it
    // is a cancelling sum ~100x larger than the result.  Differentiate with kz - 1/lambda instead (same derivative).
    p.kshift = cot_mode == ASM_B200_IN_COT_FIELD ? 1.0 : 0.0;
    p.in_scale = in_scale; p.out_scale = 1.f;
    return run(p, B, C, N, pad, lambda, px, workspace, workspace_bytes, stream);
}

extern "C" size_t asm_b200_unwrap_workspace_bytes(int B, int H, int W) {
    UnwrapLayout L;
    return unwrap_layout(B, H, W, &L) ? L.total : 0;
}

extern "C" int asm_b200_unwrap(const float* phase, float* out, int B, int H, int W, void* workspace, size_t workspace_bytes,
                               void* stream) {
    if (!phase || !out) return ASM_B200_E_NULL;
    UnwrapLayout L;
    if (!unwrap_layout(B, H, W, &L)) return ASM_B200_E_SHAPE;
    const long long E = (long long)B * ((long long)H * (W - 1) + (long long)(H - 1) * W);   // <= INT_MAX (unwrap_layout)
    if (!workspace || ((uintptr_t)workspace & 255) || workspace_bytes < L.total) return ASM_B200_E_WORKSPACE;
    int rc = check_device();
    if (rc) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    unsigned char* w = reinterpret_cast<unsigned char*>(workspace);
    float* rel = reinterpret_cast<float*>(w + L.rel);
    float* key_in = reinterpret_cast<float*>(w + L.key_in);
    float* key_out = reinterpret_cast<float*>(w + L.key_out);
    int* id_in = reinterpret_cast<int*>(w + L.id_in);
    int* id_out = reinterpret_cast<int*>(w + L.id_out);
    int* seg = reinterpret_cast<int*>(w + L.seg);
    int* parent = reinterpret_cast<int*>(w + L.parent);
    int* off = reinterpret_cast<int*>(w + L.off);
    int* size = reinterpret_cast<int*>(w + L.size);
    int* base = reinterpret_cast<int*>(w + L.base);
    // cub reports whatever non-sticky error is pending in the runtime as its own (e.g. an "invalid device ordinal" left by
    // an unrelated probe of the caller): clear it first -- such an error is not ours and says nothing about this call.
    (void)cudaGetLastError();
    const cudaError_t pending = cudaSuccess;
    const int blocks = 4 * sm_count();
    k_unwrap_reliability<<<blocks, 256, 0, st>>>(phase, rel, B, H, W);
    k_unwrap_edges<<<blocks, 256, 0, st>>>(phase, rel, key_in, id_in, seg, B, H, W);
    size_t cb = L.cub_bytes;
    cudaError_t e = cub::DeviceSegmentedRadixSort::SortPairs(w + L.cub, cb, key_in, key_out, id_in, id_out, (int)E, B, seg, seg + 1,
                                                             0, 32, st);
    if (e != cudaSuccess) return (int)e;
    if (H * W <= UW_SMEM_PIX) {
        const size_t smem = (size_t)UW_SMEM_PIX * (4 + 2 + 2 + 2 + 2);
        static std::atomic<unsigned long long> done{0};
        int dev;
        if (!attrs_done(done, &dev)) {
            if ((e = set_smem(k_unwrap_merge_smem, smem)) != cudaSuccess) return (int)e;
            attrs_mark(done, dev);
        }
        k_unwrap_merge_smem<<<B, 256, smem, st>>>(phase, id_out, parent, off, base, H, W);
    } else {
        k_unwrap_merge<<<B, 256, 0, st>>>(phase, id_out, parent, off, size, base, H, W);
    }
    k_unwrap_apply<<<blocks, 256, 0, st>>>(phase, out, parent, off, base, B, H * W);
    g_launches.fetch_add(5);
    if (pending == cudaSuccess) {
        e = cudaPeekAtLastError();
        if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
    }
    return 0;
}

extern "C" size_t asm_b200_focal_stack_workspace_bytes(int B, int K, int N, int pad) {
    if (B <= 0 || K <= 0 || (long long)B * K > 0x7fffffffll) return 0;
    const size_t single = asm_b200_workspace_bytes(B, 1, N, pad);
    if (!single) return 0;
    Geometry g;
    StackPlan sp;
    DftGeom dg;
    size_t need;
    if (make_stack_plan(B, K, N, pad, &g, &sp)) need = stack_workspace_need(g, sp);
    else if (dft_geometry(B * K, N, pad, &dg)) need = dft_workspace(dg) + dft_stack_partials(dg);
    else return 0;
    return need > single ? need : single;   // one buffer also serves asm_b200_forward on the same B, N, pad
}

extern "C" int asm_b200_focal_stack(const void* in0, const void* in1, const void* z, int z_dtype, int K,
                                    void* out0, void* out1, double* moments,
                                    int B, int N, int pad, int in_mode, int out_mode,
                                    double lambda, double px, float in_scale,
                                    void* workspace, size_t workspace_bytes, void* stream) {
    return asm_b200_focal_stack_bl(in0, in1, z, z_dtype, K, out0, out1, moments, B, N, pad, in_mode, out_mode, lambda, px,
                                   in_scale, workspace, workspace_bytes, stream, 0);
}

extern "C" int asm_b200_focal_stack_bl(const void* in0, const void* in1, const void* z, int z_dtype, int K,
                                       void* out0, void* out1, double* moments,
                                       int B, int N, int pad, int in_mode, int out_mode,
                                       double lambda, double px, float in_scale,
                                       void* workspace, size_t workspace_bytes, void* stream, int band_limit) {
    if (band_limit != 0 && band_limit != 1) return ASM_B200_E_MODE;
    if (!out0 && !moments) return ASM_B200_E_NULL;
    if (in_mode < 0 || in_mode > ASM_B200_IN_CONST_AMP_PHASE || in_mode == ASM_B200_IN_COT_FIELD) return ASM_B200_E_MODE;
    if (out_mode != ASM_B200_OUT_COMPLEX && out_mode != ASM_B200_OUT_INTENSITY && out_mode != ASM_B200_OUT_ABS_ANGLE) return ASM_B200_E_MODE;
    if (out1 && out_mode != ASM_B200_OUT_ABS_ANGLE) return ASM_B200_E_MODE;
    if (z_dtype != ASM_B200_Z_F32 && z_dtype != ASM_B200_Z_F64) return ASM_B200_E_MODE;
    if (K <= 0 || B <= 0) return ASM_B200_E_SHAPE;
    const size_t need = asm_b200_focal_stack_workspace_bytes(B, K, N, pad);
    if (!need) return ASM_B200_E_SHAPE;
    if (!(lambda > 0.0) || !(px > 0.0) || !isfinite(lambda) || !isfinite(px)) return ASM_B200_E_OPTICS;
    if (!workspace || ((uintptr_t)workspace & 255) || workspace_bytes < need) return ASM_B200_E_WORKSPACE;
    if (!in0 || !z || (needs_in1(in_mode) && !in1)) return ASM_B200_E_NULL;
    if (out0 && out_mode == ASM_B200_OUT_ABS_ANGLE && !out1) return ASM_B200_E_NULL;
    int rc = check_device();
    if (rc) return rc;
    Params p{};
    p.in0 = in0; p.in1 = in1; p.out0 = out0; p.out1 = out0 ? out1 : nullptr; p.z = z; p.z_f64 = z_dtype;
    p.in_mode = in_mode; p.out_mode = out_mode; p.h_mode = H_FWD; p.adj = 0; p.band_limit = band_limit;
    p.in_scale = in_scale; p.out_scale = 1.f;
    p.C = 1; p.N = N; p.lambda = lambda; p.inv_lambda = 1.0 / lambda;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    unsigned char* w = reinterpret_cast<unsigned char*>(workspace);
    Geometry g;
    StackPlan sp;
    if (!make_stack_plan(B, K, N, pad, &g, &sp)) {                   // matrix-product path: one transform per plane
        DftGeom dg;
        dft_geometry(B * K, N, pad, &dg);
        p.planes = B * K; p.M = dg.M; p.P = dg.P; p.kst = K;
        const double sd = lambda / ((double)dg.M * px);
        p.s2 = sd * sd;
        p.S = (double)dg.M * px;
        p.inv_m2 = 1.0f / ((float)dg.M * (float)dg.M);
        p.part = moments ? reinterpret_cast<double*>(w + dft_workspace(dg)) : nullptr;
        return launch_dft(p, dg, w, st, moments);
    }
    sp.mom = moments;
    p.planes = B; p.M = g.M; p.P = g.P;
    p.tw = reinterpret_cast<const float2*>(workspace);
    p.tw32 = p.tw + (g.n == 11 ? make_layout(11).total : 0);
    p.kzt = g.kz_bytes ? reinterpret_cast<const double*>(w + g.tw_bytes) : nullptr;
    p.ws = reinterpret_cast<float2*>(w + g.tw_bytes + g.kz_bytes);
    const double sd = lambda / ((double)g.M * px);
    p.s2 = sd * sd;
    p.S = (double)g.M * px;
    p.inv_m2 = 1.0f / ((float)g.M * (float)g.M);
    switch (g.n) {
        case 5: return launch_n<5>(p, g, st, &sp);
        case 6: return launch_n<6>(p, g, st, &sp);
        case 7: return launch_n<7>(p, g, st, &sp);
        case 8: return launch_n<8>(p, g, st, &sp);
        case 9: return launch_n<9>(p, g, st, &sp);
        case 10: return launch_32t(p, g, st, &sp);
        case 11: return knob_k64() ? launch_64(p, g, st, &sp) : launch_n<11>(p, g, st, &sp);
        case 12: return launch_n<12>(p, g, st, &sp);
    }
    return ASM_B200_E_SHAPE;
}
