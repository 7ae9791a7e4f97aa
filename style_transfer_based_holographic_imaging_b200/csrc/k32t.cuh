// k32t.cuh -- the FFT-size-1024 path with a TRANSPOSED intermediate: every pass works on contiguous 8 KB lines that are
// private to one warp, and both transposes of the 2-D transform are done by the TMA engine on 64-byte segments.
//
//   wsT[img][u][y]   u = row-pass frequency (1024), y = source row (N), complex64 -- "line u" is contiguous in y.
//
//   pass 1  k32t_rows_fwd : a CTA = 8 warps = 8 consecutive source rows, 2 CTAs per SM.  One 66 KB region of 8 lines serves
//                           every role: a warp's line is the landing line of its source row (ONE TMA bulk copy), then its
//                           exchange line (radix-32, exchange, radix-32; __syncwarp only); after a CTA barrier the same
//                           memory holds the tile [1024 u][8 y] (64-byte rows, 16-byte chunks XOR-swizzled exactly as the
//                           tensor map's SWIZZLE_64B, so a warp's column of the tile is 2-way instead of 16-way bank
//                           conflicted) and one thread hands it to the TMA engine (4 tensor stores of 256 u x 8 y).
//   pass 2  k32t_lines    : a WARP per line u, 16 independent warps per SM, no CTA barrier: the line (and, when |u| changes,
//                           its kappa row) lands in the warp's exchange line by TMA bulk copies issued during the previous
//                           line's last radix-32 stage; -> registers, FFT over y, x H(u, v), inverse FFT, coalesced stores
//                           back in place.  kappa(|u|, |v|) is a symmetric 513 x 513 table of fp32 (hi, lo) pairs and the
//                           phase t = c kappa is evaluated in double-float fp32 (exact product by FMA, no fp64, no F2F);
//                           lines are handed out sorted by |u| so that a warp's consecutive lines share one kappa row.
//   pass 3  k32t_rows_inv : mirror of pass 1: 4 tensor loads land the tile [u][8 y] of 8 output rows, a warp reads its
//                           column of the tile, the region becomes the exchange lines, inverse transform, output stage
//                           (TMA bulk store, or the generic modes through registers); pairs of adjacent groups drop their
//                           consumed 128-byte workspace lines from L2 (discard.global.L2).
// Measured (profiles/r02_experiments.md): the three passes are bound by the memory system between L2 and the SMs, not by
// arithmetic; DRAM traffic is 1.02 x algorithmic and the L2 <-> SM traffic runs at 59 % of the chip's cap.
// Reference semantics: utils/Angular_Spectrum_Method.py:7-36 (unshifted bins, H = exp(i c kz), evanescent -> H = 1).
// Included by asm_b200.cu after k32.cuh (uses its loaders, emitters and radix-32 stages).
#pragma once

namespace asmb {

#ifndef K32T_DBG
#define K32T_DBG 0      /* tools/ timing experiments only: 1 no tile store, 2 no forward row math, 3 no tile load, 4 no output store, 5 no line math */
#endif

#ifndef K32T_DISCARD
#define K32T_DISCARD 1    /* pass 3 drops the consumed workspace lines from L2 (0: A/B builds) */
#endif

#ifndef K32T_PF
#define K32T_PF 1         /* pass 1: the rows of the group this many iterations ahead are prefetched into L2 */
#endif

constexpr int KAP_STRIDE = 520;                          // entries per row of the symmetric kappa table (513 used)
constexpr unsigned KAP_ROW_B = 514 * 8;                  // bytes copied per line (multiple of 16)
constexpr int K32T_TILE_B = 1024 * 8 * 8;                // [1024 u][8 y] complex64
constexpr int K32T_ROW_WARPS = 8;
#ifndef K32T_ROW_CTAS_DEF
#define K32T_ROW_CTAS_DEF 2
#endif
constexpr int K32T_ROW_CTAS = K32T_ROW_CTAS_DEF;         // row-pass CTAs per SM
constexpr size_t K32T_FWD_SMEM = 1024 /*alignment slack*/ + (size_t)K32T_ROW_WARPS * (K32_LP * 8) + K32_TW * 8 + 64;
constexpr size_t K32T_INV_SMEM = K32T_FWD_SMEM;
#ifndef K32T_LINE_WARPS_DEF
#define K32T_LINE_WARPS_DEF 8
#endif
#ifndef K32T_LINE_CTAS_DEF
#define K32T_LINE_CTAS_DEF 2
#endif
constexpr int K32T_LINE_WARPS = K32T_LINE_WARPS_DEF;     // warps per CTA of pass 2
constexpr int K32T_LINE_CTAS = K32T_LINE_CTAS_DEF;       // ... and CTAs per SM
constexpr size_t K32T_LINES_SMEM = (size_t)K32T_LINE_WARPS * (K32_LP * 8 + KAP_STRIDE * 8) + K32_TW * 8 + 64;

// tables: half twiddle table (as k32_setup) + kappa2[ru][rv] = (hi, lo), hi + lo = kz(ru, rv) / (2 pi) to 2^-48
__global__ void k32t_setup(float2* tw, float2* kap2, double s2, double inv_2pi_lambda) {
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    for (int e = gtid; e < K32_TW; e += gsz) {
        const int ent = e / 32, Q = e % 32;
        int m = 1;
        while (m < 5 && ent >= (1 << (m - 1))) ++m;
        const int u = ent - (m == 1 ? 0 : (1 << (m - 2)));
        const int D = 32 << m, x = Q + 32 * u;
        float sn, cs;
        sincospif(2.0f * (float)x / (float)D, &sn, &cs);
        tw[e] = make_float2(cs, -sn);
    }
    for (int idx = gtid; idx < 513 * KAP_STRIDE; idx += gsz) {
        const int ru = idx / KAP_STRIDE, rv = idx % KAP_STRIDE;
        const double kk = (double)ru * ru + (double)rv * rv;
        const double arg = fma(-s2, kk, 1.0);
        const double kap = (arg > 0.0 ? sqrt(arg) : 0.0) * inv_2pi_lambda;
        const float hi = (float)kap;
        kap2[idx] = make_float2(hi, (float)(kap - (double)hi));
    }
}

// element index (float2 units) of (u, yy) in the swizzled tile: 64-byte row u, 16-byte chunk (yy / 2) ^ ((u / 2) & 3)
__device__ __forceinline__ int k32t_tile_idx(int u, int yy) { return u * 8 + ((((yy >> 1) ^ (u >> 1)) & 3) << 1) + (yy & 1); }

// H(u, v = lane + 32 i) on the registers of one line.  c = (c_hi, c_lo): the sample's phase constant (ASM.py:29), negative
// for the adjoint.  t = c kappa: p = hi c_hi rounded, e = the exact rounding error of that product (FMA), the remaining
// cross terms are O(1e-3) turns; frac(p) is exact in fp32 (|p| < 2^22 turns, i.e. |z| < 2 m).
template <bool DERIV>
__device__ __forceinline__ void k32t_apply_h(float2 (&v)[32], const Params& p, const float2* kap_s, int lane, float c_hi, float c_lo) {
    const float MAGIC = 12582912.f;                                   // 1.5 * 2^23: round to nearest integer
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        const int f = lane + 32 * i;
        const float2 k = kap_s[f <= 512 ? f : 1024 - f];
        const float pp = __fmul_rn(k.x, c_hi);
        float s = __fmaf_rn(k.x, c_hi, -pp);
        s = __fmaf_rn(k.y, c_hi, s);
        s = __fmaf_rn(k.x, c_lo, s);
        const float kk = __fadd_rn(__fadd_rn(pp, MAGIC), -MAGIC);
        const float r = __fadd_rn(__fadd_rn(pp, -kk), s);
        float sn, cn;
        __sincosf(r * 6.283185307179586f, &sn, &cn);
        if constexpr (DERIV) {
            const double kz_l = ((double)k.x + (double)k.y) * (6.283185307179586 * p.lambda);    // sqrt(1 - lambda^2 f^2)
            v[i] = cmul_scaled(v[i], -sn, cn, (float)(kz_l - p.kshift) * p.inv_m2);
        } else {
            v[i] = cmul_scaled(v[i], cn, sn, p.inv_m2);
        }
    }
}

// phase constant of sample b as a double-float pair (fp32 distances: exactly fl32(fl32(2 pi) z), lo = 0)
__device__ __forceinline__ void k32t_phase_constant(const Params& p, int b, float* c_hi, float* c_lo) {
    const double c = phase_constant_of(p, b);
    *c_hi = (float)c;
    *c_lo = (float)(c - (double)*c_hi);
}

// ---------------------------------------------------------------------------------------------------
// Row passes.  ONE shared-memory region of 8 exchange lines (66 KB) serves every role: a line is the landing line of its
// warp's source row (dense, TMA bulk copy), then its exchange line; once every warp is done the same memory holds the CTA
// tile [1024 u][8 y] that the TMA engine stores (pass 1), or the tile the TMA engine loaded before the lines were needed
// (pass 3).  A CTA therefore needs 70 KB and nothing inside a CTA overlaps with its own memory traffic -- the overlap comes
// from the K32T_ROW_CTAS independent CTAs per SM (16 or more warps, as many barrier domains as CTAs).
//
// pass 1: forward rows -> transposed workspace.  IN: 0 complex64 rows, 1 amplitude + phase rows, 2 constant amplitude +
// phase rows (TMA bulk copies into the warp's line), 3 every other input mode / unaligned rows (register loads)
// ---------------------------------------------------------------------------------------------------
template <int IN, bool PADDED>
__global__ void __launch_bounds__(32 * K32T_ROW_WARPS, K32T_ROW_CTAS)
k32t_rows_fwd(const Params p, const __grid_constant__ CUtensorMap tmapT, int plane0, int ngroups) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int XCH_B = K32_LP * 8;
    unsigned char* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-byte aligned, still a shared-memory pointer
    float2* tile = reinterpret_cast<float2*>(base);                  // [1024 u][8 y], aliases the lines
    const int t = threadIdx.x, w = t >> 5, lane = t & 31;
    float2* xch = reinterpret_cast<float2*>(base + (size_t)w * XCH_B);
    float2* tw = reinterpret_cast<float2*>(base + (size_t)K32T_ROW_WARPS * XCH_B);
    uint64_t* bars = reinterpret_cast<uint64_t*>(tw + K32_TW);
    for (int i = t; i < K32_TW; i += blockDim.x) tw[i] = __ldg(p.tw + i);
    if (t < K32T_ROW_WARPS) mbar_init(bars + t, 1);
    fence_mbar_init();
    uint64_t* bar = bars + w;
    const uint64_t pol_in = policy_evict_first();
    const int N = PADDED ? p.N : K32_L;
    const unsigned row_bytes = (unsigned)N * (IN == 2 ? 4u : 8u);
    const float amp0 = IN == 2 ? __ldg((const float*)p.in0) : 0.f;
    const bool pf_ok = IN == 3 ? k32_prefetch_ok(p) : true;
    auto request = [&](int gline) {                                  // lane 0 only
        const size_t row = ((size_t)(plane0 + gline / N) * N + gline % N) * N;
        mbar_expect_tx(bar, row_bytes);
        if constexpr (IN == 1) {
            bulk_load(xch, (const float*)p.in0 + row, row_bytes / 2, bar, pol_in);
            bulk_load(reinterpret_cast<unsigned char*>(xch) + row_bytes / 2, (const float*)p.in1 + row, row_bytes / 2, bar, pol_in);
        } else if constexpr (IN == 2) {
            bulk_load(xch, (const float*)p.in1 + row, row_bytes, bar, pol_in);
        } else {
            bulk_load(xch, (const float2*)p.in0 + row, row_bytes, bar, pol_in);
        }
    };
    unsigned phase = 0;
    // the tile column of this warp: u = lane + 32 i  ->  (u / 2) & 3 = (lane / 2) & 3 for every i
    float2* tcol = tile + k32t_tile_idx(lane, w);
    for (int g = blockIdx.x; g < ngroups; g += gridDim.x) {
        const int gline = g * 8 + w;
        __syncthreads();                                             // the region is free (the previous tile has left it)
        float2 v[32];
        if (lane == 0 && pf_ok && K32T_PF > 0 && g + K32T_PF * gridDim.x < ngroups) {   // HBM -> L2 for a later group
            const int nxt = (g + K32T_PF * gridDim.x) * 8 + w;
            k32_prefetch_row(p, plane0 + nxt / N, nxt % N);
        }
        if constexpr (IN == 3) {
            const int plane = plane0 + gline / N, y = gline % N;
            switch (p.in_mode) {
                case ASM_B200_IN_COMPLEX: load32<ASM_B200_IN_COMPLEX>(v, p, plane, y, lane); break;
                case ASM_B200_IN_AMP_PHASE: load32<ASM_B200_IN_AMP_PHASE>(v, p, plane, y, lane); break;
                case ASM_B200_IN_CONST_AMP_PHASE: load32<ASM_B200_IN_CONST_AMP_PHASE>(v, p, plane, y, lane); break;
                case ASM_B200_IN_SQRT_REAL: load32<ASM_B200_IN_SQRT_REAL>(v, p, plane, y, lane); break;
                case ASM_B200_IN_COT_FIELD: load32<ASM_B200_IN_COT_FIELD>(v, p, plane, y, lane); break;
                default: load32<ASM_B200_IN_REAL>(v, p, plane, y, lane); break;
            }
        } else {
            if (lane == 0) request(gline);
            mbar_wait(bar, phase);
            phase ^= 1u;
#pragma unroll
            for (int i = 0; i < (K32T_DBG == 6 ? 1 : 32); ++i) {
                int x = lane + 32 * i;
                bool in = true;
                if constexpr (PADDED) { x -= p.P; in = !p.adj || (x >= 0 && x < N); x = min(max(x, 0), N - 1); }
                float2 val;
                if constexpr (IN == 0) {
                    val = xch[x];
                } else {
                    const float a = IN == 1 ? reinterpret_cast<const float*>(xch)[x] : amp0;
                    const float ph = reinterpret_cast<const float*>(xch)[(IN == 1 ? N : 0) + x] * p.in_scale;
                    float sn, cs;
                    sincos_reduced(ph, &sn, &cs);
                    val = make_float2(a * cs, a * sn);
                }
                v[i] = (!PADDED || in) ? val : make_float2(0.f, 0.f);
            }
            __syncwarp();                                            // the dense row is in registers: the exchange may overwrite it
        }
        if (K32T_DBG != 2 && K32T_DBG != 6) fwd32_first(v);
        if (K32T_DBG != 6) sts16<RowLayout32, 5>(v, xch + lane);
        __syncwarp();
        if (K32T_DBG != 6) lds16<RowLayout32, 0>(v, xch + 33 * lane);
        if (K32T_DBG != 2 && K32T_DBG != 6) fwd32_table(v, tw + lane);   // v[i] = frequency lane + 32 i
        __syncthreads();                                             // every warp is done with its line: the region becomes the tile
#pragma unroll
        for (int i = 0; i < (K32T_DBG == 6 ? 1 : 32); ++i) tcol[i * 256] = v[i];
        fence_proxy_async();
        __syncthreads();
        if (t == 0) {
            const int img = (g * 8) / N, y0 = (g * 8) % N;
#pragma unroll
            for (int k = 0; k < 4; ++k) if (K32T_DBG != 1) tma_store_3d(&tmapT, tile + k * 2048, 2 * y0, 256 * k, img);
            tma_commit();
            tma_wait_read0();                                        // ... and has been read by the TMA engine
        }
    }
    if (t == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------------
// pass 2: one warp per line u of the transposed workspace: FFT over y, x H, inverse FFT, in place
// ---------------------------------------------------------------------------------------------------
template <bool PADDED>
__global__ void __launch_bounds__(32 * K32T_LINE_WARPS, K32T_LINE_CTAS) k32t_lines(const Params p, int plane0, int nlines) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int XCH_B = K32_LP * 8, KAP_B = KAP_STRIDE * 8;
    const int t = threadIdx.x, w = t >> 5, lane = t & 31;
    float2* xch = reinterpret_cast<float2*>(smem_raw + (size_t)w * (XCH_B + KAP_B));
    float2* kap_s = reinterpret_cast<float2*>(smem_raw + (size_t)w * (XCH_B + KAP_B) + XCH_B);
    float2* tw = reinterpret_cast<float2*>(smem_raw + (size_t)K32T_LINE_WARPS * (XCH_B + KAP_B));
    uint64_t* bars = reinterpret_cast<uint64_t*>(tw + K32_TW);
    for (int i = t; i < K32_TW; i += blockDim.x) tw[i] = __ldg(p.tw + i);
    if (t < K32T_LINE_WARPS) mbar_init(bars + t, 1);
    fence_mbar_init();
    __syncthreads();
    uint64_t* bar = bars + w;
    const uint64_t pol = policy_evict_normal();
    const int N = PADDED ? p.N : K32_L;
    const float2* kap2 = reinterpret_cast<const float2*>(p.kzt);
    // The warp's exchange line doubles as the landing line of its NEXT line: the request (line + kappa row, one
    // mbarrier) is issued right after the last exchange read of the current line, so it lands during the last radix-32
    // stage and the stores.
    // Lines are handed out in an order sorted by |u|: a warp takes a contiguous slice of
    //   (u = 0: every image) (|u| = 1: image 0 +, image 0 -, image 1 +, ...) ... (u = 512: every image)
    // so that its consecutive lines share the kappa row, which is then loaded once per slice instead of once per line
    // (4 MB of L2 reads per image otherwise: the pipeline is bound by L2 <-> SM transfers, see DESIGN.md).
    const int nimg = nlines >> 10;
    auto line_of = [&](int s) {
        int img, u;
        if (s < nimg) { img = s; u = 0; }
        else if (s >= nlines - nimg) { img = s - (nlines - nimg); u = 512; }
        else {
            const int q = s - nimg, r = 1 + q / (2 * nimg), rem = q - (r - 1) * 2 * nimg;
            img = rem >> 1;
            u = (rem & 1) ? 1024 - r : r;
        }
        return (img << 10) | u;
    };
    auto request = [&](int line, bool with_kappa) {                  // lane 0 only
        const int u = line & 1023, ru = u <= 512 ? u : 1024 - u;
        mbar_expect_tx(bar, (unsigned)N * 8u + (with_kappa ? KAP_ROW_B : 0u));
        const size_t src_line = ((size_t)src_slot(p, plane0, line >> 10) << 10) | (unsigned)(line & 1023);
        bulk_load(xch, src_base(p) + src_line * N, (unsigned)N * 8u, bar, pol);
        if (with_kappa) bulk_load(kap_s, kap2 + (size_t)ru * KAP_STRIDE, KAP_ROW_B, bar, pol);
    };
    const int nwarps = gridDim.x * K32T_LINE_WARPS, wg = blockIdx.x * K32T_LINE_WARPS + w;
    int s = (int)((long long)wg * nlines / nwarps);
    const int s_end = (int)((long long)(wg + 1) * nlines / nwarps);
    if (lane == 0 && s < s_end) request(line_of(s), true);
    unsigned phase = 0;
    for (; s < s_end; ++s) {
        const int line = line_of(s);
        const int img = line >> 10;
        float2* row = p.ws + (size_t)line * N;
        float c_hi, c_lo;
        k32t_phase_constant(p, (plane0 + img) / p.C, &c_hi, &c_lo);
        mbar_wait(bar, phase);
        phase ^= 1u;
        float2 v[32];
        if constexpr (!PADDED) {
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = xch[lane + 32 * i];
        } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                int y = lane + 32 * i - p.P;
                if (p.adj) v[i] = (y >= 0 && y < N) ? xch[y] : make_float2(0.f, 0.f);
                else v[i] = xch[min(max(y, 0), N - 1)];
            }
        }
        __syncwarp();                                                // the dense line is in registers: the exchange may overwrite it
        if (K32T_DBG != 5) {
        fwd32_first(v);
        sts16<RowLayout32, 5>(v, xch + lane);
        __syncwarp();
        lds16<RowLayout32, 0>(v, xch + 33 * lane);
        fwd32_table(v, tw + lane);                                   // v[i] = frequency lane + 32 i
        if (p.h_mode == H_DERIV) k32t_apply_h<true>(v, p, kap_s, lane, c_hi, c_lo);
        else k32t_apply_h<false>(v, p, kap_s, lane, c_hi, c_lo);
        inv32_first(v);
        __syncwarp();                                                // every lane has read its exchange values
        sts16<RowLayout32, 0>(v, xch + 33 * lane);
        __syncwarp();
        lds16<RowLayout32, 5>(v, xch + lane);
        }
        fence_proxy_async();                                         // exchange and kappa reads are done before the next line lands
        __syncwarp();
        if (lane == 0 && s + 1 < s_end) {
            const int nxt = line_of(s + 1), un = nxt & 1023, uc = line & 1023;
            request(nxt, (un <= 512 ? un : 1024 - un) != (uc <= 512 ? uc : 1024 - uc));
        }
        if (K32T_DBG != 5) inv32_table(v, tw + lane);                // v[i] = position lane + 32 i
        if constexpr (!PADDED) {
#pragma unroll
            for (int i = 0; i < 32; ++i) __stcg(row + lane + 32 * i, v[i]);
        } else {
            float2 fl = make_float2(0.f, 0.f), fr = make_float2(0.f, 0.f);
            if (p.adj) {   // adjoint of replicate padding: fold positions [0, P) onto y = 0 and [P + N, M) onto y = N - 1
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const int pos = lane + 32 * i;
                    if (pos < p.P) { fl.x += v[i].x; fl.y += v[i].y; }
                    if (pos >= p.P + N) { fr.x += v[i].x; fr.y += v[i].y; }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    fl.x += __shfl_xor_sync(0xffffffffu, fl.x, o); fl.y += __shfl_xor_sync(0xffffffffu, fl.y, o);
                    fr.x += __shfl_xor_sync(0xffffffffu, fr.x, o); fr.y += __shfl_xor_sync(0xffffffffu, fr.y, o);
                }
            }
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const int y = lane + 32 * i - p.P;
                if (y >= 0 && y < N) {
                    float2 o = v[i];
                    if (y == 0) { o.x += fl.x; o.y += fl.y; }
                    if (y == N - 1) { o.x += fr.x; o.y += fr.y; }
                    __stcg(row + y, o);
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// pass 3: transposed workspace -> inverse rows -> output stage.  OUT: 0 complex64 (TMA bulk store), 1 |U|^2 (TMA bulk
// store), 2 every other output mode / unaligned rows (register stores)
// ---------------------------------------------------------------------------------------------------
template <int OUT, bool PADDED>
__global__ void __launch_bounds__(32 * K32T_ROW_WARPS, K32T_ROW_CTAS)
k32t_rows_inv(const Params p, const __grid_constant__ CUtensorMap tmapT, int plane0, int ngroups) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int XCH_B = K32_LP * 8;
    unsigned char* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    float2* tile = reinterpret_cast<float2*>(base);                  // [1024 u][8 y], aliases the lines
    const int t = threadIdx.x, w = t >> 5, lane = t & 31;
    float2* xch = reinterpret_cast<float2*>(base + (size_t)w * XCH_B);
    float2* tw = reinterpret_cast<float2*>(base + (size_t)K32T_ROW_WARPS * XCH_B);
    uint64_t* bar = reinterpret_cast<uint64_t*>(tw + K32_TW);
    for (int i = t; i < K32_TW; i += blockDim.x) tw[i] = __ldg(p.tw + i);
    if (t == 0) mbar_init(bar, 1);
    fence_mbar_init();
    const uint64_t pol_out = policy_evict_first();
    const int N = PADDED ? p.N : K32_L;
    const bool folding = PADDED && p.adj;
    // A CTA works on PAIRS of adjacent groups (16 consecutive rows): once both tiles of a pair have been read, the 128-byte
    // lines that hold them in the workspace are dead and are dropped from L2 instead of being written back to HBM (the
    // slot is completely rewritten by the next forward row pass before anything reads it again).
    const int npairs = ngroups >> 1;                                 // N / 8 is even
    const float2* tcol = tile + k32t_tile_idx(lane, w);
    unsigned phase = 0;
    for (int it = 0; blockIdx.x + (it >> 1) * gridDim.x < npairs; ++it) {
        const int g = 2 * (blockIdx.x + (it >> 1) * gridDim.x) + (it & 1);
        __syncthreads();                                             // the region is free (every output row has left its line)
        if (t == 0 && K32T_DBG != 3) {
            const int img = (g * 8) / N, y0 = (g * 8) % N;
            mbar_expect_tx(bar, K32T_TILE_B);
#pragma unroll
            for (int k = 0; k < 4; ++k) tma_load_3d(tile + k * 2048, &tmapT, bar, 2 * y0, 256 * k, img);
        }
        if (K32T_DBG != 3) mbar_wait(bar, phase);
        phase ^= 1u;
        float2 v[32];
#pragma unroll
        for (int i = 0; i < (K32T_DBG == 7 ? 1 : 32); ++i) v[i] = tcol[i * 256];   // frequency lane + 32 i of row 8 g + w
        __syncthreads();                                             // the tile is in registers: the region becomes the lines
        if ((it & 1) && K32T_DISCARD) {
            const int img = ((g - 1) * 8) / N, y0 = ((g - 1) * 8) % N;   // first row of the pair: a multiple of 16
            const char* a = reinterpret_cast<const char*>(p.ws + ((size_t)img * K32_L + t) * N + y0);
#pragma unroll
            for (int j = 0; j < 4; ++j)
                asm volatile("discard.global.L2 [%0], 128;" ::"l"(a + (size_t)j * 256 * N * 8) : "memory");
        }
        if (K32T_DBG != 7) {
        inv32_first(v);
        sts16<RowLayout32, 0>(v, xch + 33 * lane);
        __syncwarp();
        lds16<RowLayout32, 5>(v, xch + lane);
        inv32_table(v, tw + lane);                                   // v[i] = natural position lane + 32 i
        }
        __syncwarp();
        const int gline = g * 8 + w;
        const int img = gline / N, y = gline % N, plane = plane0 + img;
        float2 fl = make_float2(0.f, 0.f), fr = make_float2(0.f, 0.f);
        if (folding) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const int pos = lane + 32 * i;
                if (pos < p.P) { fl.x += v[i].x; fl.y += v[i].y; }
                if (pos >= p.P + N) { fr.x += v[i].x; fr.y += v[i].y; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                fl.x += __shfl_xor_sync(0xffffffffu, fl.x, o); fl.y += __shfl_xor_sync(0xffffffffu, fl.y, o);
                fr.x += __shfl_xor_sync(0xffffffffu, fr.x, o); fr.y += __shfl_xor_sync(0xffffffffu, fr.y, o);
            }
        }
        if constexpr (OUT == 2) {
            float dot = 0.f;
            if (p.out0) switch (p.out_mode) {
                case ASM_B200_OUT_COMPLEX: emit32<ASM_B200_OUT_COMPLEX>(v, p, plane, y, lane, fl, fr); break;
                case ASM_B200_OUT_INTENSITY: emit32<ASM_B200_OUT_INTENSITY>(v, p, plane, y, lane, fl, fr); break;
                case ASM_B200_OUT_ABS_ANGLE: emit32<ASM_B200_OUT_ABS_ANGLE>(v, p, plane, y, lane, fl, fr); break;
                case ASM_B200_OUT_REIM_CAT: emit32<ASM_B200_OUT_REIM_CAT>(v, p, plane, y, lane, fl, fr); break;
                case ASM_B200_OUT_ABSANG_CAT: emit32<ASM_B200_OUT_ABSANG_CAT>(v, p, plane, y, lane, fl, fr); break;
                case ASM_B200_OUT_GRAD_AP: emit32<ASM_B200_OUT_GRAD_AP>(v, p, plane, y, lane, fl, fr); break;
                default: dot = emit32<OUT_DOT>(v, p, plane, y, lane, fl, fr); break;
            }
            if (p.out_mode == OUT_DOT) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
                const double K = p.z_f64 ? 6.283185307179586 : (double)6.2831854820251465f;
                if (lane == 0) atomicAdd((double*)p.out0 + plane / p.C, (double)dot * K * p.inv_lambda);
            }
            if (p.part) {                                            // moments of the cropped row: one partial per row
                float m[3] = {0.f, 0.f, 0.f};
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const int x = lane + 32 * i - (PADDED ? p.P : 0);
                    if (x >= 0 && x < N) mom_add(m, v[i]);
                }
                double d[3];
                mom_reduce<32>(d, m);
                if (lane == 0) {
                    double* dst = p.part + ((size_t)img * N + y) * 3;
                    dst[0] = d[0]; dst[1] = d[1]; dst[2] = d[2];
                }
            }
            fence_proxy_async();                                     // the line reads are done before the next tile lands on them
        } else {
            if constexpr (!PADDED) {
#pragma unroll
                for (int i = 0; i < (K32T_DBG == 7 ? 1 : 32); ++i) {
                    if constexpr (OUT == 1) reinterpret_cast<float*>(xch)[lane + 32 * i] = fmaf(v[i].x, v[i].x, v[i].y * v[i].y);
                    else xch[lane + 32 * i] = v[i];
                }
            } else {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const int x = lane + 32 * i - p.P;
                    if (x >= 0 && x < N) {
                        float2 o = v[i];
                        if (x == 0) { o.x += fl.x; o.y += fl.y; }
                        if (x == N - 1) { o.x += fr.x; o.y += fr.y; }
                        if constexpr (OUT == 1) reinterpret_cast<float*>(xch)[x] = fmaf(o.x, o.x, o.y * o.y);
                        else xch[x] = o;
                    }
                }
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                if (K32T_DBG != 4) {
                    const size_t row = ((size_t)plane * N + y) * N;
                    if constexpr (OUT == 1) bulk_store((float*)p.out0 + row, xch, (unsigned)N * 4u, pol_out);
                    else bulk_store((float2*)p.out0 + row, xch, (unsigned)N * 8u, pol_out);
                }
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                tma_wait_read0();                                    // the row has left the line
            }
        }
    }
    if (OUT != 2 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

}  // namespace asmb
