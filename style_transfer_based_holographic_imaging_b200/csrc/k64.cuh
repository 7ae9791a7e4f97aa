// k64.cuh -- the FFT-size-2048 path: 2048 = 2 x 1024, one radix-2 decimation-in-frequency level around the
// one-exchange 1024-point transform of k32.cuh (32 points per thread, 64 threads per line).
//
//   forward :  a[k] = x[k] + x[k+1024],  b[k] = (x[k] - x[k+1024]) W_2048^k,   X[2m] = FFT1024(a)[m],  X[2m+1] = FFT1024(b)[m]
//   inverse :  a = IFFT1024(X[2m]),  b' = W_2048^-k IFFT1024(X[2m+1]),          x[k] = a[k] + b'[k],    x[k+1024] = a[k] - b'[k]
// Thread (h, l) of a line computes half h: it reads BOTH x[k] and x[k+1024] for its 32 positions k = l + 32 i (the forward
// level costs redundant shared-memory reads instead of an exchange); the inverse level is one exchange between the two
// halves.  The twiddle W_2048^(l + 32 i) = W_2048^l W_64^i never touches a table: W_64^i is a compile-time constant of
// register i, and the per-lane factor W_2048^l commutes with the first radix-32 stage (a DFT over i) and the exchange,
// after which it has become W_2048^j of register j -- again a compile-time constant (mirrored for the inverse).
// A line's spectrum is stored in SPLIT order in the workspace: column c' = 1024 h + m holds frequency 2 m + h, so each
// half writes / reads one contiguous 8 KB piece; the kappa table is built in that column order (k64_setup), which is all
// the column kernel needs to know about it.
//   k64_rows_fwd_bulk / k64_rows_inv_bulk : a WARP PAIR per row, TMA bulk copies in and out (complex64 / amplitude+phase
//                 in, complex64 / |U|^2 out); every other mode runs the generic row kernels (their digit-reversed column
//                 order comes with its own kappa table, and k64_cols does not care).
//   k64_cols     : 4 columns x 64 threads, 2 CTAs per SM, cp.async-staged slab and kappa, same pipeline as k32_cols.
// Included by asm_b200.cu after k32.cuh.
#pragma once

namespace asmb {

constexpr int K64_L = 2048;
constexpr int K64_CC = 4;                              // columns per slab (256 threads)
constexpr int K64_PAIRS = 3;                           // warp pairs per row CTA (2 CTAs per SM)

// compile-time cos / sin (Taylor series in double, |x| <= pi): the constant twiddles become immediate operands
__host__ __device__ constexpr double cx_sin(double x) {
    double term = x, sum = x;
    for (int k = 1; k < 14; ++k) { term *= -x * x / ((2.0 * k) * (2.0 * k + 1.0)); sum += term; }
    return sum;
}
__host__ __device__ constexpr double cx_cos(double x) {
    double term = 1.0, sum = 1.0;
    for (int k = 1; k < 14; ++k) { term *= -x * x / ((2.0 * k - 1.0) * (2.0 * k)); sum += term; }
    return sum;
}
constexpr double CX_2PI = 6.283185307179586476925286766559;

// v <- v (cr + i ci): FMUL2 + FFMA2 with constant operands
__device__ __forceinline__ float2 cmulc(float2 v, float cr, float ci) {
    return upk2(fma2(pk2(-v.y, v.x), pk2(ci, ci), mul2(pk2(v), pk2(cr, cr))));
}
// register I *= exp(SIGN i 2 pi I / D), I = 1 .. 31 (SIGN = -1: forward W_D^I; +1: its conjugate)
template <int SIGN, int D, int I>
__device__ __forceinline__ void k64_twiddle_iter(float2 (&v)[32]) {
    if constexpr (I < 32) {
        constexpr float c = (float)cx_cos(CX_2PI * I / D), s = (float)(SIGN * cx_sin(CX_2PI * I / D));
        v[I] = cmulc(v[I], c, s);
        k64_twiddle_iter<SIGN, D, I + 1>(v);
    }
}
template <int SIGN>
__device__ __forceinline__ void k64_twiddle64(float2 (&v)[32]) { k64_twiddle_iter<SIGN, 64, 1>(v); }
template <int SIGN>
__device__ __forceinline__ void k64_twiddle2048(float2 (&v)[32]) { k64_twiddle_iter<SIGN, 2048, 1>(v); }
__device__ __forceinline__ void pair_barrier(int id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }

// tables: the half twiddle table of the 1024-point transform (as k32_setup) and, if kzt != nullptr, kappa in SPLIT
// column order (calls that run the generic row kernels build kappa in their column order with k_setup_tables instead)
// pairs != 0: kappa is stored as fp32 (hi, lo) pairs (same 8 bytes per entry) for the double-float H of k64_cols<.., true>
__global__ void k64_setup(float2* tw, double* kzt, double s2, double inv_2pi_lambda, int pairs = 0) {
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
    constexpr int M = K64_L;
    if (!kzt) return;
    for (int idx = gtid; idx < (M / 2 + 1) * M; idx += gsz) {
        const int ru = idx / M, c = idx % M;
        const int v = 2 * (c & 1023) + (c >> 10);                      // frequency held by workspace column c
        const int kv = v < M / 2 ? v : v - M;
        const double kk = (double)ru * ru + (double)kv * kv;
        const double arg = fma(-s2, kk, 1.0);
        const double kap = (arg > 0.0 ? sqrt(arg) : 0.0) * inv_2pi_lambda;
        if (pairs) { const float hi = (float)kap; reinterpret_cast<float2*>(kzt)[idx] = make_float2(hi, (float)(kap - (double)hi)); }
        else kzt[idx] = kap;
    }
}

// ---------------------------------------------------------------------------------------------------
// forward rows.  smem per pair: landing line (source row, <= 16 KB) | exchange line of half 0 | exchange line of half 1
// ---------------------------------------------------------------------------------------------------
constexpr int K64_PAIR_BYTES = K64_L * 8 + 2 * K32_LP * 8;
constexpr size_t K64_ROWS_SMEM = (size_t)K64_PAIRS * K64_PAIR_BYTES + (size_t)K32_TW * 8 + K64_PAIRS * 2 * 8;

// IN: 0 complex64 rows, 1 amplitude + phase rows, 2 constant amplitude + phase rows
template <int IN, bool PADDED>
__global__ void __launch_bounds__(64 * K64_PAIRS, 2) k64_rows_fwd_bulk(const Params p, int plane0, int nlines) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int LINE_B = K32_L * 8;                                 // one half of a spectrum row
    const int t = threadIdx.x, pr = t >> 6, h = (t >> 5) & 1, lane = t & 31;
    unsigned char* land = smem_raw + (size_t)pr * K64_PAIR_BYTES;
    float2* xch = reinterpret_cast<float2*>(land + K64_L * 8) + h * K32_LP;
    float2* tw = reinterpret_cast<float2*>(smem_raw + (size_t)K64_PAIRS * K64_PAIR_BYTES);
    uint64_t* bars = reinterpret_cast<uint64_t*>(tw + K32_TW);
    for (int i = t; i < K32_TW; i += blockDim.x) tw[i] = __ldg(p.tw32 + i);
    if (t < K64_PAIRS) mbar_init(bars + t, 1);
    fence_mbar_init();
    __syncthreads();
    uint64_t* bar = bars + pr;
    const uint64_t pol_in = policy_evict_first(), pol_ws = policy_evict_normal();
    const int stride = gridDim.x * K64_PAIRS;
    const int N = PADDED ? p.N : K64_L;
    const unsigned row_bytes = (unsigned)N * (IN == 2 ? 4u : 8u);
    const float amp0 = IN == 2 ? __ldg((const float*)p.in0) : 0.f;
    auto request = [&](int gline) {                                  // lane 0 of half 0 only
        const size_t row = ((size_t)(plane0 + gline / N) * N + gline % N) * N;
        mbar_expect_tx(bar, row_bytes);
        if constexpr (IN == 1) {
            bulk_load(land, (const float*)p.in0 + row, row_bytes / 2, bar, pol_in);
            bulk_load(land + row_bytes / 2, (const float*)p.in1 + row, row_bytes / 2, bar, pol_in);
        } else if constexpr (IN == 2) {
            bulk_load(land, (const float*)p.in1 + row, row_bytes, bar, pol_in);
        } else {
            bulk_load(land, (const float2*)p.in0 + row, row_bytes, bar, pol_in);
        }
    };
    auto fetch = [&](int pos) -> float2 {                            // element `pos` of the padded row
        int x = pos;
        bool in = true;
        if constexpr (PADDED) { x -= p.P; in = !p.adj || (x >= 0 && x < N); x = min(max(x, 0), N - 1); }
        float2 val;
        if constexpr (IN == 0) {
            val = reinterpret_cast<const float2*>(land)[x];
        } else {
            const float a = IN == 1 ? reinterpret_cast<const float*>(land)[x] : amp0;
            const float ph = reinterpret_cast<const float*>(land)[(IN == 1 ? N : 0) + x] * p.in_scale;
            float sn, cs;
            sincos_reduced(ph, &sn, &cs);
            val = make_float2(a * cs, a * sn);
        }
        return (!PADDED || in) ? val : make_float2(0.f, 0.f);
    };
    int gline = blockIdx.x * K64_PAIRS + pr;
    if (h == 0 && lane == 0 && gline < nlines) request(gline);
    unsigned phase = 0;
    for (; gline < nlines; gline += stride) {
        mbar_wait(bar, phase);
        phase ^= 1u;
        float2 v[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            const float2 lo = fetch(lane + 32 * i), hi = fetch(lane + 32 * i + 1024);
            v[i] = h == 0 ? make_float2(lo.x + hi.x, lo.y + hi.y) : make_float2(lo.x - hi.x, lo.y - hi.y);
        }
        loads_landed(v);
        pair_barrier(1 + pr);                                        // both halves have consumed the landing line
        if (lane == 0) {
            if (h == 0 && gline + stride < nlines) request(gline + stride);   // ... lands while this row is transformed
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");    // this half's previous store has left its line
        }
        if (h == 1) k64_twiddle64<-1>(v);
        fwd32_first(v);
        __syncwarp();
        sts16<RowLayout32, 5>(v, xch + lane);
        __syncwarp();
        lds16<RowLayout32, 0>(v, xch + 33 * lane);
        if (h == 1) k64_twiddle2048<-1>(v);
        fwd32_table(v, tw + lane);
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 32; ++i) xch[lane + 32 * i] = v[i];     // dense: column 1024 h + (lane + 32 i) = frequency 2 m + h
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
            bulk_store(p.ws + (size_t)gline * K64_L + h * K32_L, xch, LINE_B, pol_ws);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------------
// inverse rows.  smem per pair: landing halves (2 x 8 KB) | exchange line of half 0 | exchange line of half 1
// ---------------------------------------------------------------------------------------------------
template <bool INTENSITY, bool PADDED>
__global__ void __launch_bounds__(64 * K64_PAIRS, 2) k64_rows_inv_bulk(const Params p, int plane0, int nlines) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int LINE_B = K32_L * 8;
    const int t = threadIdx.x, pr = t >> 6, h = (t >> 5) & 1, lane = t & 31;
    unsigned char* pairbase = smem_raw + (size_t)pr * K64_PAIR_BYTES;
    const float2* land = reinterpret_cast<const float2*>(pairbase + h * LINE_B);
    float2* xch0 = reinterpret_cast<float2*>(pairbase + K64_L * 8);
    float2* xch = xch0 + h * K32_LP;
    const float2* xch_other = xch0 + (1 - h) * K32_LP;
    float2* tw = reinterpret_cast<float2*>(smem_raw + (size_t)K64_PAIRS * K64_PAIR_BYTES);
    uint64_t* bars = reinterpret_cast<uint64_t*>(tw + K32_TW);
    for (int i = t; i < K32_TW; i += blockDim.x) tw[i] = __ldg(p.tw32 + i);
    if (t < 2 * K64_PAIRS) mbar_init(bars + t, 1);
    fence_mbar_init();
    __syncthreads();
    uint64_t* bar = bars + 2 * pr + h;                               // every half waits for its own 8 KB piece
    const uint64_t pol_out = policy_evict_first(), pol_ws = policy_evict_normal();
    const int stride = gridDim.x * K64_PAIRS;
    const int N = PADDED ? p.N : K64_L, P = PADDED ? p.P : 0;
    const bool folding = PADDED && p.adj;
    auto request = [&](int gl) {
        mbar_expect_tx(bar, LINE_B);
        bulk_load(const_cast<float2*>(land), p.ws + (size_t)gl * K64_L + h * K32_L, LINE_B, bar, pol_ws);
    };
    int gline = blockIdx.x * K64_PAIRS + pr;
    if (lane == 0 && gline < nlines) request(gline);
    unsigned phase = 0;
    for (; gline < nlines; gline += stride) {
        mbar_wait(bar, phase);
        phase ^= 1u;
        float2 v[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = land[lane + 32 * i];     // frequency 2 (lane + 32 i) + h
        loads_landed(v);
        __syncwarp();
        {   // the intermediate piece is dead: drop its dirty L2 lines instead of writing them back to HBM
            const char* src = reinterpret_cast<const char*>(p.ws + (size_t)gline * K64_L + h * K32_L);
            asm volatile("discard.global.L2 [%0], 128;" ::"l"(src + (size_t)lane * 128) : "memory");
            asm volatile("discard.global.L2 [%0], 128;" ::"l"(src + (size_t)(lane + 32) * 128) : "memory");
        }
        if (lane == 0) {
            if (gline + stride < nlines) request(gline + stride);
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the previous output store has left this half's line
        }
        inv32_first(v);
        if (h == 1) k64_twiddle2048<1>(v);
        __syncwarp();
        sts16<RowLayout32, 0>(v, xch + 33 * lane);
        __syncwarp();
        lds16<RowLayout32, 5>(v, xch + lane);
        inv32_table(v, tw + lane);                                   // v[i] = a[k] (h = 0) or W_2048^-lane-free b[k], k = lane + 32 i
        if (h == 1) k64_twiddle64<1>(v);
        __syncwarp();
        // radix-2 level: exchange the halves through the (now free) exchange lines, dense [k]
#pragma unroll
        for (int i = 0; i < 32; ++i) xch[lane + 32 * i] = v[i];
        pair_barrier(1 + pr);
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            const float2 o = xch_other[lane + 32 * i];
            v[i] = h == 0 ? make_float2(v[i].x + o.x, v[i].y + o.y) : make_float2(o.x - v[i].x, o.y - v[i].y);   // x[k + 1024 h]
        }
        pair_barrier(1 + pr);                                        // both halves have read both lines: they become staging lines
        const int img = gline / N, y = gline % N, plane = plane0 + img;
        // half h holds positions 1024 h + lane + 32 i of the padded row; crop to [P, P + N) and stage densely
        float2 fl = make_float2(0.f, 0.f), fr = make_float2(0.f, 0.f);
        if (folding) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const int pos = 1024 * h + lane + 32 * i;
                if (pos < P) { fl.x += v[i].x; fl.y += v[i].y; }
                if (pos >= P + N) { fr.x += v[i].x; fr.y += v[i].y; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                fl.x += __shfl_xor_sync(0xffffffffu, fl.x, o); fl.y += __shfl_xor_sync(0xffffffffu, fl.y, o);
                fr.x += __shfl_xor_sync(0xffffffffu, fr.x, o); fr.y += __shfl_xor_sync(0xffffffffu, fr.y, o);
            }
        }
        // this half's first output column and how many it owns (P <= 1024 <= P + N always: both halves own N / 2 columns)
        const int x0 = PADDED ? (h == 0 ? 0 : 1024 - P) : 1024 * h;
        const int cnt = PADDED ? (h == 0 ? 1024 - P : P + N - 1024) : 1024;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            const int x = 1024 * h + lane + 32 * i - P;
            if (!PADDED || (x >= 0 && x < N)) {
                float2 u = v[i];
                if (PADDED && x == 0) { u.x += fl.x; u.y += fl.y; }          // fold sums live in the half that owns the edge column
                if (PADDED && x == N - 1) { u.x += fr.x; u.y += fr.y; }
                if constexpr (INTENSITY) reinterpret_cast<float*>(xch)[x - x0] = fmaf(u.x, u.x, u.y * u.y);
                else xch[x - x0] = u;
            }
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0 && cnt > 0) {
            const size_t row = ((size_t)plane * N + y) * N + x0;
            if constexpr (INTENSITY) bulk_store((float*)p.out0 + row, xch, (unsigned)cnt * 4u, pol_out);
            else bulk_store((float2*)p.out0 + row, xch, (unsigned)cnt * 8u, pol_out);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------------
// column pass: slabs of 4 columns, thread (h, tl, c), 256 threads, 2 CTAs per SM.  Works for any workspace column order
// (the kappa table is in that order).
//   smem: exchange slabs [2][1056][4] float2 (their first N dense rows double as the landing zone) | kappa [1025][4]
//         double | half twiddle table | fold [2][4]
// ---------------------------------------------------------------------------------------------------
constexpr int K64_XROWS = ColLayout32<K64_CC>::rows(K32_L);           // 1056
constexpr size_t K64_COLS_SMEM = (size_t)2 * K64_XROWS * K64_CC * 8 + (size_t)(K64_L / 2 + 1) * K64_CC * 8 + (size_t)K32_TW * 8 + 2 * 8 * K64_CC * 8;   // ... | fold partials [2][8 warps][4]

__device__ __forceinline__ void k64_stage_raw(float2* raw, const float2* img_ws, int col0, int nrows) {
    constexpr int Q = K64_CC / 2;
    for (int j = threadIdx.x; j < nrows * Q; j += 64 * K64_CC) {
        const int r = j / Q, q = j % Q;
        cp_async16(raw + r * K64_CC + 2 * q, img_ws + (size_t)r * K64_L + col0 + 2 * q);
    }
}
__device__ __forceinline__ void k64_stage_kz(double* kz_s, const double* kzt, int col0) {
    constexpr int Q = K64_CC / 2;
    for (int j = threadIdx.x; j < (K64_L / 2 + 1) * Q; j += 64 * K64_CC) {
        const int ru = j / Q, q = j % Q;
        cp_async16(kz_s + ru * K64_CC + 2 * q, kzt + (size_t)ru * K64_L + col0 + 2 * q);
    }
}

// PAIRS: the kappa slab holds fp32 (hi, lo) pairs and t = c kappa is formed in double-float fp32 (no fp64, no F2F; see
// k32t_apply_h); otherwise fp64 entries (the table of the generic row kernels' column order).
// BL: band-limited calls (p.band_limit).  A template parameter here, not a runtime test as in the other column kernels:
// the padded kernel is at its register limit, and the plain instantiations stay the code they were.
template <bool PADDED, bool PAIRS, bool BL = false>
__global__ void __launch_bounds__(64 * K64_CC, 2) k64_cols(const Params p, int plane0, int nimg) {
    constexpr int L = K64_L, CC = K64_CC, nslab = L / CC;
    using LAY = ColLayout32<CC>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* raw = reinterpret_cast<float2*>(smem_raw);               // dense [N][CC] landing zone = start of the exchange slabs
    double* kz_s = reinterpret_cast<double*>(raw + 2 * K64_XROWS * CC);
    float2* tw = reinterpret_cast<float2*>(kz_s + (L / 2 + 1) * CC);
    float2* fold = tw + K32_TW;
    const int t = threadIdx.x, c = t % CC, tl = (t / CC) & 31, h = t / (32 * CC);
    float2* slab = raw + (size_t)h * K64_XROWS * CC;                  // this half's exchange slab [1056][CC]
    const float2* slab_other = raw + (size_t)(1 - h) * K64_XROWS * CC;
    const int N = PADDED ? p.N : L, P = PADDED ? p.P : 0;
    const int total = nimg * nslab, step = gridDim.x;
    for (int i = t; i < K32_TW; i += 64 * CC) tw[i] = __ldg(p.tw32 + i);
    int wi = blockIdx.x;
    if (wi < total) {
        k64_stage_raw(raw, src_base(p) + (size_t)src_slot(p, plane0, wi / nslab) * N * L, (wi % nslab) * CC, N);
        k64_stage_kz(kz_s, p.kzt, (wi % nslab) * CC);
        cp_async_commit();
    }
    float2* col = slab + c;
    const double MAGIC = 6755399441055744.0;
    for (; wi < total; wi += step) {
        const int img = wi / nslab, slab_i = wi % nslab, plane = plane0 + img;
        const int col0 = slab_i * CC;
        const int nxt = wi + step;
        float2* img_ws = p.ws + (size_t)img * N * L;
        cp_async_wait<0>();
        __syncthreads();
        // ---- radix-2 DIF level straight from the dense rows: positions k = tl + 32 i and k + 1024 ----
        float2 v[32];
        if (!PADDED) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const float2 lo = raw[(tl + 32 * i) * CC + c], hi = raw[(tl + 32 * i + 1024) * CC + c];
                v[i] = h == 0 ? make_float2(lo.x + hi.x, lo.y + hi.y) : make_float2(lo.x - hi.x, lo.y - hi.y);
            }
        } else if (p.adj) {                                          // zero embedding
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const int r0 = tl + 32 * i - P, r1 = r0 + 1024;
                const float2 lo = (r0 >= 0 && r0 < N) ? raw[r0 * CC + c] : make_float2(0.f, 0.f);
                const float2 hi = (r1 >= 0 && r1 < N) ? raw[r1 * CC + c] : make_float2(0.f, 0.f);
                v[i] = h == 0 ? make_float2(lo.x + hi.x, lo.y + hi.y) : make_float2(lo.x - hi.x, lo.y - hi.y);
            }
        } else {                                                     // replicate padding
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const int r0 = tl + 32 * i - P, r1 = r0 + 1024;
                const float2 lo = raw[min(max(r0, 0), N - 1) * CC + c], hi = raw[min(max(r1, 0), N - 1) * CC + c];
                v[i] = h == 0 ? make_float2(lo.x + hi.x, lo.y + hi.y) : make_float2(lo.x - hi.x, lo.y - hi.y);
            }
        }
        __syncthreads();                                             // the dense rows are consumed
        const double cph = phase_constant_of(p, plane / p.C);
        // band limit: column col0 + c holds frequency v (split order with the warp-pair row kernels, digit-reversed
        // otherwise); rows |k(u)| <= lim_u are kept if |k(v)| is within the limit, none otherwise
        int lim_u = L;
        if constexpr (BL) {
            const int vpos = PAIRS ? 2 * ((col0 + c) & 1023) + ((col0 + c) >> 10) : freq_of_pos(11, col0 + c);
            const int lim = band_limit_of(p, plane / p.C);
            lim_u = (vpos <= L / 2 ? vpos : L - vpos) <= lim ? lim : -1;
        }
        // ---- forward 1024-point transform of this half ----
        if (h == 1) k64_twiddle64<-1>(v);
        fwd32_first(v);
        sts16<LAY, 5>(v, col + tl * CC);
        __syncthreads();
        lds16<LAY, 0>(v, col + 33 * tl * CC);
        if (h == 1) k64_twiddle2048<-1>(v);
        fwd32_table(v, tw + tl);                                     // v[i] = column frequency u = 2 (tl + 32 i) + h
        // ---- transfer function ----
        if constexpr (PAIRS) {
            const float c_hi = (float)cph, c_lo = (float)(cph - (double)c_hi);
            const float MAGICF = 12582912.f;
            const float2* kp = reinterpret_cast<const float2*>(kz_s);
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const int u = 2 * (tl + 32 * i) + h;
                const int ru = u <= L / 2 ? u : L - u;
                const float2 k = kp[ru * CC + c];
                const float pp = __fmul_rn(k.x, c_hi);
                float sacc = __fmaf_rn(k.x, c_hi, -pp);
                sacc = __fmaf_rn(k.y, c_hi, sacc);
                sacc = __fmaf_rn(k.x, c_lo, sacc);
                const float kk = __fadd_rn(__fadd_rn(pp, MAGICF), -MAGICF);
                const float r = __fadd_rn(__fadd_rn(pp, -kk), sacc);
                float sn, cn;
                __sincosf(r * 6.283185307179586f, &sn, &cn);
                const float sc = ru <= lim_u ? p.inv_m2 : 0.f;       // H = 0 outside the band limit
                if (p.h_mode == H_DERIV) {
                    const double kz_l = ((double)k.x + (double)k.y) * (6.283185307179586 * p.lambda);
                    v[i] = cmul_scaled(v[i], -sn, cn, (float)(kz_l - p.kshift) * sc);
                } else {
                    v[i] = cmul_scaled(v[i], cn, sn, sc);
                }
            }
        } else {
            const double k2pl = 6.283185307179586 * p.lambda;
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const int u = 2 * (tl + 32 * i) + h;
                const int ru = u <= L / 2 ? u : L - u;
                const double kap = kz_s[ru * CC + c];
                const double tt = kap * cph;
                const double rr = tt - __dadd_rn(__dadd_rn(tt, MAGIC), -MAGIC);
                float sn, cn;
                __sincosf((float)rr * 6.283185307179586f, &sn, &cn);
                const float sc = ru <= lim_u ? p.inv_m2 : 0.f;       // H = 0 outside the band limit
                if (p.h_mode == H_DERIV) v[i] = cmul_scaled(v[i], -sn, cn, (float)(kap * k2pl - p.kshift) * sc);
                else v[i] = cmul_scaled(v[i], cn, sn, sc);
            }
        }
        // ---- inverse 1024-point transform of this half ----
        inv32_first(v);
        if (h == 1) k64_twiddle2048<1>(v);
        sts16<LAY, 0>(v, col + 33 * tl * CC);
        __syncthreads();                                             // every thread is done with kz_s too
        if (nxt < total && (nxt % nslab) != slab_i) k64_stage_kz(kz_s, p.kzt, (nxt % nslab) * CC);
        lds16<LAY, 5>(v, col + tl * CC);
        inv32_table(v, tw + tl);
        if (h == 1) k64_twiddle64<1>(v);
        __syncthreads();                                             // all exchange reads done: the slabs become the radix-2 buffers
        // ---- radix-2 level: x[k] = a + b', x[k + 1024] = a - b' (dense rows k = tl + 32 i of each half's slab) ----
#pragma unroll
        for (int i = 0; i < 32; ++i) slab[(tl + 32 * i) * CC + c] = v[i];
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            const float2 o = slab_other[(tl + 32 * i) * CC + c];
            v[i] = h == 0 ? make_float2(v[i].x + o.x, v[i].y + o.y) : make_float2(o.x - v[i].x, o.y - v[i].y);   // row 1024 h + tl + 32 i
        }
        __syncthreads();                                             // the slabs are dead: land the next item in them
        if (nxt < total) k64_stage_raw(raw, src_base(p) + (size_t)src_slot(p, plane0, nxt / nslab) * N * L, (nxt % nslab) * CC, N);
        cp_async_commit();
        // ---- store rows [P, P+N) (crop); adjoint: fold the padding rows onto rows P and P+N-1 first ----
        float2* dst = img_ws + col0 + c;
        if constexpr (!PADDED) {
#pragma unroll
            for (int i = 0; i < 32; ++i) __stcg(dst + (size_t)(1024 * h + tl + 32 * i) * L, v[i]);
        } else {
            float2 fl = make_float2(0.f, 0.f), fr = make_float2(0.f, 0.f);
            if (p.adj) {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const int pos = 1024 * h + tl + 32 * i;
                    if (pos < P) { fl.x += v[i].x; fl.y += v[i].y; }
                    if (pos >= P + N) { fr.x += v[i].x; fr.y += v[i].y; }
                }
                // deterministic column sums (no floating-point atomics): lanes of a warp = 8 rows x 4 columns -> xor shuffles
                // over the row bits, then the 8 warps' partials are added in a fixed order by every thread
#pragma unroll
                for (int o = CC; o < 32; o <<= 1) {
                    fl.x += __shfl_xor_sync(0xffffffffu, fl.x, o); fl.y += __shfl_xor_sync(0xffffffffu, fl.y, o);
                    fr.x += __shfl_xor_sync(0xffffffffu, fr.x, o); fr.y += __shfl_xor_sync(0xffffffffu, fr.y, o);
                }
                if ((t & 31) < CC) { fold[(t >> 5) * CC + c] = fl; fold[8 * CC + (t >> 5) * CC + c] = fr; }
                __syncthreads();
                fl = make_float2(0.f, 0.f); fr = make_float2(0.f, 0.f);
#pragma unroll
                for (int w = 0; w < 8; ++w) {
                    const float2 a = fold[w * CC + c], b2 = fold[8 * CC + w * CC + c];
                    fl.x += a.x; fl.y += a.y; fr.x += b2.x; fr.y += b2.y;
                }
                __syncthreads();
            }
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const int r = 1024 * h + tl + 32 * i - P;
                if (r >= 0 && r < N) {
                    float2 u = v[i];
                    if (r == 0) { u.x += fl.x; u.y += fl.y; }
                    if (r == N - 1) { u.x += fr.x; u.y += fr.y; }
                    __stcg(dst + (size_t)r * L, u);
                }
            }
        }
    }
    cp_async_wait<0>();
}

}  // namespace asmb
