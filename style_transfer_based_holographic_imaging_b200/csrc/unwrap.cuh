// unwrap.cuh -- 2-D phase unwrapping on the device (SURVEY.md 8f row 4): the per-image host loop of
// utils/functions.py:44-59 (skimage.restoration.unwrap_phase after a .cpu() sync) as three stream-ordered launches.
//
// Algorithm: Herraez, Burton, Lalor, Gdeisat, "Fast two-dimensional phase-unwrapping algorithm based on sorting by
// reliability following a noncontinuous path", Appl. Opt. 41 (2002) -- the algorithm scikit-image's unwrap_phase implements
// for 2-D input (scikit-image is NOT in this image and not vendored by the reference: parity with it is unpinned; the
// restatement under oracle/unwrap_oracle.py follows the same published steps and pins this kernel instead):
//   1. reliability of an interior pixel = H^2 + V^2 + D1^2 + D2^2 of the wrapped second differences (small = reliable);
//      border pixels get a large constant (they join last);
//   2. an edge (horizontal / vertical neighbours) has the sum of its pixels' reliabilities and the 2 pi jump count
//      between them: -1 if left - right > pi, +1 if < -pi, else 0;
//   3. edges are sorted by reliability (ascending; cub segmented radix sort, stable: ties in edge order: all horizontal
//      edges row by row, then all vertical ones);
//   4. edges are visited in that order; two pixels of different groups merge their groups, the group that joins is shifted
//      by the multiple of 2 pi that makes the edge consistent: a single pixel joins its neighbour's group, otherwise the
//      group with fewer pixels joins the larger one (ties: the first pixel's group joins);
//   5. unwrapped = fl32(wrapped + 2 pi * increment), the sum in double.
// Step 4 is sequential per image (a weighted union-find with per-node offsets, one thread per image, images in parallel);
// everything else is data parallel.
#pragma once
#include <cub/device/device_segmented_radix_sort.cuh>

namespace asmb {

__device__ __forceinline__ float uw_wrap(float x) {
    const float PI = 3.14159265358979323846f, TWO_PI = 6.28318530717958647692f;
    return x > PI ? x - TWO_PI : (x < -PI ? x + TWO_PI : x);
}

// reliability per pixel
__global__ void k_unwrap_reliability(const float* __restrict__ ph, float* __restrict__ rel, int B, int H, int W) {
    const size_t n = (size_t)B * H * W;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < n; idx += (size_t)gridDim.x * blockDim.x) {
        const int j = (int)(idx % W), i = (int)((idx / W) % H);
        if (i == 0 || j == 0 || i == H - 1 || j == W - 1) { rel[idx] = 9999999.f; continue; }
        const float* p = ph + idx;
        const float c = p[0];
        const float h = uw_wrap(p[-1] - c) - uw_wrap(c - p[1]);
        const float v = uw_wrap(p[-W] - c) - uw_wrap(c - p[W]);
        const float d1 = uw_wrap(p[-W - 1] - c) - uw_wrap(c - p[W + 1]);
        const float d2 = uw_wrap(p[-W + 1] - c) - uw_wrap(c - p[W - 1]);
        rel[idx] = __fadd_rn(__fadd_rn(__fmul_rn(h, h), __fmul_rn(v, v)), __fadd_rn(__fmul_rn(d1, d1), __fmul_rn(d2, d2)));
    }
}

// edge e of an image: e < H (W - 1): horizontal (i, j)-(i, j + 1), i = e / (W - 1); else vertical (i, j)-(i + 1, j)
__device__ __forceinline__ void uw_edge_pixels(int e, int H, int W, int* p1, int* p2) {
    const int nh = H * (W - 1);
    if (e < nh) { const int i = e / (W - 1), j = e % (W - 1); *p1 = i * W + j; *p2 = *p1 + 1; }
    else { const int q = e - nh; *p1 = q; *p2 = q + W; }
}

__global__ void k_unwrap_edges(const float* __restrict__ ph, const float* __restrict__ rel, float* __restrict__ key,
                               int* __restrict__ id, int* __restrict__ seg, int B, int H, int W) {
    const int E = H * (W - 1) + (H - 1) * W;
    const size_t n = (size_t)B * E;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < n; idx += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(idx / E), e = (int)(idx % E);
        int p1, p2;
        uw_edge_pixels(e, H, W, &p1, &p2);
        const float* r = rel + (size_t)b * H * W;
        key[idx] = __fadd_rn(r[p1], r[p2]);
        id[idx] = (p1 << 1) | (e >= H * (W - 1) ? 1 : 0);             // payload: first pixel + direction (the merge loop needs no division)
    }
    if (blockIdx.x == 0) for (int b = threadIdx.x; b <= B; b += blockDim.x) seg[b] = b * E;
}

// Sequential merge, one thread per image.  parent / off / size / base: [B][H W] ints in the workspace.
//   inc(x) = base[root(x)] + sum of off[] on the path from x to its root
__global__ void k_unwrap_merge(const float* __restrict__ ph, const int* __restrict__ order, int* __restrict__ parent,
                               int* __restrict__ off, int* __restrict__ size, int* __restrict__ base, int H, int W) {
    const int P = H * W, E = H * (W - 1) + (H - 1) * W;
    const int b = blockIdx.x;
    ph += (size_t)b * P; order += (size_t)b * E;
    parent += (size_t)b * P; off += (size_t)b * P; size += (size_t)b * P; base += (size_t)b * P;
    for (int x = threadIdx.x; x < P; x += blockDim.x) { parent[x] = x; off[x] = 0; size[x] = 1; base[x] = 0; }
    __syncthreads();
    if (threadIdx.x != 0) return;
    const float PI = 3.14159265358979323846f;
    auto find = [&](int x, int* o) {          // root of x and inc(x) - base[root]; path halving keeps the offsets consistent
        int acc = 0;
        while (parent[x] != x) {
            const int px = parent[x];
            if (parent[px] != px) { off[x] += off[px]; parent[x] = parent[px]; }
            acc += off[x];
            x = parent[x];
        }
        *o = acc;
        return x;
    };
    for (int k = 0; k < E; ++k) {
        const int ev = order[k], p1 = ev >> 1, p2 = p1 + ((ev & 1) ? W : 1);
        int o1, o2;
        const int r1 = find(p1, &o1), r2 = find(p2, &o2);
        if (r1 == r2) continue;
        const float d = ph[p1] - ph[p2];
        const int e = d > PI ? -1 : (d < -PI ? 1 : 0);
        const int inc1 = base[r1] + o1, inc2 = base[r2] + o2;
        const bool group2_joins = size[r2] == 1 ? true : (size[r1] == 1 ? false : size[r1] > size[r2]);
        if (group2_joins) {                   // every pixel of group 2 += inc1 - e - inc2
            off[r2] = base[r2] + (inc1 - e - inc2) - base[r1];
            parent[r2] = r1; size[r1] += size[r2];
        } else {                              // every pixel of group 1 += inc2 + e - inc1
            off[r1] = base[r1] + (inc2 + e - inc1) - base[r2];
            parent[r1] = r2; size[r2] += size[r1];
        }
    }
}

// The same merge with every array in shared memory (images of up to 128 x 128 pixels: 16-bit parents / sizes / offsets and
// the wrapped phase itself, 192 KB): the sequential loop runs at shared-memory instead of L2 latency (~10x).
constexpr int UW_SMEM_PIX = 16384;
__global__ void k_unwrap_merge_smem(const float* __restrict__ ph_g, const int* __restrict__ order, int* __restrict__ parent_g,
                                    int* __restrict__ off_g, int* __restrict__ base_g, int H, int W) {
    extern __shared__ __align__(16) unsigned char uw_smem[];
    const int P = H * W, E = H * (W - 1) + (H - 1) * W;
    float* ph = reinterpret_cast<float*>(uw_smem);
    unsigned short* parent = reinterpret_cast<unsigned short*>(ph + UW_SMEM_PIX);
    unsigned short* size = parent + UW_SMEM_PIX;
    short* off = reinterpret_cast<short*>(size + UW_SMEM_PIX);
    short* base = off + UW_SMEM_PIX;
    const int b = blockIdx.x;
    ph_g += (size_t)b * P; order += (size_t)b * E;
    for (int x = threadIdx.x; x < P; x += blockDim.x) { ph[x] = ph_g[x]; parent[x] = (unsigned short)x; off[x] = 0; size[x] = 1; base[x] = 0; }
    __syncthreads();
    if (threadIdx.x == 0) {
        const float PI = 3.14159265358979323846f;
        auto find = [&](int x, int* o) {
            int acc = 0;
            while (parent[x] != x) {
                const int px = parent[x];
                if (parent[px] != px) { off[x] = (short)(off[x] + off[px]); parent[x] = parent[px]; }
                acc += off[x];
                x = parent[x];
            }
            *o = acc;
            return x;
        };
        int nxt = E > 0 ? order[0] : 0;
        for (int k = 0; k < E; ++k) {
            const int e_id = nxt;
            if (k + 1 < E) nxt = order[k + 1];                       // the next edge id is in flight during this merge
            const int p1 = e_id >> 1, p2 = p1 + ((e_id & 1) ? W : 1);
            int o1, o2;
            const int r1 = find(p1, &o1), r2 = find(p2, &o2);
            if (r1 == r2) continue;
            const float d = ph[p1] - ph[p2];
            const int e = d > PI ? -1 : (d < -PI ? 1 : 0);
            const int inc1 = base[r1] + o1, inc2 = base[r2] + o2;
            const bool group2_joins = size[r2] == 1 ? true : (size[r1] == 1 ? false : size[r1] > size[r2]);
            if (group2_joins) {
                off[r2] = (short)(base[r2] + (inc1 - e - inc2) - base[r1]);
                parent[r2] = (unsigned short)r1; size[r1] = (unsigned short)(size[r1] + size[r2]);
            } else {
                off[r1] = (short)(base[r1] + (inc2 + e - inc1) - base[r2]);
                parent[r1] = (unsigned short)r2; size[r2] = (unsigned short)(size[r2] + size[r1]);
            }
        }
    }
    __syncthreads();
    for (int x = threadIdx.x; x < P; x += blockDim.x) {              // hand the forest to k_unwrap_apply
        parent_g[(size_t)b * P + x] = parent[x]; off_g[(size_t)b * P + x] = off[x]; base_g[(size_t)b * P + x] = base[x];
    }
}

// unwrapped = fl32(ph + 2 pi k) with the sum in double: the value the reference's float64 unwrap gives after its callers'
// .float().  (ph and out are not __restrict__: out may alias ph.)
__global__ void k_unwrap_apply(const float* ph, float* out, const int* __restrict__ parent,
                               const int* __restrict__ off, const int* __restrict__ base, int B, int P) {
    const size_t n = (size_t)B * P;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < n; idx += (size_t)gridDim.x * blockDim.x) {
        const size_t img = idx / P * P;
        int x = (int)(idx - img), acc = 0;
        while (parent[img + x] != x) { acc += off[img + x]; x = parent[img + x]; }
        out[idx] = __double2float_rn(__dadd_rn((double)ph[idx], __dmul_rn(6.283185307179586476925, (double)(acc + base[img + x]))));
    }
}

struct UnwrapLayout { size_t rel, key_in, key_out, id_in, id_out, seg, parent, off, size, base, cub, cub_bytes, total; };

// false for every shape asm_b200_unwrap rejects, so that asm_b200_unwrap_workspace_bytes reports 0 for exactly those:
// H, W >= 3, H W <= 2^28, and B E <= INT_MAX (E edges per image; cub's item count and the segment offsets are ints).
static bool unwrap_layout(int B, int H, int W, UnwrapLayout* L) {
    if (B <= 0 || H < 3 || W < 3 || (long long)H * W > (1ll << 28)) return false;
    if ((long long)B * ((long long)H * (W - 1) + (long long)(H - 1) * W) > 0x7fffffffll) return false;
    const size_t P = (size_t)B * H * W, E = (size_t)B * ((size_t)H * (W - 1) + (size_t)(H - 1) * W);
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o += (bytes + 255) / 256 * 256; return at; };
    L->rel = take(P * 4); L->key_in = take(E * 4); L->key_out = take(E * 4); L->id_in = take(E * 4); L->id_out = take(E * 4);
    L->seg = take((size_t)(B + 1) * 4);
    L->parent = take(P * 4); L->off = take(P * 4); L->size = take(P * 4); L->base = take(P * 4);
    // cub's temporary storage for the pair sort: one alternate buffer for the keys and one for the values (each rounded up
    // to 256 bytes) plus alignment slack.  A closed-form bound instead of cub's size query keeps the layout a pure function
    // of (B, H, W): the query goes through the CUDA runtime and would report (and swallow) an unrelated pending error.
    const size_t cb = 2 * ((E * 4 + 255) / 256 * 256) + 4096;
    L->cub_bytes = cb; L->cub = take(cb);
    L->total = o;
    return true;
}

}  // namespace asmb
