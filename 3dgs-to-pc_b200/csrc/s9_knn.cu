// s9_knn.cu — exact k-nearest-neighbour mean distances and the statistical outlier mask (point-cloud cleaning).
//
// Reference semantics restated (not copied):
//   mesh_handler.py:89-94       clean_point_cloud -> Open3D PointCloud.remove_statistical_outlier(nb_neighbors=20,
//                               std_ratio): per point the mean distance to its k nearest points (itself included),
//                               mean / std (Bessel) of those over the points with a non-zero mean distance (divided by
//                               the FULL point count), keep 0 < avg < mean + std_ratio * std.
// Here, per call of g2pc_knn_mean_distance (no host sync):
//   1. bounds        one grid-stride min/max reduction over the finite points + a one-CTA fold;
//   2. morton keys   63-bit keys (21 bits per axis over the bounding box), cub radix sort of (key, index) pairs (library),
//                    then a Morton-ordered packed copy {x, y, z, bits(original index)} (16 bytes per point);
//   3. tree          buckets of 32 consecutive sorted points; an implicit complete binary tree of AABBs over them (node 1
//                    = root, leaves P..2P-1), built bottom-up in ONE kernel (the second child to finish builds its
//                    parent).  The boxes hold the real float32 coordinates, so they bound the points exactly;
//   4. queries       one warp per bucket: the warp's 32 queries seed their top-k from their own bucket (shuffles), then
//                    walk the tree together — a node is opened when ANY lane's lower bound beats its k-th distance, a
//                    leaf's 32 points are loaded coalesced and broadcast.  The stack lives in the lanes' registers (one
//                    entry per lane, depth <= 27).  Layout only changes the speed: the pruning is conservative, so the
//                    result is the exact kNN whatever the Morton order looks like.
// Selection and pruning run on float32 squared distances.  The lower bound is scaled by (1 - 1e-6) before it is compared
// with the k-th distance, which covers the rounding of both (a few ulp each), so no node holding a point that would enter
// the top-k is ever pruned.  Candidates whose float32 distances tie within rounding may swap at the k-th place; the k
// chosen distances are then recomputed in float64 from the float32 coordinates, so avg is off by at most that rounding
// (~1e-7 relative).  A query with a non-finite coordinate gets avg = NaN (counted by g2pc_outlier_mask).
#include <cub/cub.cuh>
#include <float.h>
#include <math.h>

#include "common.cuh"

namespace {

constexpr int BUCKET = 32;       // points per leaf bucket = queries per warp
constexpr int QB = 256;          // threads per CTA of the query kernel
constexpr int NB_BOUNDS = 592;   // CTAs of the bounds reduction (4 per SM)
constexpr int RED_CTAS = 1024;   // max CTAs of the outlier reductions
constexpr float PRUNE_SCALE = 0.999999f;

inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

inline int64_t pow2_at_least(int64_t v) {
    int64_t p = 1;
    while (p < v) p <<= 1;
    return p;
}

struct KnnLayout {
    int64_t nb, P;
    size_t keys, vals_in, vals_out, lo, hi, flags, bounds, tmp, tmp_bytes, total;
};

// [keys_in n u64 | keys_out n u64] (reused as the packed float4 points after the sort) [vals_in n i32] [vals_out n i32]
// [box lo 2P float4] [box hi 2P float4] [flags P u32] [bounds partials (NB_BOUNDS + 1) x 8 f32] [cub temp]
KnnLayout knn_layout(int64_t n) {
    KnnLayout L;
    L.nb = (n + BUCKET - 1) / BUCKET;
    L.P = pow2_at_least(L.nb > 0 ? L.nb : 1);
    size_t off = 0;
    L.keys = off; off += align256((size_t)n * 16);
    L.vals_in = off; off += align256((size_t)n * 4);
    L.vals_out = off; off += align256((size_t)n * 4);
    L.lo = off; off += align256((size_t)L.P * 2 * 16);
    L.hi = off; off += align256((size_t)L.P * 2 * 16);
    L.flags = off; off += align256((size_t)L.P * 4);
    L.bounds = off; off += align256((size_t)(NB_BOUNDS + 1) * 8 * 4);
    size_t tb = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                    (const int32_t*)nullptr, (int32_t*)nullptr, n, 0, 63);
    L.tmp = off; L.tmp_bytes = align256(tb); off += L.tmp_bytes;
    L.total = off;
    return L;
}

__device__ __forceinline__ bool finite3(float x, float y, float z) {
    return isfinite(x) && isfinite(y) && isfinite(z);
}

// ---- 1. bounds ---------------------------------------------------------------------------------------------------
// partial[b] = {min x, min y, min z, -, max x, max y, max z, -} over the finite points of CTA b's grid-stride share
__global__ void __launch_bounds__(256) bounds_kernel(const float* __restrict__ xyz, int64_t n, float* __restrict__ partial) {
    __shared__ float s[8][8];
    float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
        const float x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2];
        if (!finite3(x, y, z)) continue;
        lo[0] = fminf(lo[0], x); lo[1] = fminf(lo[1], y); lo[2] = fminf(lo[2], z);
        hi[0] = fmaxf(hi[0], x); hi[1] = fmaxf(hi[1], y); hi[2] = fmaxf(hi[2], z);
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
    }
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        for (int a = 0; a < 3; ++a) { s[w][a] = lo[a]; s[w][4 + a] = hi[a]; }
    }
    __syncthreads();
    if (threadIdx.x < 8) {
        const int a = threadIdx.x;
        if (a != 3 && a != 7) {
            float v = s[0][a];
            for (int k = 1; k < 8; ++k) v = a < 4 ? fminf(v, s[k][a]) : fmaxf(v, s[k][a]);
            partial[blockIdx.x * 8 + a] = v;
        }
    }
}

// one CTA: fold the partials -> out = {min x, min y, min z, -, scale x, scale y, scale z, -}
__global__ void __launch_bounds__(32) bounds_final_kernel(const float* __restrict__ partial, int nparts,
                                                         float* __restrict__ out) {
    const int a = threadIdx.x;
    if (a >= 3) return;
    float lo = FLT_MAX, hi = -FLT_MAX;
    for (int b = 0; b < nparts; ++b) { lo = fminf(lo, partial[b * 8 + a]); hi = fmaxf(hi, partial[b * 8 + 4 + a]); }
    const float ext = hi - lo;
    out[a] = lo;
    out[4 + a] = (ext > 0.f && isfinite(ext)) ? 2097151.0f / ext : 0.f;  // 2^21 - 1 cells per axis
}

// ---- 2. Morton keys, sort, packed copy ---------------------------------------------------------------------------
__device__ __forceinline__ uint64_t spread3(uint32_t v) {  // 21 bits -> every third bit of 63
    uint64_t x = v & 0x1FFFFFu;
    x = (x | (x << 32)) & 0x1F00000000FFFFull;
    x = (x | (x << 16)) & 0x1F0000FF0000FFull;
    x = (x | (x << 8)) & 0x100F00F00F00F00Full;
    x = (x | (x << 4)) & 0x10C30C30C30C30C3ull;
    x = (x | (x << 2)) & 0x1249249249249249ull;
    return x;
}

__device__ __forceinline__ uint32_t quantise(float x, float lo, float scale) {
    const float q = fminf(fmaxf((x - lo) * scale, 0.f), 2097151.0f);  // NaN -> 0 (fmaxf drops it)
    return (uint32_t)q;
}

__global__ void __launch_bounds__(256) morton_kernel(const float* __restrict__ xyz, int64_t n, const float* __restrict__ bnd,
                                                     unsigned long long* __restrict__ keys, int32_t* __restrict__ vals) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const uint32_t qx = quantise(xyz[3 * i], bnd[0], bnd[4]);
    const uint32_t qy = quantise(xyz[3 * i + 1], bnd[1], bnd[5]);
    const uint32_t qz = quantise(xyz[3 * i + 2], bnd[2], bnd[6]);
    keys[i] = (spread3(qx) << 2) | (spread3(qy) << 1) | spread3(qz);
    vals[i] = (int32_t)i;
}

__global__ void __launch_bounds__(256) pack_kernel(const float* __restrict__ xyz, const int32_t* __restrict__ order,
                                                   int64_t n, float4* __restrict__ pts) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const int32_t v = order[i];
    pts[i] = make_float4(xyz[3 * (int64_t)v], xyz[3 * (int64_t)v + 1], xyz[3 * (int64_t)v + 2], __int_as_float(v));
}

// ---- 3. bucket boxes + implicit tree -----------------------------------------------------------------------------
// one warp per leaf (P leaves, the ones past the last bucket hold the empty box): warp min/max of the bucket, then lane 0
// walks up; the second child to arrive at a parent (atomic counter) builds it from both children.
__global__ void __launch_bounds__(256) tree_kernel(const float4* __restrict__ pts, int64_t n, int64_t P,
                                                   float4* __restrict__ lo, float4* __restrict__ hi,
                                                   uint32_t* __restrict__ flags) {
    const int64_t leaf = ((int64_t)blockIdx.x * 256 + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (leaf >= P) return;
    const int64_t i = leaf * BUCKET + lane;
    float4 p = i < n ? pts[i] : make_float4(FLT_MAX, FLT_MAX, FLT_MAX, 0.f);
    float l[3] = {p.x, p.y, p.z}, h[3] = {p.x, p.y, p.z};
    if (i >= n) { h[0] = h[1] = h[2] = -FLT_MAX; }
    if (i < n && !finite3(p.x, p.y, p.z)) {  // a non-finite point would poison the box: it is never a neighbour anyway
        l[0] = l[1] = l[2] = FLT_MAX; h[0] = h[1] = h[2] = -FLT_MAX;
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            l[a] = fminf(l[a], __shfl_xor_sync(0xffffffffu, l[a], o));
            h[a] = fmaxf(h[a], __shfl_xor_sync(0xffffffffu, h[a], o));
        }
    }
    if (lane != 0) return;
    int64_t node = P + leaf;
    float4 bl = make_float4(l[0], l[1], l[2], 0.f), bh = make_float4(h[0], h[1], h[2], 0.f);
    lo[node] = bl; hi[node] = bh;
    while (node > 1) {
        __threadfence();  // this node's box is visible before the sibling's builder can see the counter
        const int64_t parent = node >> 1;
        if (atomicAdd(&flags[parent], 1u) == 0) return;  // first child: the sibling's thread builds the parent
        const int64_t sib = node ^ 1;
        const float4 sl = __ldcg(&lo[sib]), sh = __ldcg(&hi[sib]);
        bl = make_float4(fminf(bl.x, sl.x), fminf(bl.y, sl.y), fminf(bl.z, sl.z), 0.f);
        bh = make_float4(fmaxf(bh.x, sh.x), fmaxf(bh.y, sh.y), fmaxf(bh.z, sh.z), 0.f);
        lo[parent] = bl; hi[parent] = bh;
        node = parent;
    }
}

// ---- 4. queries --------------------------------------------------------------------------------------------------
// sorted top-k of float32 squared distances with the sorted-point index as payload; slots [0, K - k) hold the sentinel
// -1 (never displaced), so the k-th distance is always bd[K - 1] whatever the runtime k <= K.
template <int K>
__device__ __forceinline__ void topk_insert(float (&bd)[K], int32_t (&bi)[K], float d, int32_t id) {
    if (!(d < bd[K - 1])) return;
#pragma unroll
    for (int j = K - 1; j > 0; --j) {
        const bool up = d < bd[j - 1];
        const bool here = d < bd[j];
        bd[j] = up ? bd[j - 1] : (here ? d : bd[j]);
        bi[j] = up ? bi[j - 1] : (here ? id : bi[j]);
    }
    if (d < bd[0]) { bd[0] = d; bi[0] = id; }
}

__device__ __forceinline__ float sqdist(float qx, float qy, float qz, float px, float py, float pz) {
    const float dx = px - qx, dy = py - qy, dz = pz - qz;
    return fmaf(dz, dz, fmaf(dy, dy, dx * dx));
}

__device__ __forceinline__ float box_lb(float qx, float qy, float qz, float4 l, float4 h) {
    const float gx = fmaxf(fmaxf(l.x - qx, qx - h.x), 0.f);
    const float gy = fmaxf(fmaxf(l.y - qy, qy - h.y), 0.f);
    const float gz = fmaxf(fmaxf(l.z - qz, qz - h.z), 0.f);
    return fmaf(gz, gz, fmaf(gy, gy, gx * gx));
}

template <int K>
__global__ void __launch_bounds__(QB, 2) knn_query_kernel(const float4* __restrict__ pts, int64_t n, int32_t k,
                                                       int64_t P, int32_t levels, const float4* __restrict__ lo,
                                                       const float4* __restrict__ hi, double* __restrict__ avg) {
    const int64_t i = (int64_t)blockIdx.x * QB + threadIdx.x;  // sorted position of this lane's query
    const int lane = threadIdx.x & 31;
    const int64_t bucket = i >> 5;                             // warp-uniform
    const int64_t nb = (n + BUCKET - 1) / BUCKET;
    if (bucket >= nb) return;                                  // whole warps only
    const bool active = i < n;
    const float4 q = active ? pts[i] : make_float4(0.f, 0.f, 0.f, __int_as_float(-1));

    float bd[K];
    int32_t bi[K];
#pragma unroll
    for (int j = 0; j < K; ++j) { bd[j] = j < K - k ? -1.0f : INFINITY; bi[j] = -1; }

    // seed from the own bucket (includes the query itself at distance 0)
#pragma unroll 4
    for (int j = 0; j < BUCKET; ++j) {
        const float px = __shfl_sync(0xffffffffu, q.x, j), py = __shfl_sync(0xffffffffu, q.y, j),
                    pz = __shfl_sync(0xffffffffu, q.z, j);
        const int64_t pj = bucket * BUCKET + j;
        if (active && pj < n) topk_insert<K>(bd, bi, sqdist(q.x, q.y, q.z, px, py, pz), (int32_t)pj);
    }

    // pruned depth-first walk, stack entry s held by lane s
    const int32_t own_leaf = (int32_t)(P + bucket);  // P <= 2^26 for n < 2^31
    int32_t slot = 1;
    int sp = 1;
    while (sp > 0) {
        --sp;
        const int32_t node = __shfl_sync(0xffffffffu, slot, sp);
        const float4 l = lo[node], h = hi[node];
        const float lb = box_lb(q.x, q.y, q.z, l, h);
        if (!__any_sync(0xffffffffu, active && lb * PRUNE_SCALE < bd[K - 1])) continue;
        if (node >= P) {
            if (node == own_leaf) continue;
            const int64_t base = (int64_t)(node - P) * BUCKET;  // leaves past the last bucket have the empty box: never opened
            const float4 p = base + lane < n ? pts[base + lane] : make_float4(FLT_MAX, FLT_MAX, FLT_MAX, 0.f);
#pragma unroll 4
            for (int j = 0; j < BUCKET; ++j) {
                const float px = __shfl_sync(0xffffffffu, p.x, j), py = __shfl_sync(0xffffffffu, p.y, j),
                            pz = __shfl_sync(0xffffffffu, p.z, j);
                if (active && base + j < n) topk_insert<K>(bd, bi, sqdist(q.x, q.y, q.z, px, py, pz), (int32_t)(base + j));
            }
        } else {
            // near child first: the one on the side of the own leaf (Morton order ~ space)
            const int depth = 31 - __clz(node);
            const int32_t anc = own_leaf >> (levels - depth - 1);
            const int32_t c0 = 2 * node, c1 = 2 * node + 1;
            const int32_t nearc = anc >= c1 ? c1 : c0, farc = anc >= c1 ? c0 : c1;
            if (lane == sp) slot = farc;
            if (lane == sp + 1) slot = nearc;
            sp += 2;
        }
    }
    if (!active) return;

    const int32_t orig = __float_as_int(q.w);
    if (!finite3(q.x, q.y, q.z)) { avg[orig] = __longlong_as_double(0x7FF8000000000000ll); return; }
    const int32_t keff = (int32_t)(n < (int64_t)k ? n : (int64_t)k);
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < K; ++j) {
        if (bi[j] >= 0) {
            const float4 p = pts[bi[j]];
            const double dx = (double)p.x - (double)q.x, dy = (double)p.y - (double)q.y, dz = (double)p.z - (double)q.z;
            s += sqrt(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
        }
    }
    avg[orig] = s / (double)keff;
}

template <int K>
void launch_query(const float4* pts, int64_t n, int32_t k, int64_t P, int32_t levels, const float4* lo, const float4* hi,
                  double* avg, cudaStream_t st) {
    const int64_t nb = (n + BUCKET - 1) / BUCKET;
    const int64_t threads = nb * BUCKET;
    knn_query_kernel<K><<<(unsigned)((threads + QB - 1) / QB), QB, 0, st>>>(pts, n, k, P, levels, lo, hi, avg);
}

// ---- outlier statistics ------------------------------------------------------------------------------------------
inline int red_ctas(int64_t n) { return (int)(n / 256 + 1 < RED_CTAS ? n / 256 + 1 : RED_CTAS); }

// pass 0: per-CTA {sum of avg over avg > 0, count of non-finite avg};  pass 1: per-CTA sum of (avg - mean)^2 over
// avg > 0.  Grid-stride in a fixed order with a fixed tree: the result depends on n only (bit-identical re-runs).
template <int PASS>
__global__ void __launch_bounds__(256) moment_kernel(const double* __restrict__ avg, int64_t n,
                                                     const double* __restrict__ stats, double* __restrict__ partial) {
    __shared__ double s_a[8], s_b[8];
    const double mean = PASS == 1 ? stats[0] : 0.0;
    double a = 0.0, b = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
        const double v = avg[i];
        if (PASS == 0) {
            if (v > 0.0) a += v;
            if (!isfinite(v)) b += 1.0;
        } else if (v > 0.0) {
            const double d = v - mean;
            a += d * d;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if ((threadIdx.x & 31) == 0) { s_a[threadIdx.x >> 5] = a; s_b[threadIdx.x >> 5] = b; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ta = 0.0, tb = 0.0;
        for (int w = 0; w < 8; ++w) { ta += s_a[w]; tb += s_b[w]; }
        partial[2 * blockIdx.x] = ta;
        partial[2 * blockIdx.x + 1] = tb;
    }
}

// one CTA: fixed-order sum of the partials.  pass 0 -> stats[0] = mean (over ALL n points), stats[3] = non-finite count;
// pass 1 -> stats[1] = std (Bessel), stats[2] = threshold.
template <int PASS>
__global__ void __launch_bounds__(256) moment_final_kernel(const double* __restrict__ partial, int nparts, int64_t n,
                                                           double std_ratio, double* __restrict__ stats) {
    __shared__ double s_a[256], s_b[256];
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < nparts; i += 256) { a += partial[2 * i]; b += partial[2 * i + 1]; }
    s_a[threadIdx.x] = a; s_b[threadIdx.x] = b;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) { s_a[threadIdx.x] += s_a[threadIdx.x + o]; s_b[threadIdx.x] += s_b[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x != 0) return;
    if (PASS == 0) {
        stats[0] = s_a[0] / (double)n;
        stats[3] = s_b[0];
    } else {
        const double sd = sqrt(s_a[0] / (double)(n - 1));  // n == 1: 0/0 = NaN, nothing is kept
        stats[1] = sd;
        stats[2] = stats[0] + std_ratio * sd;
    }
}

__global__ void __launch_bounds__(256) outlier_mask_kernel(const double* __restrict__ avg, int64_t n,
                                                           const double* __restrict__ stats, uint8_t* __restrict__ keep) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const double v = avg[i];
    keep[i] = (v > 0.0 && v < stats[2]) ? 1 : 0;
}

}  // namespace

extern "C" int64_t g2pc_knn_workspace_bytes(int64_t n, int32_t k) {
    if (n < 0 || k < 1 || k > 32) return 0;
    return (int64_t)knn_layout(n).total;
}

/* avg[i] (float64) = mean distance of point i to its k nearest points of the cloud (itself included; all n if n < k). */
extern "C" int g2pc_knn_mean_distance(const float* xyz, int64_t n, int32_t k, double* avg, void* workspace,
                                      int64_t workspace_bytes, void* stream) {
    G2PC_CHECK_ARG(n >= 0, "n < 0");
    G2PC_CHECK_ARG(k >= 1 && k <= 32, "k must be in [1, 32]");
    G2PC_CHECK_ARG(n < 0x7FFFFFFFll, "n must fit int32 indices");
    if (n == 0) return G2PC_OK;
    G2PC_CHECK_ARG(xyz && avg && workspace, "null pointer");
    G2PC_CHECK_ARG(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
    const KnnLayout L = knn_layout(n);
    G2PC_CHECK_ARG(workspace_bytes >= (int64_t)L.total, "workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    unsigned long long* keys_in = (unsigned long long*)(ws + L.keys);
    unsigned long long* keys_out = keys_in + n;
    int32_t* vals_in = (int32_t*)(ws + L.vals_in);
    int32_t* vals_out = (int32_t*)(ws + L.vals_out);
    float4* pts = (float4*)(ws + L.keys);  // the keys are dead once the order is known
    float4* lo = (float4*)(ws + L.lo);
    float4* hi = (float4*)(ws + L.hi);
    uint32_t* flags = (uint32_t*)(ws + L.flags);
    float* bparts = (float*)(ws + L.bounds);
    float* bnd = bparts + NB_BOUNDS * 8;
    int32_t levels = 0;
    while (((int64_t)1 << levels) < L.P) ++levels;

    const unsigned g = (unsigned)((n + 255) / 256);
    bounds_kernel<<<NB_BOUNDS, 256, 0, st>>>(xyz, n, bparts);
    G2PC_CHECK_LAUNCH();
    bounds_final_kernel<<<1, 32, 0, st>>>(bparts, NB_BOUNDS, bnd);
    G2PC_CHECK_LAUNCH();
    morton_kernel<<<g, 256, 0, st>>>(xyz, n, bnd, keys_in, vals_in);
    G2PC_CHECK_LAUNCH();
    size_t tb = L.tmp_bytes;
    G2PC_CUDA(cub::DeviceRadixSort::SortPairs(ws + L.tmp, tb, keys_in, keys_out, vals_in, vals_out, n, 0, 63, st));
    pack_kernel<<<g, 256, 0, st>>>(xyz, vals_out, n, pts);
    G2PC_CHECK_LAUNCH();
    G2PC_CUDA(cudaMemsetAsync(flags, 0, (size_t)L.P * 4, st));
    tree_kernel<<<(unsigned)((L.P * 32 + 255) / 256), 256, 0, st>>>(pts, n, L.P, lo, hi, flags);
    G2PC_CHECK_LAUNCH();
    if (k <= 8) launch_query<8>(pts, n, k, L.P, levels, lo, hi, avg, st);
    else if (k <= 16) launch_query<16>(pts, n, k, L.P, levels, lo, hi, avg, st);
    else if (k == 20) launch_query<20>(pts, n, k, L.P, levels, lo, hi, avg, st);
    else launch_query<32>(pts, n, k, L.P, levels, lo, hi, avg, st);
    G2PC_CHECK_LAUNCH();
    return G2PC_OK;
}

extern "C" int64_t g2pc_outlier_workspace_bytes(int64_t n) {
    if (n < 0) return 0;
    return (int64_t)(2 * RED_CTAS * sizeof(double));
}

/* keep[i] = 0 < avg[i] < mean + std_ratio * std; stats4 = {mean, std, threshold, non-finite count of avg}. */
extern "C" int g2pc_outlier_mask(const double* avg, int64_t n, double std_ratio, uint8_t* keep, double* stats4,
                                 void* workspace, int64_t workspace_bytes, void* stream) {
    G2PC_CHECK_ARG(n >= 0, "n < 0");
    G2PC_CHECK_ARG(std_ratio > 0.0, "std_ratio must be > 0");
    G2PC_CHECK_ARG(n < 0x7FFFFFFFll, "n must fit int32 indices");
    G2PC_CHECK_ARG(stats4, "null stats");
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) { G2PC_CUDA(cudaMemsetAsync(stats4, 0, 4 * sizeof(double), st)); return G2PC_OK; }
    G2PC_CHECK_ARG(avg && keep && workspace, "null pointer");
    G2PC_CHECK_ARG(((uintptr_t)workspace & 7) == 0, "workspace must be 8-byte aligned");
    G2PC_CHECK_ARG(workspace_bytes >= g2pc_outlier_workspace_bytes(n), "workspace too small");
    double* partial = (double*)workspace;
    const int nc = red_ctas(n);
    moment_kernel<0><<<nc, 256, 0, st>>>(avg, n, stats4, partial);
    G2PC_CHECK_LAUNCH();
    moment_final_kernel<0><<<1, 256, 0, st>>>(partial, nc, n, std_ratio, stats4);
    G2PC_CHECK_LAUNCH();
    moment_kernel<1><<<nc, 256, 0, st>>>(avg, n, stats4, partial);
    G2PC_CHECK_LAUNCH();
    moment_final_kernel<1><<<1, 256, 0, st>>>(partial, nc, n, std_ratio, stats4);
    G2PC_CHECK_LAUNCH();
    outlier_mask_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(avg, n, stats4, keep);
    G2PC_CHECK_LAUNCH();
    return G2PC_OK;
}
