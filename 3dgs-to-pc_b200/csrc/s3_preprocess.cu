// s3_preprocess.cu — S3: per-camera, per-Gaussian projection + quadtree membership counting; S4b: instance emission.
//
// Reference semantics restated (not copied), renderer_type=python:
//   gauss_render.py:101-148  build_covariance_2d   (EWA: cov2d = J W Sigma W^T J^T [:2,:2] + 0.3 I)
//   gauss_render.py:151-168  projection_ndc        (p_h = [p,1] V P, p_w = 1/(w + 1e-6), in front <=> z_view <= -1e-6)
//   gauss_render.py:171-193  get_radius / get_rect (radius = 3*ceil(sqrt(lambda_max)), rect clipped to the image)
//   gauss_render.py:349      conic = inverse(cov2d)
//   gauss_render.py:43-99    eval_sh (+0.5, clamp >= 0 as forward.cu:65-72) when SH coefficients are supplied
//   gauss_render.py:301-319  tile membership: min(rect_max, tile_max) > max(rect_min, tile_min), strict, fp32
// One thread per Gaussian, 1024 Gaussians per CTA.  Inputs come from the packed geometry array built once per renderer
// (g2pc_pack_geometry: 3 x float4 per Gaussian = xyz, Sigma as 6 floats, log2(opacity); three 16-byte loads per thread,
// a warp reads 1536 contiguous bytes) and the SH rows (16-byte loads).  Membership is evaluated by range queries on the
// per-level interval tables (g2pc/quadtree.py) instead of testing every tile against every Gaussian, and only on the
// tables (g2pc/quadtree.py).  Exact overlap counts are taken on the CANDIDATE levels only (levels that have nodes small
// enough to be leaves); above them every node splits by its size and only a non-empty flag is raised (plain stores, found
// by walking up from the base range).  Counts and flags live in a shared-memory array flushed once per CTA.  The node range at the first candidate level is packed into the high word of
// `val` (low word = Gaussian id): after the depth sort the multisplit kernels (s4_tree.cu) read their ranges from the
// sorted stream and never gather.
#include "colour_common.cuh"

namespace {

struct PreParams {
    const float4* geom;    // 3 x float4 per Gaussian: {x,y,z,S00} {S01,S02,S11,S12} {S22,log2(opacity),0,0}
    const float* colours;  // (n,3) f32 or null
    const float* shs;      // (n,3,sh_stride) f32 or null
    int32_t sh_stride, sh_degree;
    int64_t n;
    g2pc_camera_t cam;
    QtMeta meta;
    QtTables tab;
    const uint16_t* luts;  // per level [x lo (W)][x hi+1 (W)][y lo (H)][y hi+1 (H)] (g2pc/quadtree.py pixel_luts)
    int32_t n1;  // entries per 1-D table array
    float4* proj;
    uint32_t* node_cnt;
    uint32_t* depth_key;  // bits(-z_view) for Gaussians in front of the camera, 0xFFFFFFFF otherwise
    unsigned long long* val;  // (packed node range at the base level << 32) | Gaussian id
    int32_t nodes_2d;     // histogram entries (0: no shared-memory histogram, global atomics)
    uint32_t level_mask;  // bit l: level l has leaf-candidate nodes
    uint32_t clean_mask;  // bit l: level l has no dropped / degenerate node (membership = the looked-up range)
    int32_t base_level;   // lowest set bit of level_mask
};

__device__ __forceinline__ float3 sh_to_rgb(const float* __restrict__ sh, int stride, int deg, float3 d) {
    // sh: 3 channels x stride coefficients (channel-major).  16-byte loads when the row is 16-byte aligned.
    float out[3];
    const int ncoef = (deg + 1) * (deg + 1);
    const bool vec = ((stride & 3) == 0) && ((((uintptr_t)sh) & 15) == 0);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        float s[16];
        if (vec) {
            const float4* s4 = reinterpret_cast<const float4*>(sh + c * stride);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (4 * q < ncoef) {
                    const float4 v = __ldg(s4 + q);
                    s[4 * q] = v.x; s[4 * q + 1] = v.y; s[4 * q + 2] = v.z; s[4 * q + 3] = v.w;
                }
            }
        } else {
#pragma unroll
            for (int k = 0; k < 16; ++k) if (k < ncoef) s[k] = sh[c * stride + k];
        }
        out[c] = sh_channel(deg, d, [&](int k) { return s[k]; });
    }
    return make_float3(out[0], out[1], out[2]);
}

// Persistent CTAs (grid = SMs x resident CTAs): the tables / pixel LUTs are staged and the histogram is flushed once per
// CTA, not once per 1024 Gaussians (at 1920x1080 with two extra levels that was 96 KB of LUT + 21845 flush atomics per
// 1024 Gaussians and one 256-thread CTA per SM: 15 ms per camera for 6 M Gaussians).  256, 512 or 1024 threads per CTA,
// whichever fills the SM for the shared-memory footprint.
__global__ void __launch_bounds__(1024, 1) preprocess_kernel(const PreParams p) {
    extern __shared__ int32_t smem_tab[];
    uint32_t* s_hist = reinterpret_cast<uint32_t*>(smem_tab + 6 * p.n1);
    for (int k = threadIdx.x; k < p.nodes_2d; k += blockDim.x) s_hist[k] = 0u;
    // pixel -> node-range lookups of every level (replace the per-Gaussian interval walks: ~80 % of this kernel's
    // instructions in the r02a capture)
    uint16_t* s_lut = reinterpret_cast<uint16_t*>(s_hist + p.nodes_2d);
    const int lut_level = 2 * (p.cam.width + p.cam.height);
    {
        const int words = (lut_level * p.meta.num_levels + 1) / 2;
        const uint32_t* src = reinterpret_cast<const uint32_t*>(p.luts);
        uint32_t* dst = reinterpret_cast<uint32_t*>(s_lut);
        for (int k = threadIdx.x; k < words; k += blockDim.x) dst[k] = src[k];
    }
    const QtTables T = load_tables(p.tab, p.n1, smem_tab);  // ends with __syncthreads()
    const bool use_hist = p.nodes_2d > 0;
  for (int64_t cta_base = (int64_t)blockIdx.x * blockDim.x; cta_base < p.n; cta_base += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = cta_base + threadIdx.x;
    const int64_t il = i < p.n ? i : p.n - 1;  // lanes past the end shadow the last Gaussian and write nothing

    const float* V = p.cam.view;
    const float* P = p.cam.proj;
    const float4 g0 = __ldg(p.geom + 3 * il), g1 = __ldg(p.geom + 3 * il + 1), g2 = __ldg(p.geom + 3 * il + 2);
    const float m0 = g0.x, m1 = g0.y, m2 = g0.z;

    // p_view = [mu, 1] @ V   (row-vector convention)
    float pv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) pv[j] = fmaf(m2, V[8 + j], fmaf(m1, V[4 + j], fmaf(m0, V[j], V[12 + j])));
    const bool in_front = (pv[2] <= -0.000001f) && (i < p.n);
    bool has_rect = false;
    float x0 = 0.f, x1 = 0.f, y0 = 0.f, y1 = 0.f;

    float4 q0 = make_float4(0.f, 0.f, 0.f, 0.f), q1 = q0, q2 = q0;
    uint32_t range = G2PC_RANGE_EMPTY;
    if (in_front) {
        // p_h = p_view @ P ; ndc = p_h / (w + 1e-6) ; pixel centre convention of gauss_render.py:435-436
        float ph[4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
            ph[j] = fmaf(pv[3], P[12 + j], fmaf(pv[2], P[8 + j], fmaf(pv[1], P[4 + j], pv[0] * P[j])));
        const float pw = 1.0f / (ph[3] + 0.000001f);
        const float mx = ((ph[0] * pw + 1.0f) * (float)p.cam.width - 1.0f) * 0.5f;
        const float my = ((ph[1] * pw + 1.0f) * (float)p.cam.height - 1.0f) * 0.5f;

        // t = mu @ V[:3,:3] + V[3,:3]
        const float t0 = fmaf(m2, V[8], fmaf(m1, V[4], m0 * V[0])) + V[12];
        const float t1 = fmaf(m2, V[9], fmaf(m1, V[5], m0 * V[1])) + V[13];
        const float tz = fmaf(m2, V[10], fmaf(m1, V[6], m0 * V[2])) + V[14];
        const float limx = p.cam.tan_fovx * 1.3f, limy = p.cam.tan_fovy * 1.3f;
        const float tx = fminf(fmaxf(t0 / tz, -limx), limx) * tz;
        const float ty = fminf(fmaxf(t1 / tz, -limy), limy) * tz;
        const float itz = 1.0f / tz;
        const float ja = itz * p.cam.focal_x, jb = -tx / (tz * tz) * p.cam.focal_x;
        const float jc = itz * p.cam.focal_y, jd = -ty / (tz * tz) * p.cam.focal_y;
        // W = V[:3,:3]^T  =>  W[r][c] = V[c][r] = V[4*c + r]
        float M[2][3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            M[0][c] = fmaf(jb, V[4 * c + 2], ja * V[4 * c + 0]);
            M[1][c] = fmaf(jd, V[4 * c + 2], jc * V[4 * c + 1]);
        }
        // Sigma is symmetric by construction (S1 kernel); the packed copy keeps the upper triangle
        const float S[9] = {g0.w, g1.x, g1.y, g1.x, g1.z, g1.w, g1.y, g1.w, g2.x};
        float A[2][3], B[2][3];
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c)
                A[r][c] = fmaf(M[r][2], S[6 + c], fmaf(M[r][1], S[3 + c], M[r][0] * S[c]));
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c)  // (A @ W^T)[r][c] = sum_k A[r][k] * W[c][k] = sum_k A[r][k] * V[4*k + c]
                B[r][c] = fmaf(A[r][2], V[8 + c], fmaf(A[r][1], V[4 + c], A[r][0] * V[c]));
        const float c00 = fmaf(B[0][2], jb, B[0][0] * ja) + 0.3f;
        const float c01 = fmaf(B[0][2], jd, B[0][1] * jc);
        const float c10 = fmaf(B[1][2], jb, B[1][0] * ja);
        const float c11 = fmaf(B[1][2], jd, B[1][1] * jc) + 0.3f;

        const float det = c00 * c11 - c01 * c10;
        const float mid = 0.5f * (c00 + c11);
        const float root = sqrtf(fmaxf(mid * mid - det, 0.1f));
        const float radius = 3.0f * ceilf(sqrtf(fmaxf(mid + root, mid - root)));

        const float idet = 1.0f / det;
        const float K = -0.72134752044448170368f;  // -0.5 * log2(e): the blend evaluates exp2 directly
        const float k00 = c11 * idet, k01 = -c01 * idet, k10 = -c10 * idet, k11 = c00 * idet;

        float3 rgb;
        if (p.shs) {
            const float dx = m0 - p.cam.campos[0], dy = m1 - p.cam.campos[1], dz = m2 - p.cam.campos[2];
            const float inv = 1.0f / sqrtf(dx * dx + dy * dy + dz * dz);
            rgb = sh_to_rgb(p.shs + (int64_t)il * 3 * p.sh_stride, p.sh_stride, p.sh_degree,
                            make_float3(dx * inv, dy * inv, dz * inv));
        } else {
            rgb = make_float3(p.colours[3 * il], p.colours[3 * il + 1], p.colours[3 * il + 2]);
        }
        q0 = make_float4(mx, my, k00 * K, (k01 + k10) * K);
        // alpha = min(0.99, opacity * exp(power)) = min(0.99, exp2(power' + log2(opacity)))
        q1 = make_float4(k11 * K, g2.y, rgb.x, rgb.y);
        q2 = make_float4(rgb.z, pv[2], radius, 1.0f);

        gaussian_rect(mx, my, radius, p.cam.width, p.cam.height, x0, x1, y0, y1);
        has_rect = true;
    }
    // ---- quadtree membership (all 32 lanes: the base-level walk is warp-cooperative) ----------------------------------
    // the rect lies in [0, W-1] x [0, H-1]: lo = first node with end > floor(min), hi = last node with start < ceil(max)
    const int qx0 = (int)x0, qy0 = (int)y0, cx1 = (int)ceilf(x1), cy1 = (int)ceilf(y1);
    int bxlo = 1, bxhi = 0, bylo = 1, byhi = 0;
    {
        const int l = p.base_level;
        const int o1 = (1 << l) - 1;
        if (has_rect && x1 > x0 && y1 > y0) {
            const uint16_t* L = s_lut + l * lut_level;
            bxlo = L[qx0]; bxhi = (int)L[p.cam.width + cx1] - 1;
            bylo = L[2 * p.cam.width + qy0]; byhi = (int)L[2 * p.cam.width + p.cam.height + cy1] - 1;
            if (bxlo > bxhi || bylo > byhi) { bxlo = 1; bxhi = 0; bylo = 1; byhi = 0; }
            else range = g2pc_pack_range(bxlo, bxhi, bylo, byhi);
        }
        uint32_t* cnt = p.node_cnt + off2(l);
        uint32_t* hcnt = s_hist + off2(l);
        if ((p.clean_mask >> l) & 1u) {
            warp_for_each_node(range, 0u, [&](int ix, int iy, int, uint32_t) {
                if (use_hist) atomicAdd(hcnt + (iy << l) + ix, 1u);
                else atomicAdd(cnt + (iy << l) + ix, 1u);
            });
        } else {
            warp_for_each_node(range, 0u, [&](int ix, int iy, int, uint32_t) {
                if (!axis_member(T.ys + o1, T.ye + o1, T.yf + o1, iy) || !axis_member(T.xs + o1, T.xe + o1, T.xf + o1, ix)) return;
                if (use_hist) atomicAdd(hcnt + (iy << l) + ix, 1u);
                else atomicAdd(cnt + (iy << l) + ix, 1u);
            });
        }
    }
    const bool in_tree = has_rect && bxlo <= bxhi;
    // deeper candidate levels exist only after a count-driven split asked for them (1920 px / 6 M Gaussians: two of them,
    // ~40 nodes per Gaussian): the same warp-cooperative walk as the base level when the level is clean
    for (int l = p.base_level + 1; l < p.meta.num_levels; ++l) {  // (uniform)
        if (!((p.level_mask >> l) & 1u)) continue;
        const int o1 = (1 << l) - 1;
        int xlo = 1, xhi = 0, ylo = 1, yhi = 0;
        if (in_tree) {
            const uint16_t* L = s_lut + l * lut_level;
            xlo = L[qx0]; xhi = (int)L[p.cam.width + cx1] - 1;
            ylo = L[2 * p.cam.width + qy0]; yhi = (int)L[2 * p.cam.width + p.cam.height + cy1] - 1;
        }
        const bool some = xlo <= xhi && ylo <= yhi;
        uint32_t* cnt = p.node_cnt + off2(l);
        uint32_t* hcnt = s_hist + off2(l);  // (kept apart: shared-memory atomics, not generic ones)
        if (((p.clean_mask >> l) & 1u) && l <= G2PC_RANGE_MAX_LEVEL) {
            const uint32_t rl = some ? g2pc_pack_range(xlo, xhi, ylo, yhi) : (uint32_t)G2PC_RANGE_EMPTY;
            warp_for_each_node(rl, 0u, [&](int ix, int iy, int, uint32_t) {
                if (use_hist) atomicAdd(hcnt + (iy << l) + ix, 1u);
                else atomicAdd(cnt + (iy << l) + ix, 1u);
            });
            continue;
        }
        if (!some) continue;
        for (int iy = ylo; iy <= yhi; ++iy) {
            if (!axis_member(T.ys + o1, T.ye + o1, T.yf + o1, iy)) continue;
            for (int ix = xlo; ix <= xhi; ++ix) {
                if (!axis_member(T.xs + o1, T.xe + o1, T.xf + o1, ix)) continue;
                if (use_hist) atomicAdd(hcnt + (iy << l) + ix, 1u);
                else atomicAdd(cnt + (iy << l) + ix, 1u);
            }
        }
    }
    if (in_tree) {
        // levels above: every node splits by its size, only "is anything in it" matters (an empty tile is background
        // and has no children, gauss_render.py:313-315).  A child tile may overhang its parent by a pixel, so this is
        // NOT implied by the leaf-level counts: look the exact range of every level up and raise plain flags.
        for (int l = p.base_level - 1; l >= 0; --l) {
            const int o1 = (1 << l) - 1;
            const uint16_t* L = s_lut + l * lut_level;
            const int xlo = L[qx0], xhi = (int)L[p.cam.width + cx1] - 1;
            const int ylo = L[2 * p.cam.width + qy0], yhi = (int)L[2 * p.cam.width + p.cam.height + cy1] - 1;
            if (xlo > xhi || ylo > yhi) continue;
            if (use_hist && ((p.clean_mask >> l) & 1u)) {
                // the common case, kept branch-light: shared-memory flags, no per-node table checks, and almost always a
                // single node (one predicated store)
                uint32_t* f = s_hist + off2(l);
                if (xlo == xhi && ylo == yhi) {
                    f[(ylo << l) + xlo] = 1u;
                } else {
                    for (int iy = ylo; iy <= yhi; ++iy)
                        for (int ix = xlo; ix <= xhi; ++ix) f[(iy << l) + ix] = 1u;
                }
                continue;
            }
            uint32_t* flags = (use_hist ? s_hist : p.node_cnt) + off2(l);
            if ((p.clean_mask >> l) & 1u) {
                for (int iy = ylo; iy <= yhi; ++iy)
                    for (int ix = xlo; ix <= xhi; ++ix) flags[(iy << l) + ix] = 1u;
                continue;
            }
            for (int iy = ylo; iy <= yhi; ++iy) {
                if (!axis_member(T.ys + o1, T.ye + o1, T.yf + o1, iy)) continue;
                for (int ix = xlo; ix <= xhi; ++ix) {
                    if (!axis_member(T.xs + o1, T.xe + o1, T.xf + o1, ix)) continue;
                    flags[(iy << l) + ix] = 1u;
                }
            }
        }
    }
    if (i < p.n) {
    float4* rec = p.proj + 3 * i;
    rec[0] = q0; rec[1] = q1; rec[2] = q2;
    p.depth_key[i] = in_front ? __float_as_uint(-pv[2]) : 0xFFFFFFFFu;
    p.val[i] = ((unsigned long long)range << 32) | (unsigned long long)(uint32_t)i;
    }
  }
    if (use_hist) {
        __syncthreads();
        for (int k = threadIdx.x; k < p.nodes_2d; k += blockDim.x) {
            const uint32_t v = s_hist[k];
            if (v) atomicAdd(p.node_cnt + k, v);
        }
    }
}

// Packed geometry (once per renderer): xyz (n,3), Sigma (n,3,3) and opacity (n) -> 3 float4 per Gaussian, log2 of the
// opacity taken here (the blend evaluates alpha = min(0.99, exp2(power' + log2 o))).
__global__ void __launch_bounds__(256) pack_geometry_kernel(const float* __restrict__ xyz, const float* __restrict__ cov,
                                                            const float* __restrict__ opacity, int64_t n,
                                                            float4* __restrict__ geom) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* c = cov + 9 * i;
    geom[3 * i] = make_float4(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], c[0]);
    geom[3 * i + 1] = make_float4(c[1], c[2], c[4], c[5]);
    geom[3 * i + 2] = make_float4(c[8], log2f(opacity[i]), 0.0f, 0.0f);
}

}  // namespace

extern "C" int g2pc_pack_geometry(const float* xyz, const float* cov, const float* opacity, int64_t n, void* geom,
                                  void* stream) {
    G2PC_CHECK_ARG(n >= 0, "n < 0");
    if (n == 0) return G2PC_OK;
    G2PC_CHECK_ARG(xyz && cov && opacity && geom, "null pointer");
    G2PC_CHECK_ARG(((uintptr_t)geom & 15) == 0, "geom must be 16-byte aligned");
    pack_geometry_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(xyz, cov, opacity, n,
                                                                                         (float4*)geom);
    G2PC_CHECK_LAUNCH();
    return G2PC_OK;
}

extern "C" int g2pc_preprocess(const void* geom, const float* colours, const float* shs, int32_t sh_stride,
                               int32_t sh_degree, int64_t n, const g2pc_camera_t* cam_host, const int32_t* tables,
                               const uint16_t* luts, int32_t num_levels, uint32_t level_mask, uint32_t clean_mask,
                               void* proj,
                               uint32_t* node_cnt, uint32_t* depth_key, uint64_t* val, void* stream) {
    G2PC_CHECK_ARG(n >= 0, "n < 0");
    if (n == 0) return G2PC_OK;
    G2PC_CHECK_ARG(geom && cam_host && tables && luts && proj && node_cnt && depth_key && val, "null pointer");
    G2PC_CHECK_ARG(((uintptr_t)luts & 3) == 0, "luts must be 4-byte aligned");
    G2PC_CHECK_ARG(n <= 0xFFFFFFFFll, "more than 2^32 Gaussians");
    G2PC_CHECK_ARG((colours != nullptr) != (shs != nullptr), "provide exactly one of colours / shs");
    G2PC_CHECK_ARG(num_levels >= 1 && num_levels <= G2PC_MAX_LEVELS, "bad num_levels");
    G2PC_CHECK_ARG(!shs || (sh_degree >= 0 && sh_degree <= 3 && sh_stride >= (sh_degree + 1) * (sh_degree + 1)),
                   "SH degree must be 0..3 and sh_stride >= (deg+1)^2");
    G2PC_CHECK_ARG(level_mask != 0u && (level_mask >> num_levels) == 0u, "level_mask must name tabulated levels");
    PreParams p;
    p.geom = (const float4*)geom; p.colours = colours; p.shs = shs;
    p.sh_stride = sh_stride; p.sh_degree = sh_degree; p.n = n; p.cam = *cam_host;
    p.meta.num_levels = num_levels; p.meta.max_gaussians_per_tile = 0;
    p.n1 = (1 << num_levels) - 1;
    p.tab = make_tables(tables, p.n1);
    p.luts = luts;
    p.proj = (float4*)proj; p.node_cnt = node_cnt; p.depth_key = depth_key; p.val = (unsigned long long*)val;
    p.level_mask = level_mask;
    p.clean_mask = clean_mask;
    p.base_level = __builtin_ctz(level_mask);
    G2PC_CHECK_ARG(p.base_level <= G2PC_RANGE_MAX_LEVEL, "first leaf-candidate level too deep for the packed node range");
    const int nodes_all = ((1 << (2 * num_levels)) - 1) / 3;
    p.nodes_2d = nodes_all <= 24 * 1024 ? nodes_all : 0;  // histogram in shared memory when it fits (<= 96 KB)
    const size_t lut_bytes = ((size_t)2 * (cam_host->width + cam_host->height) * num_levels * sizeof(uint16_t) + 3) & ~(size_t)3;
    const size_t smem = (size_t)6 * p.n1 * sizeof(int32_t) + (size_t)p.nodes_2d * sizeof(uint32_t) + lut_bytes;
    G2PC_CHECK_ARG(smem <= 220 * 1024, "quadtree tables do not fit the shared memory of one SM");
    if (smem > 48 * 1024)
        G2PC_CUDA(cudaFuncSetAttribute(preprocess_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int threads = smem <= 56 * 1024 ? 256 : smem <= 113 * 1024 ? 512 : 1024;
    const int64_t resident = resident_ctas(preprocess_kernel, threads, smem, 1);
    const int64_t granules = (n + threads - 1) / threads;
    const unsigned grid = (unsigned)(granules < resident ? granules : resident);
    preprocess_kernel<<<grid, threads, smem, (cudaStream_t)stream>>>(p);
    G2PC_CHECK_LAUNCH();
    return G2PC_OK;
}
