// TSPSRNet helper operators: GroupNorm(+swish), AdaIN+concat over per-character windows, and the
// last-writer-wins window write-back.  HBM-bound; see include/marconet_b200.h for call sites.
#include "mn_common.cuh"

namespace {

// ---------------------------------------------------------------- GroupNorm statistics
// Each thread owns 4 consecutive channels (float4 loads, fully coalesced rows); a block walks a pixel chunk with
// blockDim/(C/4) pixels per iteration.  fp32 partials are flushed to fp64 every 32 pixels, reduced over the 8 lanes of a
// 32-channel group by shuffles, over the block in shared memory, then one fp64 atomicAdd per (block, group, moment).
__global__ void __launch_bounds__(256) gn_stats_kernel(const float* __restrict__ x, int x_cs, int H, int W, int C, int cpg,
                                                       const int32_t* __restrict__ valid_w, double* __restrict__ stats, int pix_per_block) {
    mn_pdl_prologue();
    const int n = blockIdx.y;
    const int tpp = C >> 2;                        // threads per pixel
    const int ppi = blockDim.x / tpp;              // pixels per iteration (host guarantees >= 1)
    const int my_c = (threadIdx.x % tpp) * 4;
    const int my_p = threadIdx.x / tpp;
    const int wv = valid_w ? valid_w[n] : W;
    const int HW = H * W;
    const int p_begin = blockIdx.x * pix_per_block;
    const int p_end = min(HW, p_begin + pix_per_block);
    const float* xn = x + (size_t)n * HW * x_cs + my_c;
    float s = 0.f, ss = 0.f;
    double ds = 0.0, dss = 0.0;
    int cnt = 0;
    if (my_p < ppi) {
        // 4 pixels per trip: the four 128-bit loads are issued before any of them is consumed
        for (int p = p_begin + my_p; p < p_end; p += 4 * ppi) {
            float4 v[4];
            bool on[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int pk = p + k * ppi;
                on[k] = pk < p_end && !(valid_w && (pk % W) >= wv);
                v[k] = on[k] ? *reinterpret_cast<const float4*>(xn + (size_t)pk * x_cs) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (!on[k]) continue;
                s += (v[k].x + v[k].y) + (v[k].z + v[k].w);
                ss = fmaf(v[k].x, v[k].x, ss); ss = fmaf(v[k].y, v[k].y, ss); ss = fmaf(v[k].z, v[k].z, ss); ss = fmaf(v[k].w, v[k].w, ss);
                if (++cnt == 32) { ds += (double)s; dss += (double)ss; s = 0.f; ss = 0.f; cnt = 0; }
            }
        }
    }
    ds += (double)s; dss += (double)ss;
    const int lpg = cpg >> 2;                      // lanes per group (8 for 32-channel groups)
    for (int o = lpg >> 1; o > 0; o >>= 1) {
        ds += __shfl_xor_sync(0xffffffffu, ds, o);
        dss += __shfl_xor_sync(0xffffffffu, dss, o);
    }
    __shared__ double red[2][64];                  // [moment][group-slot]: blockDim/lpg <= 32 slots used
    const int slot = threadIdx.x / lpg;            // (pixel slot, group) pair index
    if ((threadIdx.x % lpg) == 0) { red[0][slot] = ds; red[1][slot] = dss; }
    __syncthreads();
    const int G = C / cpg;
    if (threadIdx.x < G) {
        double a = 0.0, b2 = 0.0;
        for (int k = 0; k < ppi; ++k) { a += red[0][k * G + threadIdx.x]; b2 += red[1][k * G + threadIdx.x]; }
        atomicAdd(&stats[((size_t)n * G + threadIdx.x) * 2 + 0], a);
        atomicAdd(&stats[((size_t)n * G + threadIdx.x) * 2 + 1], b2);
    }
}

// (sum, sumsq) fp64 -> (mean, rstd) fp32 per (sample, group); biased variance like torch.nn.GroupNorm.
__global__ void gn_finalize_kernel(const double* __restrict__ stats, float2* __restrict__ mr, int N, int G, int H, int W, int cpg, float eps,
                                   const int32_t* __restrict__ valid_w) {
    mn_pdl_prologue();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * G) return;
    const int n = i / G;
    const int wv = valid_w ? valid_w[n] : W;
    const double cnt = (double)H * wv * cpg;
    const double mean = cnt > 0 ? stats[2 * i] / cnt : 0.0;
    double var = cnt > 0 ? stats[2 * i + 1] / cnt - mean * mean : 0.0;
    if (var < 0.0) var = 0.0;
    mr[i] = make_float2((float)mean, (float)(1.0 / sqrt(var + (double)eps)));
}

// One thread normalises 4 channels of GN_PPT pixels (pixel stride = a quarter of the tensor, so every warp access stays a
// contiguous run of channels); all loads are issued before the first use.  Measured 3.4-3.9 TB/s in round 1 (issue-bound, see below); a capped grid-stride
// variant (8 CTAs/SM) was slower (2.7-3.0 TB/s: 56 registers leave only 4 resident CTAs), one item per thread 3.1-3.4.
constexpr int GN_PPT = 4;
__global__ void __launch_bounds__(256) gn_apply_kernel(const float* __restrict__ x, int x_cs, float* __restrict__ y, int y_cs,
                                const float* __restrict__ gamma, const float* __restrict__ beta,
                                int N, int H, int W, int C, int cpg, float eps, int swish,
                                const int32_t* __restrict__ valid_w, const float2* __restrict__ mr, uint32_t pix_stride) {
    mn_pdl_prologue();
    const int c4 = C >> 2;
    const uint32_t npix = (uint32_t)N * H * W;
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;     // host guarantees N*H*W*C/4 < 2^31: 32-bit div/mod only
    if (idx >= pix_stride * (uint32_t)c4) return;
    const int c = (int)(idx % c4) * 4;
    const uint32_t pix0 = idx / c4;
    const int G = C / cpg, g = c / cpg;
    const float4 ga = *reinterpret_cast<const float4*>(gamma + c), be = *reinterpret_cast<const float4*>(beta + c);
    const float gam[4] = {ga.x, ga.y, ga.z, ga.w}, bet[4] = {be.x, be.y, be.z, be.w};
    float4 v[GN_PPT];
    float2 m2[GN_PPT];
    bool live[GN_PPT], on[GN_PPT];
#pragma unroll
    for (int k = 0; k < GN_PPT; ++k) {
        const uint32_t pix = pix0 + (uint32_t)k * pix_stride;
        live[k] = pix < npix;
        on[k] = false;
        v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        m2[k] = make_float2(0.f, 0.f);
        if (live[k]) {
            const int px = (int)(pix % W);
            const int n = (int)(pix / (uint32_t)(H * W));
            on[k] = px < (valid_w ? valid_w[n] : W);
            if (on[k]) {
                v[k] = *reinterpret_cast<const float4*>(x + (size_t)pix * x_cs + c);
                m2[k] = mr[(size_t)n * G + g];
            }
        }
    }
#pragma unroll
    for (int k = 0; k < GN_PPT; ++k) {
        if (!live[k]) continue;
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        if (on[k]) {
            const float mean = m2[k].x, rstd = m2[k].y;
            float t[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float u = (t[j] - mean) * rstd * gam[j] + bet[j];
                // ex2.approx + IEEE-rounded reciprocal: ~2e-7 relative on the sigmoid.  expf + a full-range division cost ~25 of this
                // kernel's ~40 instructions per element and made it ISSUE-bound at 3.9 TB/s (round 2; same transform as conv_tc2's fused path)
                if (swish) u = u * __frcp_rn(1.f + __expf(-u));
                t[j] = u;
            }
            o = make_float4(t[0], t[1], t[2], t[3]);
        }
        *reinterpret_cast<float4*>(y + (size_t)(pix0 + (uint32_t)k * pix_stride) * y_cs + c) = o;
    }
}

// ---------------------------------------------------------------- AdaIN + concat
// Pass 1: per (character, channel) sum / sum-of-squares of the prior crop and of the LR-feature window, fp64 atomics.
// Pass 2: elementwise normalise + concat.  Both passes use float4 channel vectors (coalesced pixel rows).
__global__ void __launch_bounds__(256) adain_stats_kernel(const float* __restrict__ prior, int prior_cs, const float* __restrict__ feat, int feat_cs,
                                                          const mn_window* __restrict__ win, double* __restrict__ stats,
                                                          int H, int Wp, int W, int C, int pix_per_block) {
    mn_pdl_prologue();
    const int i = blockIdx.y;
    const mn_window wn = win[i];
    const int wv = wn.x2 - wn.x1;
    const int npix = H * wv;
    const int tpp = C >> 2, ppi = blockDim.x / tpp;
    const int my_c = (threadIdx.x % tpp) * 4, my_p = threadIdx.x / tpp;
    const int p_begin = blockIdx.x * pix_per_block, p_end = min(npix, p_begin + pix_per_block);
    const float* pr = prior + (size_t)i * H * Wp * prior_cs + my_c;
    const float* ft = feat + (size_t)wn.line * H * W * feat_cs + my_c;
    float4 sp = make_float4(0.f, 0.f, 0.f, 0.f), qp = sp, sl = sp, ql = sp;
    double acc[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) acc[k] = 0.0;
    int cnt = 0;
    auto flush = [&]() {
        acc[0] += sp.x; acc[1] += sp.y; acc[2] += sp.z; acc[3] += sp.w; acc[4] += qp.x; acc[5] += qp.y; acc[6] += qp.z; acc[7] += qp.w;
        acc[8] += sl.x; acc[9] += sl.y; acc[10] += sl.z; acc[11] += sl.w; acc[12] += ql.x; acc[13] += ql.y; acc[14] += ql.z; acc[15] += ql.w;
        sp = qp = sl = ql = make_float4(0.f, 0.f, 0.f, 0.f);
        cnt = 0;
    };
    if (my_p < ppi && wv > 0) {
        // four pixels per trip, all eight loads issued before the first add (two loads in flight per thread left the kernel at
        // ~2.7 TB/s); same pixel order and flush cadence per thread, the zero-filled tail adds nothing: bit-identical sums
        for (int p = p_begin + my_p; p < p_end; p += 4 * ppi) {
            float4 a[4], b[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int pu = p + u * ppi;
                a[u] = b[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (pu < p_end) {
                    const int yy = pu / wv, xx = pu - yy * wv;
                    a[u] = *reinterpret_cast<const float4*>(pr + ((size_t)yy * Wp + wn.y1 + xx) * prior_cs);
                    b[u] = *reinterpret_cast<const float4*>(ft + ((size_t)yy * W + wn.x1 + xx) * feat_cs);
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                sp.x += a[u].x; sp.y += a[u].y; sp.z += a[u].z; sp.w += a[u].w;
                qp.x = fmaf(a[u].x, a[u].x, qp.x); qp.y = fmaf(a[u].y, a[u].y, qp.y); qp.z = fmaf(a[u].z, a[u].z, qp.z); qp.w = fmaf(a[u].w, a[u].w, qp.w);
                sl.x += b[u].x; sl.y += b[u].y; sl.z += b[u].z; sl.w += b[u].w;
                ql.x = fmaf(b[u].x, b[u].x, ql.x); ql.y = fmaf(b[u].y, b[u].y, ql.y); ql.z = fmaf(b[u].z, b[u].z, ql.z); ql.w = fmaf(b[u].w, b[u].w, ql.w);
            }
            cnt += 4;
            if (cnt >= 16) flush();
        }
    }
    flush();
    // reduce the ppi pixel slots of the block in shared memory, then one atomic per (block, channel, moment)
    __shared__ double red[256][17];
#pragma unroll
    for (int k = 0; k < 16; ++k) red[threadIdx.x][k] = acc[k];
    __syncthreads();
    if (my_p == 0) {
        for (int sl2 = 1; sl2 < ppi; ++sl2)
#pragma unroll
            for (int k = 0; k < 16; ++k) acc[k] += red[sl2 * tpp + threadIdx.x][k];
        double* st = stats + ((size_t)i * C + my_c) * 4;          // [i][c][{sum_p, sq_p, sum_l, sq_l}]
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            atomicAdd(st + j * 4 + 0, acc[j]); atomicAdd(st + j * 4 + 1, acc[4 + j]);
            atomicAdd(st + j * 4 + 2, acc[8 + j]); atomicAdd(st + j * 4 + 3, acc[12 + j]);
        }
    }
}

// fp64 moments -> fp32 {prior mean, prior std, lq mean, lq std} per (character, channel); unbiased variance + 1e-5.
__global__ void adain_finalize_kernel(const double* __restrict__ stats, const mn_window* __restrict__ win, float4* __restrict__ ms,
                                      int Nc, int C, int H) {
    mn_pdl_prologue();
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= Nc * C) return;
    const mn_window wn = win[idx / C];
    const double cnt = (double)H * (wn.x2 - wn.x1);
    const double* st = stats + (size_t)idx * 4;
    const double pm = st[0] / cnt, lm = st[2] / cnt;
    double pvar = (st[1] - st[0] * pm) / (cnt - 1.0), lvar = (st[3] - st[2] * lm) / (cnt - 1.0);
    pvar = pvar < 0.0 ? 0.0 : pvar; lvar = lvar < 0.0 ? 0.0 : lvar;
    ms[idx] = make_float4((float)pm, sqrtf((float)pvar + 1e-5f), (float)lm, sqrtf((float)lvar + 1e-5f));
}

__global__ void adain_apply_kernel(const float* __restrict__ prior, int prior_cs, const float* __restrict__ feat, int feat_cs,
                                   const mn_window* __restrict__ win, const float4* __restrict__ ms, float* __restrict__ out,
                                   int Nc, int H, int Wp, int W, int C) {
    mn_pdl_prologue();
    const int c4 = C >> 2;
    const int64_t total = (int64_t)Nc * H * Wp * c4;
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;     // host guarantees total < 2^31: 32-bit div/mod only
    if (idx >= (uint32_t)total) return;
    const int c = (int)(idx % c4) * 4;
    uint32_t pix = idx / c4;
    const int xx = (int)(pix % Wp);
    const int yy = (int)((pix / Wp) % H);
    const int i = (int)(pix / (uint32_t)(Wp * H));
    const mn_window wn = win[i];
    const int wv = wn.x2 - wn.x1;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    if (xx < wv) {
        const float4 pv = *reinterpret_cast<const float4*>(prior + (((size_t)i * H + yy) * Wp + wn.y1 + xx) * prior_cs + c);
        b = *reinterpret_cast<const float4*>(feat + (((size_t)wn.line * H + yy) * W + wn.x1 + xx) * feat_cs + c);
        float pvv[4] = {pv.x, pv.y, pv.z, pv.w}, o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float4 q = ms[(size_t)i * C + c + j];          // {prior mean, prior std, lq mean, lq std}
            o[j] = __fadd_rn(__fmul_rn(__fdiv_rn(pvv[j] - q.x, q.y), q.w), q.z);
        }
        a = make_float4(o[0], o[1], o[2], o[3]);
    }
    float* op = out + (size_t)pix * (2 * C);
    *reinterpret_cast<float4*>(op + c) = a;
    *reinterpret_cast<float4*>(op + C + c) = b;
}

// ---------------------------------------------------------------- window write-back
__global__ void window_scatter_kernel(const float* __restrict__ feat, int feat_cs, const float* __restrict__ scale,
                                      const float* __restrict__ shift, const int32_t* __restrict__ owner,
                                      const mn_window* __restrict__ win, float* __restrict__ out, int out_cs,
                                      int B, int H, int W, int Wp, int C) {
    mn_pdl_prologue();
    const int c4 = C >> 2;
    const int64_t total = (int64_t)B * H * W * c4;
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;     // host guarantees total < 2^31: 32-bit div/mod only
    if (idx >= (uint32_t)total) return;
    const int c = (int)(idx % c4) * 4;
    const uint32_t pix = idx / c4;
    const int x = (int)(pix % W);
    const int y = (int)((pix / W) % H);
    const int b = (int)(pix / (uint32_t)(H * W));
    const float4 f = *reinterpret_cast<const float4*>(feat + (size_t)pix * feat_cs + c);
    float4 o = f;
    const int i = owner[(size_t)b * W + x];
    if (i >= 0) {
        const int xx = x - win[i].x1;
        const size_t off = (((size_t)i * H + y) * Wp + xx) * C + c;
        const float4 sc = *reinterpret_cast<const float4*>(scale + off);
        const float4 sh = *reinterpret_cast<const float4*>(shift + off);
        o.x = __fadd_rn(f.x, __fadd_rn(__fmul_rn(f.x, sc.x), sh.x));
        o.y = __fadd_rn(f.y, __fadd_rn(__fmul_rn(f.y, sc.y), sh.y));
        o.z = __fadd_rn(f.z, __fadd_rn(__fmul_rn(f.z, sc.z), sh.z));
        o.w = __fadd_rn(f.w, __fadd_rn(__fmul_rn(f.w, sc.w), sh.w));
    }
    *reinterpret_cast<float4*>(out + (size_t)pix * out_cs + c) = o;
}

// ---------------------------------------------------------------- window integers on the device (networks.py:426-441 / :460-474)
// One CTA per LR line.  Phase 1: one thread per character computes (x1, x2, y1) with the reference's arithmetic
// (fp32 multiply, truncation toward zero).  Phase 2: one thread per column finds its owner = the LAST character in
// program order whose window covers it (networks.py:448,481).  An empty window (the reference dies on the empty slice
// at networks.py:443) raises bit 1 of *err and is replaced by a zero-width window so that no consumer reads out of bounds.
__global__ void char_windows_kernel(const float* __restrict__ locs, int locs_stride, const int32_t* __restrict__ line_first,
                                    int W, int half, mn_window* __restrict__ win, int32_t* __restrict__ valid,
                                    int32_t* __restrict__ owner, int32_t* __restrict__ err) {
    mn_pdl_prologue();
    extern __shared__ int32_t sw[];            // [n][2] = x1, x2 of this line's characters
    const int b = blockIdx.x;
    const int first = line_first[b], n = line_first[b + 1] - first;
    for (int c = threadIdx.x; c < n; c += blockDim.x) {
        const int center = __float2int_rz(__fmul_rn(locs[(size_t)b * locs_stride + 2 * c], (float)W));
        int x1 = center < half ? 0 : center - half;
        int x2 = center + half > W ? W : center + half;
        int wv = x2 - x1;
        if (wv <= 0 || x1 >= W) { atomicOr(err, 2); x1 = 0; x2 = 0; wv = 0; }
        mn_window w;
        w.line = b; w.x1 = x1; w.x2 = x2; w.y1 = half - wv / 2;
        win[first + c] = w;
        valid[first + c] = wv;
        sw[2 * c] = x1; sw[2 * c + 1] = x2;
    }
    __syncthreads();
    for (int x = threadIdx.x; x < W; x += blockDim.x) {
        int o = -1;
        for (int c = 0; c < n; ++c)
            if (x >= sw[2 * c] && x < sw[2 * c + 1]) o = first + c;
        owner[(size_t)b * W + x] = o;
    }
}

// ---------------------------------------------------------------- style per character of a wide line
// A line wider than the encoder's 512 columns is encoded as `segs` segments of seg_w columns (one style row each).  Character c
// of line b takes the style of the segment holding its centre, computed with the 32-level window centre's arithmetic
// (networks.py:426: fp32 multiply, truncation toward zero) and clamped into [0, segs).  One CTA per character.
__global__ void char_segment_styles_kernel(const float* __restrict__ w, int w_stride, const float* __restrict__ locs, int locs_stride,
                                           const int32_t* __restrict__ line_first, int W, int seg_w, int segs, int dim,
                                           float* __restrict__ styles, int styles_stride, int32_t* __restrict__ seg_out) {
    mn_pdl_prologue();
    const int b = blockIdx.y, c = blockIdx.x;
    const int first = line_first[b];
    if (c >= line_first[b + 1] - first) return;
    const int center = __float2int_rz(__fmul_rn(locs[(size_t)b * locs_stride + 2 * c], (float)W));
    int seg = center < 0 ? 0 : center / seg_w;
    if (seg > segs - 1) seg = segs - 1;
    const float* src = w + (size_t)(b * segs + seg) * w_stride;
    float* dst = styles + (size_t)(first + c) * styles_stride;
    for (int k = threadIdx.x; k < dim; k += blockDim.x) dst[k] = src[k];
    if (seg_out && threadIdx.x == 0) seg_out[first + c] = seg;
}

// ---------------------------------------------------------------- standalone helper functions of the reference module
// swish (networks.py:492-493), calc_mean_std_4D (:518-525), adaptive_instance_normalization (:528-533) on NCHW-contiguous
// tensors, rows = B*C, len = H*W.  The hot path uses the fused NHWC kernels above; these keep the reference's module-level
// function names usable on CUDA tensors.
__global__ void swish_kernel(const float* __restrict__ x, float* __restrict__ y, int64_t n) {
    mn_pdl_prologue();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float v = x[i];
        y[i] = v * (1.f / (1.f + expf(-v)));
    }
}

// one block per row: mean and sqrt(unbiased variance + eps); two-pass in fp64 partials (matches torch.var to fp32 rounding)
__global__ void row_mean_std_kernel(const float* __restrict__ x, float* __restrict__ mean, float* __restrict__ stdv, int len, float eps) {
    mn_pdl_prologue();
    __shared__ double red[32];
    __shared__ double s_mean;
    const float* xr = x + (size_t)blockIdx.x * len;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    double a = 0.0;
    for (int i = threadIdx.x; i < len; i += blockDim.x) a += (double)xr[i];
    a = mn_warp_sum_d(a);
    if (lane == 0) red[warp] = a;
    __syncthreads();
    if (threadIdx.x == 0) { double t = 0.0; for (int w = 0; w < nw; ++w) t += red[w]; s_mean = t / (double)len; }
    __syncthreads();
    const double m = s_mean;
    double q = 0.0;
    for (int i = threadIdx.x; i < len; i += blockDim.x) { const double d = (double)xr[i] - m; q += d * d; }
    q = mn_warp_sum_d(q);
    __syncthreads();
    if (lane == 0) red[warp] = q;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < nw; ++w) t += red[w];
        mean[blockIdx.x] = (float)m;
        stdv[blockIdx.x] = sqrtf((float)(t / (double)(len > 1 ? len - 1 : 1)) + eps);
    }
}

__global__ void adain_rows_kernel(const float* __restrict__ prior, const float* __restrict__ pm, const float* __restrict__ ps,
                                  const float* __restrict__ lm, const float* __restrict__ ls, float* __restrict__ out, int len) {
    mn_pdl_prologue();
    const size_t base = (size_t)blockIdx.x * len;
    const float m = pm[blockIdx.x], sd = ps[blockIdx.x], a = ls[blockIdx.x], b = lm[blockIdx.x];
    for (int i = threadIdx.x; i < len; i += blockDim.x) out[base + i] = (prior[base + i] - m) / sd * a + b;
}

}  // namespace

extern "C" int mn_swish(const float* x, float* y, long long n, void* stream) {
    MN_REQUIRE(x && y && n >= 0, "mn_swish: bad args");
    if (n == 0) return MN_OK;
    const int blocks = (int)(mn_cdiv64(n, 256) < 148 * 8 ? mn_cdiv64(n, 256) : 148 * 8);
    MN_CUDA_CHECK(mn_launch(swish_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, x, y, (int64_t)n));
    return MN_OK;
}

extern "C" int mn_row_mean_std(const float* x, float* mean, float* stdv, int rows, int len, float eps, void* stream) {
    MN_REQUIRE(x && mean && stdv && rows > 0 && len > 0, "mn_row_mean_std: bad args");
    MN_CUDA_CHECK(mn_launch(row_mean_std_kernel, dim3(rows), dim3(256), 0, (cudaStream_t)stream, x, mean, stdv, len, eps));
    return MN_OK;
}

extern "C" int mn_adain_rows(const float* prior, const float* prior_mean, const float* prior_std, const float* lq_mean,
                             const float* lq_std, float* out, int rows, int len, void* stream) {
    MN_REQUIRE(prior && prior_mean && prior_std && lq_mean && lq_std && out && rows > 0 && len > 0, "mn_adain_rows: bad args");
    MN_CUDA_CHECK(mn_launch(adain_rows_kernel, dim3(rows), dim3(256), 0, (cudaStream_t)stream, prior, prior_mean, prior_std, lq_mean, lq_std, out, len));
    return MN_OK;
}

static int gn_check(const float* x, int x_cs, int N, int H, int W, int C, int cpg) {
    MN_REQUIRE(x && N > 0 && H > 0 && W > 0 && C > 0, "groupnorm: bad dims");
    MN_REQUIRE(cpg == 32 && C % 32 == 0 && (256 % (C >> 2)) == 0 && C <= 1024, "groupnorm: needs 32 channels per group and C/4 dividing 256");
    MN_REQUIRE((x_cs & 3) == 0 && ((uintptr_t)x & 15) == 0, "groupnorm: alignment");
    return MN_OK;
}

extern "C" int mn_groupnorm_stats(const float* x, int x_cs, int N, int H, int W, int C, int cpg, float eps,
                                  const int32_t* valid_w, double* stats_ws, float* mean_rstd, void* stream) {
    int rc = gn_check(x, x_cs, N, H, W, C, cpg);
    if (rc != MN_OK) return rc;
    MN_REQUIRE(stats_ws && mean_rstd, "mn_groupnorm_stats: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const int G = C / cpg;
    MN_CUDA_CHECK(cudaMemsetAsync(stats_ws, 0, sizeof(double) * 2 * N * G, st));
    const int HW = H * W;
    int blocks = mn_cdiv(mn_num_sms() * 8, N);
    if (blocks > mn_cdiv(HW, 32)) blocks = mn_cdiv(HW, 32);
    if (blocks < 1) blocks = 1;
    const int ppb = mn_cdiv(HW, blocks);
    blocks = mn_cdiv(HW, ppb);
    MN_CUDA_CHECK((mn_launch(gn_stats_kernel, dim3(dim3(blocks, N)), dim3(256), 0, st, x, x_cs, H, W, C, cpg, valid_w, stats_ws, ppb)));
    MN_LAUNCH_CHECK();
    MN_CUDA_CHECK((mn_launch(gn_finalize_kernel, dim3(mn_cdiv(N * G, 128)), dim3(128), 0, st, stats_ws, reinterpret_cast<float2*>(mean_rstd), N, G, H, W, cpg, eps, valid_w)));
    MN_LAUNCH_CHECK();
    return MN_OK;
}

extern "C" int mn_groupnorm_finalize(const double* stats_ws, int N, int H, int W, int C, int cpg, float eps, const int32_t* valid_w,
                                     float* mean_rstd, void* stream) {
    MN_REQUIRE(stats_ws && mean_rstd && N > 0 && H > 0 && W > 0 && C > 0 && cpg == 32 && C % 32 == 0, "mn_groupnorm_finalize: bad args");
    const int G = C / cpg;
    MN_CUDA_CHECK((mn_launch(gn_finalize_kernel, dim3(mn_cdiv(N * G, 128)), dim3(128), 0, (cudaStream_t)stream, stats_ws,
                             reinterpret_cast<float2*>(mean_rstd), N, G, H, W, cpg, eps, valid_w)));
    MN_LAUNCH_CHECK();
    return MN_OK;
}

extern "C" int mn_groupnorm_apply(const float* x, int x_cs, float* y, int y_cs, const float* gamma, const float* beta,
                                  const float* mean_rstd, int N, int H, int W, int C, int cpg, int swish,
                                  const int32_t* valid_w, void* stream) {
    int rc = gn_check(x, x_cs, N, H, W, C, cpg);
    if (rc != MN_OK) return rc;
    MN_REQUIRE(y && gamma && beta && mean_rstd && (y_cs & 3) == 0 && ((uintptr_t)y & 15) == 0, "mn_groupnorm_apply: bad args");
    const int64_t total = (int64_t)N * H * W * (C >> 2);
    MN_REQUIRE(total < (1ll << 31), "tensor too large for 32-bit indexing");
    const uint32_t pix_stride = (uint32_t)mn_cdiv64((int64_t)N * H * W, GN_PPT);
    MN_CUDA_CHECK((mn_launch(gn_apply_kernel, dim3((unsigned)mn_cdiv64((int64_t)pix_stride * (C >> 2), 256)), dim3(256), 0, (cudaStream_t)stream, x, x_cs, y, y_cs, gamma, beta, N, H, W, C, cpg, 0.f, swish, valid_w,
                             reinterpret_cast<const float2*>(mean_rstd), pix_stride)));
    MN_LAUNCH_CHECK();
    return MN_OK;
}

extern "C" int mn_groupnorm_swish(const float* x, int x_cs, float* y, int y_cs, const float* gamma, const float* beta,
                                  int N, int H, int W, int C, int cpg, float eps, int swish,
                                  const int32_t* valid_w, double* stats_ws, void* stream) {
    MN_REQUIRE(stats_ws != nullptr, "mn_groupnorm_swish: null workspace");
    float* mr = reinterpret_cast<float*>(stats_ws + 2 * (size_t)N * (C / (cpg > 0 ? cpg : 1)));   // second part of the workspace
    int rc = mn_groupnorm_stats(x, x_cs, N, H, W, C, cpg, eps, valid_w, stats_ws, mr, stream);
    if (rc != MN_OK) return rc;
    return mn_groupnorm_apply(x, x_cs, y, y_cs, gamma, beta, mr, N, H, W, C, cpg, swish, valid_w, stream);
}

extern "C" int mn_adain_concat(const float* prior, int prior_cs, const float* feat, int feat_cs, const mn_window* win,
                               float* out, int Nc, int H, int Wp, int W, int C, double* stats_ws, void* stream) {
    MN_REQUIRE(prior && feat && win && out && stats_ws && Nc > 0 && H > 0 && Wp > 0 && W > 0 && C > 0, "mn_adain_concat: bad args");
    MN_REQUIRE((C & 3) == 0 && 256 % (C >> 2) == 0 && (prior_cs & 3) == 0 && (feat_cs & 3) == 0 &&
               ((uintptr_t)prior & 15) == 0 && ((uintptr_t)feat & 15) == 0 && ((uintptr_t)out & 15) == 0,
               "mn_adain_concat: C/4 must divide 256 and all operands must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    MN_CUDA_CHECK(cudaMemsetAsync(stats_ws, 0, sizeof(double) * 4 * (size_t)Nc * C, st));
    const int npix_max = H * Wp;
    int blocks = mn_cdiv(mn_num_sms() * 4, Nc);
    if (blocks > mn_cdiv(npix_max, 32)) blocks = mn_cdiv(npix_max, 32);
    if (blocks < 1) blocks = 1;
    const int ppb = mn_cdiv(npix_max, blocks);
    blocks = mn_cdiv(npix_max, ppb);
    MN_CUDA_CHECK((mn_launch(adain_stats_kernel, dim3(dim3(blocks, Nc)), dim3(256), 0, st, prior, prior_cs, feat, feat_cs, win, stats_ws, H, Wp, W, C, ppb)));
    MN_LAUNCH_CHECK();
    float4* ms = reinterpret_cast<float4*>(stats_ws + 4 * (size_t)Nc * C);    // second part of the workspace
    MN_CUDA_CHECK((mn_launch(adain_finalize_kernel, dim3(mn_cdiv(Nc * C, 256)), dim3(256), 0, st, stats_ws, win, ms, Nc, C, H)));
    MN_LAUNCH_CHECK();
    const int64_t total = (int64_t)Nc * H * Wp * (C >> 2);
    MN_REQUIRE(total < (1ll << 31), "tensor too large for 32-bit indexing");
    MN_CUDA_CHECK((mn_launch(adain_apply_kernel, dim3((unsigned)mn_cdiv64(total, 256)), dim3(256), 0, st, prior, prior_cs, feat, feat_cs, win, ms, out, Nc, H, Wp, W, C)));
    MN_LAUNCH_CHECK();
    return MN_OK;
}

extern "C" int mn_window_scatter(const float* feat, int feat_cs, const float* scale, const float* shift,
                                 const int32_t* owner, const mn_window* win, float* out, int out_cs,
                                 int B, int H, int W, int Wp, int C, void* stream) {
    MN_REQUIRE(feat && scale && shift && owner && win && out, "mn_window_scatter: null pointer");
    MN_REQUIRE(B > 0 && H > 0 && W > 0 && Wp > 0 && (C & 3) == 0 && (feat_cs & 3) == 0 && (out_cs & 3) == 0, "mn_window_scatter: bad dims");
    const int64_t total = (int64_t)B * H * W * (C >> 2);
    MN_REQUIRE(total < (1ll << 31), "tensor too large for 32-bit indexing");
    MN_CUDA_CHECK((mn_launch(window_scatter_kernel, dim3((unsigned)mn_cdiv64(total, 256)), dim3(256), 0, (cudaStream_t)stream, feat, feat_cs, scale, shift, owner, win, out, out_cs, B, H, W, Wp, C)));
    MN_LAUNCH_CHECK();
    return MN_OK;
}

extern "C" int mn_char_windows(const float* locs, int locs_stride, const int32_t* line_first, int B, int max_chars, int W, int half,
                               mn_window* win, int32_t* valid, int32_t* owner, int32_t* err, void* stream) {
    MN_REQUIRE(locs && line_first && win && valid && owner && err, "mn_char_windows: null pointer");
    MN_REQUIRE(B > 0 && W > 0 && half > 0 && max_chars >= 0 && max_chars <= 4096, "mn_char_windows: bad dims");
    MN_CUDA_CHECK((mn_launch(char_windows_kernel, dim3(B), dim3(256), (size_t)max_chars * 2 * sizeof(int32_t), (cudaStream_t)stream,
                             locs, locs_stride, line_first, W, half, win, valid, owner, err)));
    MN_LAUNCH_CHECK();
    return MN_OK;
}

extern "C" int mn_char_segment_styles(const float* w, int w_stride, const float* locs, int locs_stride, const int32_t* line_first,
                                      int B, int max_chars, int W, int seg_w, int segs, int dim, float* styles, int styles_stride,
                                      int32_t* seg_out, void* stream) {
    MN_REQUIRE(w && locs && line_first && styles, "mn_char_segment_styles: null pointer");
    MN_REQUIRE(B > 0 && W > 0 && seg_w > 0 && segs > 0 && dim > 0 && max_chars >= 0 && max_chars <= 65535 && B <= 65535 &&
               w_stride >= dim && styles_stride >= dim && (int64_t)B * segs < (1ll << 31), "mn_char_segment_styles: bad dims");
    if (max_chars == 0) return MN_OK;
    MN_CUDA_CHECK((mn_launch(char_segment_styles_kernel, dim3(max_chars, B), dim3(128), 0, (cudaStream_t)stream,
                             w, w_stride, locs, locs_stride, line_first, W, seg_w, segs, dim, styles, styles_stride, seg_out)));
    MN_LAUNCH_CHECK();
    return MN_OK;
}
