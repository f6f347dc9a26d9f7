// Geometry + fused epilogue shared by the convolution kernels (SIMT fp32 and tcgen05).
#pragma once
#include "mn_common.cuh"

struct ConvGeom {
    const float* x; const float* w;
    float* y; float* y2;
    const float* bias; const float* out_scale; const float* residual; const float* y2_scale;
    const int32_t* valid_w; float* ws; int64_t ws_bytes;
    const float2* gn_mr; const float* gn_gamma; const float* gn_beta; int gn_swish;   // fused GroupNorm(+swish) on the input (tensor-core path only)
    int N, H, W, Cin, x_cs;
    int KH, KW, sh, sw, ph, pw, Cout;
    int OH, OW, y_cs, y2_cs, res_cs, res_bcast, os_stride, y2s_stride;
    int act; float gain;
    int M, K;
    int ktiles, ktiles_per_split, splits;
    float x_scale; float* x_absmax; int32_t* range_flag; int32_t range_tag;   // fp16-range management (tensor-core precisions)
    float* const* y2_ptrs;     // per-sample base pointers of the second output (peer-GPU stores), tensor-core path only
    double* gn_stats_out;      // [N][Cout/32][2] sum / sum of squares of the output (GroupNorm statistics in the epilogue), tensor-core path only
};

// Range bookkeeping of the operand-split stage: `amax` = bits of the running fmaxf(|x * x_scale|) a thread has seen (fmaxf drops
// NaNs: a NaN input is not flagged -- it reaches the output as NaN -- an Inf or an out-of-range finite value is).
__device__ __forceinline__ void conv_range_report(const ConvGeom& g, uint32_t amax, bool fp16_mode) {
    if (!g.x_absmax && !g.range_flag) return;
    amax = __reduce_max_sync(0xffffffffu, amax);
    if ((threadIdx.x & 31) == 0) {
        if (g.x_absmax) atomicMax(reinterpret_cast<unsigned int*>(g.x_absmax), amax);
        // 65504 = 0x477FE000; Inf / NaN >= 0x7F800000
        if (g.range_flag && amax >= (fp16_mode ? 0x477FE000u : 0x7F800000u)) *reinterpret_cast<volatile int32_t*>(g.range_flag) = g.range_tag;
    }
}

// Epilogue for 4 consecutive output channels [o, o+4) of GEMM row m (pixel index in [N,OH,OW]).
//   v = acc*out_scale[n][o] + bias[o] + residual ; v = act(v)*gain ; masked by valid_w ; y, y2 stores.
__device__ __forceinline__ void conv_epilogue4(const ConvGeom& g, int m, int o, float v[4]) {
    const int hw = g.OH * g.OW;
    const int n = m / hw;
    const int nvalid = min(4, g.Cout - o);
    bool masked = false;
    if (g.valid_w) {
        const int ox = m % g.OW;
        masked = ox >= g.valid_w[n];
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (j < nvalid) {
            float t = v[j];
            if (g.out_scale) t *= g.out_scale[(size_t)n * g.os_stride + o + j];
            if (g.bias) t += g.bias[o + j];
            if (g.residual) {
                const size_t rm = g.res_bcast ? (size_t)(m - n * hw) : (size_t)m;
                t += g.residual[rm * g.res_cs + o + j];
            }
            t = mn_apply_act(t, g.act) * g.gain;
            v[j] = masked ? 0.f : t;
        }
    }
    const bool full = nvalid == 4;
    if (g.y) {
        float* dst = g.y + (size_t)m * g.y_cs + o;
        if (full && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
        else for (int j = 0; j < nvalid; ++j) dst[j] = v[j];
    }
    if (g.y2) {
        float u[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) u[j] = (j < nvalid && g.y2_scale) ? v[j] * g.y2_scale[(size_t)n * g.y2s_stride + o + j] : v[j];
        float* dst = g.y2 + (size_t)m * g.y2_cs + o;
        if (full && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) *reinterpret_cast<float4*>(dst) = make_float4(u[0], u[1], u[2], u[3]);
        else for (int j = 0; j < nvalid; ++j) dst[j] = u[j];
    }
}

// Vectorised epilogue for the tensor-core kernels: 4 consecutive channels [o,o+4) (o % 4 == 0, Cout % 4 == 0) of pixel m
// belonging to sample n; float4 loads of the per-channel / per-sample vectors, no integer division.
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void conv_epilogue_vec4(const ConvGeom& g, int m, int n, bool masked, int o, float4 v, float4 bias4) {
    if (g.out_scale) {
        const float4 s = ldg4(g.out_scale + (size_t)n * g.os_stride + o);
        v.x *= s.x; v.y *= s.y; v.z *= s.z; v.w *= s.w;
    }
    v.x += bias4.x; v.y += bias4.y; v.z += bias4.z; v.w += bias4.w;
    if (g.residual) {
        const size_t rm = g.res_bcast ? (size_t)(m - n * g.OH * g.OW) : (size_t)m;
        const float4 r = ldg4(g.residual + rm * g.res_cs + o);
        v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
    }
    if (g.act != MN_ACT_NONE) {
        v.x = mn_apply_act(v.x, g.act); v.y = mn_apply_act(v.y, g.act); v.z = mn_apply_act(v.z, g.act); v.w = mn_apply_act(v.w, g.act);
    }
    v.x *= g.gain; v.y *= g.gain; v.z *= g.gain; v.w *= g.gain;
    if (masked) v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (g.y) *reinterpret_cast<float4*>(g.y + (size_t)m * g.y_cs + o) = v;
    if (g.y2) {
        if (g.y2_scale) {
            const float4 s = ldg4(g.y2_scale + (size_t)n * g.y2s_stride + o);
            v.x *= s.x; v.y *= s.y; v.z *= s.z; v.w *= s.w;
        }
        *reinterpret_cast<float4*>(g.y2 + (size_t)m * g.y2_cs + o) = v;
    }
}

// Specialised row epilogue of the tensor-core kernels: the activation is a template parameter (ACT < 0: runtime g.act, the
// rarely used tanh / GELU / sigmoid heads) and the per-sample scale vectors may be passed in registers when every row of the tile
// belongs to one sample.  The generic conv_epilogue_vec4 above costs ~120 SASS instructions per float4 (jump table on the
// activation, predicated 64-bit address arithmetic for every optional operand); with four warps storing a 128x128 tile that was
// ~10k cycles per tile -- more than the MMA time of a Cin <= 128 tile (ncu source page, profiles/r2_tc2_epilogue_before.txt).
template <int ACT>
__device__ __forceinline__ float mn_act_t(float v, int act) {
    if (ACT == MN_ACT_NONE) return v;
    if (ACT == MN_ACT_RELU) return fmaxf(v, 0.f);
    if (ACT == MN_ACT_LRELU02) return v > 0.f ? v : 0.2f * v;
    return mn_apply_act(v, act);
}
template <int ACT>
__device__ __forceinline__ float4 conv_epilogue_row4(const ConvGeom& g, int m, int n, bool masked, int o, float4 v, const float4 bias4,
                                                     bool have_os, const float4 os4, bool have_y2s, const float4 y2s4, float* y2base) {
    if (g.out_scale) {
        const float4 s = have_os ? os4 : ldg4(g.out_scale + (size_t)n * g.os_stride + o);
        v.x *= s.x; v.y *= s.y; v.z *= s.z; v.w *= s.w;
    }
    v.x += bias4.x; v.y += bias4.y; v.z += bias4.z; v.w += bias4.w;
    if (g.residual) {
        const size_t rm = g.res_bcast ? (size_t)(m - n * g.OH * g.OW) : (size_t)m;
        const float4 r = ldg4(g.residual + rm * g.res_cs + o);
        v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
    }
    v.x = mn_act_t<ACT>(v.x, g.act) * g.gain; v.y = mn_act_t<ACT>(v.y, g.act) * g.gain;
    v.z = mn_act_t<ACT>(v.z, g.act) * g.gain; v.w = mn_act_t<ACT>(v.w, g.act) * g.gain;
    if (masked) v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (g.y) *reinterpret_cast<float4*>(g.y + (size_t)m * g.y_cs + o) = v;
    if (g.y2) {
        float4 u = v;
        if (g.y2_scale) {
            const float4 s = have_y2s ? y2s4 : ldg4(g.y2_scale + (size_t)n * g.y2s_stride + o);
            u.x *= s.x; u.y *= s.y; u.z *= s.z; u.w *= s.w;
        }
        *reinterpret_cast<float4*>(y2base + (size_t)m * g.y2_cs + o) = u;     // y2base = g.y2, or the sample's (peer) block rebased to m
    }
    return v;      // the stored y values (GroupNorm statistics in the epilogue)
}

int mn_conv_simt_plan_splits(const ConvGeom& g, int64_t ws_bytes, int requested);
int mn_conv_simt_launch(ConvGeom g, const float* unused, cudaStream_t st);
int mn_conv_splitk_reduce_launch(const ConvGeom& g, cudaStream_t st);   // sums g.splits partial tiles in g.ws and runs the fused epilogue

// tcgen05 path: halo tiles + weight multicast + persistent CTAs (conv_tc2.cu)
int mn_conv_tc2_supported(const ConvGeom& g, const char** why);
int mn_conv_tc2_launch(const ConvGeom& g, const void* w_hi, const void* w_lo, const float* w_scale, int prec, cudaStream_t st);
// direct 3x3 conv for Cout <= 4 (conv_small.cu)
bool mn_conv_small_supported(const ConvGeom& g);
int mn_conv_small_launch(const ConvGeom& g, cudaStream_t st);
