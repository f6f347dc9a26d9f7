// mn_conv2d_nhwc: argument validation and dispatch between the convolution kernels.
#include "mn_common.cuh"
#include "conv_common.cuh"

static int make_geom(const mn_conv_params* p, ConvGeom& g) {
    MN_REQUIRE(p != nullptr, "mn_conv2d_nhwc: null params");
    MN_REQUIRE(p->x && p->w && (p->y || p->y2), "mn_conv2d_nhwc: null x/w/y");
    MN_REQUIRE(p->N > 0 && p->H > 0 && p->W > 0 && p->Cin > 0 && p->Cout > 0, "mn_conv2d_nhwc: non-positive dims");
    MN_REQUIRE(p->KH > 0 && p->KW > 0 && p->stride_h > 0 && p->stride_w > 0 && p->pad_h >= 0 && p->pad_w >= 0,
               "mn_conv2d_nhwc: bad kernel/stride/pad");
    MN_REQUIRE(p->x_cs >= p->Cin, "mn_conv2d_nhwc: x_cs < Cin");
    g.x = p->x; g.w = p->w; g.y = p->y; g.y2 = p->y2;
    g.bias = p->bias; g.out_scale = p->out_scale; g.residual = p->residual; g.y2_scale = p->y2_scale;
    g.valid_w = p->valid_w; g.ws = p->workspace; g.ws_bytes = p->workspace ? p->workspace_bytes : 0;
    g.gn_mr = reinterpret_cast<const float2*>(p->gn_mean_rstd); g.gn_gamma = p->gn_gamma; g.gn_beta = p->gn_beta; g.gn_swish = p->gn_swish;
    MN_REQUIRE(!p->gn_mean_rstd || (p->gn_gamma && p->gn_beta && p->Cin % 32 == 0), "mn_conv2d_nhwc: fused GroupNorm needs gamma, beta and Cin % 32 == 0");
    g.N = p->N; g.H = p->H; g.W = p->W; g.Cin = p->Cin; g.x_cs = p->x_cs;
    g.KH = p->KH; g.KW = p->KW; g.sh = p->stride_h; g.sw = p->stride_w; g.ph = p->pad_h; g.pw = p->pad_w; g.Cout = p->Cout;
    g.OH = (p->H + 2 * p->pad_h - p->KH) / p->stride_h + 1;
    g.OW = (p->W + 2 * p->pad_w - p->KW) / p->stride_w + 1;
    MN_REQUIRE(g.OH > 0 && g.OW > 0, "mn_conv2d_nhwc: empty output");
    g.y_cs = p->y_cs; g.y2_cs = p->y2_cs; g.res_cs = p->res_cs; g.res_bcast = p->res_broadcast_n;
    MN_REQUIRE(!p->y || p->y_cs >= p->Cout, "mn_conv2d_nhwc: y_cs < Cout");
    MN_REQUIRE(!p->y2 || p->y2_cs >= p->Cout, "mn_conv2d_nhwc: y2_cs < Cout");
    MN_REQUIRE(!p->residual || p->res_cs >= p->Cout, "mn_conv2d_nhwc: res_cs < Cout");
    g.os_stride = p->out_scale_stride > 0 ? p->out_scale_stride : p->Cout;
    g.y2s_stride = p->y2_scale_stride > 0 ? p->y2_scale_stride : p->Cout;
    g.act = p->act; g.gain = p->act_gain;
    const int64_t M = (int64_t)p->N * g.OH * g.OW;
    MN_REQUIRE(M < (1ll << 31) && (int64_t)p->KH * p->KW * p->Cin < (1ll << 31), "mn_conv2d_nhwc: problem too large");
    g.M = (int)M; g.K = p->KH * p->KW * p->Cin;
    g.ktiles = g.ktiles_per_split = 0; g.splits = 1;
    g.x_scale = p->x_scale > 0.f ? p->x_scale : 1.f; g.x_absmax = p->x_absmax; g.range_flag = p->range_flag; g.range_tag = p->range_tag;
    g.y2_ptrs = p->y2_ptrs; g.gn_stats_out = p->gn_stats_out;
    MN_REQUIRE(!p->gn_stats_out || (p->Cout % 32 == 0 && p->y), "mn_conv2d_nhwc: gn_stats_out needs Cout % 32 == 0 and the y output");
    MN_REQUIRE(!p->y2_ptrs || p->y2, "mn_conv2d_nhwc: y2_ptrs needs the second output enabled (y2 != NULL)");
    return MN_OK;
}

extern "C" int64_t mn_conv2d_workspace_bytes(const mn_conv_params* p) {
    ConvGeom g;
    if (make_geom(p, g) != MN_OK) return -1;
    const int splits = mn_conv_simt_plan_splits(g, (int64_t)1 << 60, p->split_k);
    return splits > 1 ? (int64_t)splits * g.M * g.Cout * 4 : 0;
}

extern "C" int mn_conv2d_nhwc(const mn_conv_params* p, void* stream) {
    ConvGeom g;
    int rc = make_geom(p, g);
    if (rc != MN_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (p->precision) {
        case MN_PREC_FP32_SIMT:
            if (g.gn_mr || g.y2_ptrs || g.gn_stats_out) {
                mn_set_error("mn_conv2d_nhwc: the fused GroupNorm input transform (gn_mean_rstd), per-sample output pointers (y2_ptrs) and "
                             "epilogue GroupNorm statistics (gn_stats_out) need the tensor-core path");
                return MN_ERR_UNSUPPORTED;
            }
            if (mn_conv_small_supported(g)) return mn_conv_small_launch(g, st);
            g.splits = mn_conv_simt_plan_splits(g, p->workspace ? p->workspace_bytes : 0, p->split_k);
            return mn_conv_simt_launch(g, nullptr, st);
        case MN_PREC_F16X3_TC:
        case MN_PREC_BF16X3_TC:
        case MN_PREC_F16X1_TC:
            return mn_conv_tc2_launch(g, p->w_tc_hi, p->w_tc_lo, p->w_tc_scale, p->precision, st);
        default:
            mn_set_error("mn_conv2d_nhwc: unknown precision mode %d", p->precision);
            return MN_ERR_UNSUPPORTED;
    }
}

extern "C" int mn_conv2d_tc_supported(const mn_conv_params* p) {
    ConvGeom g;
    if (make_geom(p, g) != MN_OK) return 0;
    const char* why = "";
    const int ok = mn_conv_tc2_supported(g, &why);
    if (!ok) mn_set_error("tensor-core path unsupported: %s", why);
    return ok;
}
