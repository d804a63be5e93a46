// Standalone layers either side of the cifar10 NeuralODE (SURVEY 8f n3, experiments/src/construct.jl:220-227):
// Conv((3,3), in => out, act; pad=1) with bias -- the AugmenterLayer's convolution (src/layers/common.jl:80-92) and the
// classifier's Conv(8 => 1, gelu) -- and BatchNorm(C, act).  Included by lrnde_api.cu; kernels in lrnde_conv.cuh.
#pragma once

namespace convops {

static int tile_rows(int PT, int Wd, int Ht) { return std::min(PT / (Wd >> 2), Ht); }

static void launch_conv(lrnde_ctx* ctx, ConvP& q, int64_t B) {
  q.B = (int)B;
  const bool nar = q.Cout <= 16;
  const int TR = tile_rows(nar ? 256 : 64, q.Wd, q.Ht);
  dim3 g((unsigned)(B * ((q.Ht + TR - 1) / TR)), (q.Cout + (nar ? 8 : 64) - 1) / (nar ? 8 : 64));
  if (nar) conv3x3_kernel<8, 8, 4><<<g, 256, 0, ctx->stream>>>(q);
  else conv3x3_kernel<64, 16, 8><<<g, 256, 0, ctx->stream>>>(q);
  LR_COUNT(ctx);
}

static void check_shape(const char* who, int in_ch, int out_ch, int W, int H, int64_t B) {
  if (in_ch < 1 || out_ch < 1 || B < 1 || H < 1 || W < 4 || W > 32 || (W & 3))
    lr_fail(LRNDE_EINVAL, "%s: bad shape (channels %d => %d, %d x %d, batch %lld; width must be a multiple of 4 in 4..32)",
            who, in_ch, out_ch, W, H, (long long)B);
}

}  // namespace convops

extern "C" int lrnde_conv2d_forward(lrnde_ctx* ctx, int32_t in_ch, int32_t out_ch, int32_t use_bias, int32_t act,
                                    int32_t width, int32_t height, const float* ps, const float* x, int64_t B,
                                    int32_t host_buffers, float* y) {
  LR_API_BEGIN
  if (!ctx || !ps || !x || !y) lr_fail(LRNDE_EINVAL, "lrnde_conv2d_forward: bad args");
  convops::check_shape("lrnde_conv2d_forward", in_ch, out_ch, width, height, B);
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t HW = (size_t)width * height, nx = HW * in_ch * B, ny = HW * out_ch * B;
  const size_t nw = (size_t)9 * in_ch * out_ch, np = nw + (use_bias ? out_ch : 0);
  CallerBufs io(ctx, host_buffers);
  const float* psd = io.in(ps, np);
  const float* xd = io.in(x, nx);
  float* yd = io.out(y, ny);
  DevBuf pack(ctx, nw);
  conv_pack_kernel<<<lr_ew_blocks(nw), 256, 0, st>>>(psd, in_ch, out_ch, 0, 0, pack.p);
  LR_COUNT(ctx);
  ConvP q;
  memset(&q, 0, sizeof(q));
  q.X = xd; q.Wp = pack.p; q.Wd = width; q.Ht = height; q.Cin = in_ch; q.Cout = out_ch; q.Y = yd; q.out_scale = 1.0f;
  q.bias = use_bias ? psd + nw : nullptr; q.out_act = lr_map_act(act);
  convops::launch_conv(ctx, q, B);
  LR_CHECK_LAUNCH();
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  LR_API_END
}

extern "C" int lrnde_conv2d_backward(lrnde_ctx* ctx, int32_t in_ch, int32_t out_ch, int32_t use_bias, int32_t act,
                                     int32_t width, int32_t height, const float* ps, const float* x, const float* d_y,
                                     int64_t B, int32_t host_buffers, float* d_x, float* d_ps) {
  LR_API_BEGIN
  if (!ctx || !ps || !x || !d_y || !d_ps) lr_fail(LRNDE_EINVAL, "lrnde_conv2d_backward: bad args");
  convops::check_shape("lrnde_conv2d_backward", in_ch, out_ch, width, height, B);
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int a = lr_map_act(act);
  const size_t HW = (size_t)width * height, nx = HW * in_ch * B, ny = HW * out_ch * B;
  const size_t nw = (size_t)9 * in_ch * out_ch, np = nw + (use_bias ? out_ch : 0);
  CallerBufs io(ctx, host_buffers);
  const float* psd = io.in(ps, np);
  const float* xd = io.in(x, nx);
  float* dg = io.copy_in(d_y, ny);   // owned copy: overwritten by the pullback through the activation
  float* dpsd = io.out(d_ps, np);
  float* dxd = io.out(d_x, nx);
  DevBuf pre(ctx, a != ACT_IDENTITY ? ny : 1);
  DevBuf pack(ctx, nw), packT(ctx, nw), ydummy(ctx, a != ACT_IDENTITY ? ny : 1);
  if (a != ACT_IDENTITY) {   // recompute the pre-activation, then delta = d_y * act'(pre)
    conv_pack_kernel<<<lr_ew_blocks(nw), 256, 0, st>>>(psd, in_ch, out_ch, 0, 0, pack.p);
    LR_COUNT(ctx);
    ConvP q;
    memset(&q, 0, sizeof(q));
    q.X = xd; q.Wp = pack.p; q.Wd = width; q.Ht = height; q.Cin = in_ch; q.Cout = out_ch; q.Y = ydummy.p; q.out_scale = 1.0f;
    q.bias = use_bias ? psd + nw : nullptr; q.out_act = ACT_IDENTITY; q.pre = pre.p;
    convops::launch_conv(ctx, q, B);
    bn_bwd_apply_kernel<<<lr_ew_blocks(ny), 256, 0, st>>>(dg, pre.p, nullptr, nullptr, nullptr, a, out_ch, HW, ny, nullptr);
    LR_COUNT(ctx);
  }
  // weight gradient (split over the batch, fixed-order reduce) and bias gradient
  {
    const bool swapped = out_ch <= 16 && in_ch > out_ch;
    const int pt = swapped ? out_ch : in_ch, qt = swapped ? in_ch : out_ch;
    const int chunks = (pt + 15) / 16, cic = (pt + chunks - 1) / chunks, nqb = (qt + 63) / 64;
    int S = std::max(1, std::min((int)B, (4 * 148) / (chunks * nqb)));
    const int img = (int)((B + S - 1) / S);
    S = (int)((B + img - 1) / img);
    DevBuf part(ctx, (size_t)S * nw);
    ConvWgP w;
    memset(&w, 0, sizeof(w));
    ConvWgOp ox, od;
    memset(&ox, 0, sizeof(ox)); memset(&od, 0, sizeof(od));
    ox.ptr = xd; ox.act = ACT_IDENTITY; ox.C = in_ch; ox.td = 0;
    od.ptr = dg; od.act = ACT_IDENTITY; od.C = out_ch; od.td = 0;
    w.swapped = swapped ? 1 : 0;
    w.P = swapped ? od : ox; w.Q = swapped ? ox : od;
    w.Wd = width; w.Ht = height; w.B = (int)B; w.CinTot = in_ch; w.Cout = out_ch;
    w.pcc = cic; w.img_per_split = img; w.part = part.p; w.block = nw;
    conv3x3_wgrad_kernel<<<dim3(chunks, S, nqb), 256, 0, st>>>(w);
    LR_COUNT(ctx);
    wgrad_reduce_kernel<<<lr_ew_blocks(nw), 256, 0, st>>>(part.p, S, nw, dpsd, nullptr, 0, 1.0f, 0.0f, nullptr);
    LR_COUNT(ctx);
    if (use_bias) {
      channel_sum_kernel<<<out_ch, 256, 0, st>>>(dg, out_ch, HW, (int)B, dpsd + nw);
      LR_COUNT(ctx);
    }
  }
  if (d_x) {
    conv_pack_kernel<<<lr_ew_blocks(nw), 256, 0, st>>>(psd, in_ch, out_ch, 1, in_ch, packT.p);
    LR_COUNT(ctx);
    ConvP q;
    memset(&q, 0, sizeof(q));
    q.X = dg; q.Wp = packT.p; q.Wd = width; q.Ht = height; q.Cin = out_ch; q.Cout = in_ch; q.Y = dxd; q.out_scale = 1.0f;
    convops::launch_conv(ctx, q, B);
  }
  LR_CHECK_LAUNCH();
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  LR_API_END
}

namespace convops {
// per-channel scale / shift of x (batch statistics, or the running ones in testmode) -> ab, stat
static void bn_statistics(lrnde_ctx* ctx, int C, size_t HW, int64_t B, const float* psd, const float* xd, float* state,
                          int testmode, int update, float* ab, float* stat) {
  cudaStream_t st = ctx->stream;
  int S = (int)std::max<int64_t>(1, std::min<int64_t>(B, 16));
  const int img = (int)((B + S - 1) / S);
  S = (int)((B + img - 1) / img);
  DevBuf part(ctx, 2 * (size_t)S * C);
  if (!testmode) {
    bn_stats_kernel<<<dim3(C, S), 256, 0, st>>>(xd, C, HW, (int)B, img, (float2*)part.p);
    LR_COUNT(ctx);
  }
  bn_finalize_kernel<<<C, 128, 0, st>>>((const float2*)part.p, S, C, (double)HW * (double)B, psd, 1e-5f, ab, stat, state,
                                        testmode, update, nullptr, ctx->bn_dist());
  LR_COUNT(ctx);
}
}  // namespace convops

extern "C" int lrnde_batchnorm_forward(lrnde_ctx* ctx, int32_t C, int64_t HW, int32_t act, const float* ps, const float* x,
                                       int64_t B, float* state, int32_t testmode, int32_t host_buffers, float* y) {
  LR_API_BEGIN
  if (!ctx || !ps || !x || !y || C < 1 || HW < 1 || B < 1) lr_fail(LRNDE_EINVAL, "lrnde_batchnorm_forward: bad args");
  if (ctx->nranks > 1 && C > LR_BN_MAXC) lr_fail(LRNDE_EINVAL, "BatchNorm with %d channels on a multi-rank ctx (max %d)", C, LR_BN_MAXC);
  if (testmode && !state) lr_fail(LRNDE_EINVAL, "lrnde_batchnorm_forward: testmode needs the running statistics");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t n = (size_t)HW * C * B;
  CallerBufs io(ctx, host_buffers);
  const float* psd = io.in(ps, 2 * (size_t)C);
  const float* xd = io.in(x, n);
  float* yd = io.out(y, n);
  // running statistics: read in testmode, else updated and returned
  float* sd = testmode ? const_cast<float*>(io.in(state, 2 * (size_t)C)) : io.inout(state, 2 * (size_t)C);
  DevBuf ab(ctx, 2 * C), stat(ctx, 2 * C);
  convops::bn_statistics(ctx, C, (size_t)HW, B, psd, xd, sd, testmode, 1, ab.p, stat.p);
  bn_apply_kernel<<<lr_ew_blocks(n), 256, 0, st>>>(xd, ab.p, lr_map_act(act), C, (size_t)HW, n, yd);
  LR_COUNT(ctx);
  LR_CHECK_LAUNCH();
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  ctx->bn_check();
  LR_API_END
}

extern "C" int lrnde_batchnorm_backward(lrnde_ctx* ctx, int32_t C, int64_t HW, int32_t act, const float* ps, const float* x,
                                        const float* d_y, int64_t B, const float* state, int32_t testmode,
                                        int32_t host_buffers, float* d_x, float* d_ps) {
  LR_API_BEGIN
  if (!ctx || !ps || !x || !d_y || !d_x || !d_ps || C < 1 || HW < 1 || B < 1)
    lr_fail(LRNDE_EINVAL, "lrnde_batchnorm_backward: bad args");
  if (testmode && !state) lr_fail(LRNDE_EINVAL, "lrnde_batchnorm_backward: testmode needs the running statistics");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int a = lr_map_act(act);
  const size_t n = (size_t)HW * C * B;
  CallerBufs io(ctx, host_buffers);
  const float* psd = io.in(ps, 2 * (size_t)C);
  const float* xd = io.in(x, n);
  const float* sd = io.in(state, 2 * (size_t)C);
  float* gd = io.out(d_x, n);   // the pullback is formed in place over a copy of d_y
  io.copy_in(gd, d_y, n);
  float* dgbd = io.out(d_ps, 2 * (size_t)C);
  DevBuf ab(ctx, 2 * C), stat(ctx, 2 * C), coef(ctx, 2 * C);
  convops::bn_statistics(ctx, C, (size_t)HW, B, psd, xd, const_cast<float*>(sd), testmode, 0, ab.p, stat.p);
  int S = (int)std::max<int64_t>(1, std::min<int64_t>(B, 16));
  const int img = (int)((B + S - 1) / S);
  S = (int)((B + img - 1) / img);
  DevBuf bpart(ctx, 4 * (size_t)C * S);
  bn_bwd_stats_kernel<<<dim3(C, S), 256, 0, st>>>(gd, xd, ab.p, stat.p, a, C, (size_t)HW, (int)B, img, (double2*)bpart.p, nullptr);
  LR_COUNT(ctx);
  bn_bwd_finalize_kernel<<<(C + 63) / 64, 64, 0, st>>>((const double2*)bpart.p, S, C, (double)HW * (double)B, coef.p, dgbd,
                                                     testmode, nullptr, ctx->bn_dist());
  LR_COUNT(ctx);
  bn_bwd_apply_kernel<<<lr_ew_blocks(n), 256, 0, st>>>(gd, xd, ab.p, stat.p, coef.p, a, C, (size_t)HW, n, nullptr);
  LR_COUNT(ctx);
  LR_CHECK_LAUNCH();
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  ctx->bn_check();
  LR_API_END
}
