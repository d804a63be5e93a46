// Included at the end of lrnde_api.cu (single translation unit):
//   * lrnde_sosri_step  -- _perform_step(::FourStageSRIConstantCache), src/perform_step.jl:49-106
//   * lrnde_head_ce     -- classifier Dense + logitcrossentropy (experiments/src/construct.jl:199,
//                          experiments/src/utils.jl:88) with its gradients (SURVEY 8f, row n1)
//   * lrnde_ipc_*       -- CUDA IPC plumbing for the data-parallel mailboxes
#pragma once

// SOSRI coefficients (StochasticDiffEq FourStageSRIConstantCache; SURVEY App. A.6)
struct SosriTab {
  float a021, a031, a032, a041, a042, a043, a121, a131, a132, a141, a142, a143;
  float b021, b031, b032, b041, b042, b043, b121, b131, b132, b141, b142, b143;
  float al1, al2, al3, al4, c02, c03, c04, c11, c12, c13, c14;
  float be11, be12, be13, be14, be21, be22, be23, be24, be31, be32, be33, be34, be41, be42,
      be43, be44;
};
static SosriTab lr_sosri_tab() {
  SosriTab c;
  c.a021 = -0.04199224421316468f; c.a031 = 2.842612915017106f; c.a032 = -2.0527723684000727f;
  c.a041 = 4.338237071435815f; c.a042 = -2.8895936137439793f; c.a043 = 2.3017575594644466f;
  c.a121 = 0.26204282091330466f; c.a131 = 0.20903646383505375f; c.a132 = -0.1502377115150361f;
  c.a141 = 0.05836595312746999f; c.a142 = 0.6149440396332373f; c.a143 = 0.08535117634046772f;
  c.b021 = -0.21641093549612528f; c.b031 = 1.5336352863679572f; c.b032 = 0.26066223492647056f;
  c.b041 = -1.0536037558179159f; c.b042 = 1.7015284721089472f; c.b043 = -0.20725685784180017f;
  c.b121 = -0.5119011827621657f; c.b131 = 2.67767339866713f; c.b132 = -4.9395031322250995f;
  c.b141 = 0.15580956238299215f; c.b142 = 3.2361551006624674f; c.b143 = -1.4223118283355949f;
  c.al1 = 1.140099274172029f; c.al2 = -0.6401334255743456f; c.al3 = 0.4736296532772559f;
  c.al4 = 0.026404498125060714f;
  c.c02 = -0.04199224421316468f; c.c03 = 0.7898405466170333f; c.c04 = 3.7504010171562823f;
  c.c11 = 0.0f; c.c12 = 0.26204282091330466f; c.c13 = 0.05879875232001766f; c.c14 = 0.758661169101175f;
  c.be11 = -1.8453464565104432f; c.be12 = 2.688764531100726f; c.be13 = -0.2523866501071323f;
  c.be14 = 0.40896857551684956f;
  c.be21 = 0.4969658141589478f; c.be22 = -0.5771202869753592f; c.be23 = -0.12919702470322217f;
  c.be24 = 0.2093514975196336f;
  c.be31 = 2.8453464565104425f; c.be32 = -2.688764531100725f; c.be33 = 0.2523866501071322f;
  c.be34 = -0.40896857551684945f;
  c.be41 = 0.11522663875443433f; c.be42 = -0.57877086147738f; c.be43 = 0.2857851028163886f;
  c.be44 = 0.17775911990655704f;
  return c;
}

struct SosriP {
  SosriTab c;
  const float* uprev; const float* dW; const float* dZ;
  float* k[4]; float* g[4]; float* H0; float* H1; float* u;
  float t, dt, sqdt, abstol, reltol, delta;
  size_t n;
  double* partials;
};

__device__ __forceinline__ float sosri_chi2(const SosriP& p, size_t i) {
  return (p.dW[i] + p.dZ[i] / sqrtf(3.0f)) / 2.0f;
}

// stage = 1..3: H0_stage / H1_stage from k1..k_stage, g1..g_stage (perform_step.jl:65-82)
__global__ void __launch_bounds__(256) sosri_stage_kernel(SosriP p, int stage) {
  const SosriTab& c = p.c;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < p.n;
       i += (size_t)gridDim.x * blockDim.x) {
    float chi2 = sosri_chi2(p, i), up = p.uprev[i];
    float h0, h1;
    if (stage == 1) {
      h0 = up + p.dt * c.a021 * p.k[0][i] + c.b021 * chi2 * p.g[0][i];
      h1 = up + p.dt * c.a121 * p.k[0][i] + p.sqdt * c.b121 * p.g[0][i];
    } else if (stage == 2) {
      h0 = up + p.dt * (c.a031 * p.k[0][i] + c.a032 * p.k[1][i]) +
           chi2 * (c.b031 * p.g[0][i] + c.b032 * p.g[1][i]);
      h1 = up + p.dt * (c.a131 * p.k[0][i] + c.a132 * p.k[1][i]) +
           p.sqdt * (c.b131 * p.g[0][i] + c.b132 * p.g[1][i]);
    } else {
      h0 = up + p.dt * (c.a041 * p.k[0][i] + c.a042 * p.k[1][i] + c.a043 * p.k[2][i]) +
           chi2 * (c.b041 * p.g[0][i] + c.b042 * p.g[1][i] + c.b043 * p.g[2][i]);
      h1 = up + p.dt * (c.a141 * p.k[0][i] + c.a142 * p.k[1][i] + c.a143 * p.k[2][i]) +
           p.sqdt * (c.b141 * p.g[0][i] + c.b142 * p.g[1][i] + c.b143 * p.g[2][i]);
    }
    p.H0[i] = h0;
    p.H1[i] = h1;
  }
}

// u, E1, E2 and the partial sums of the scaled residual (perform_step.jl:87-103)
__global__ void __launch_bounds__(256) sosri_final_kernel(SosriP p) {
  const SosriTab& c = p.c;
  double acc = 0.0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < p.n;
       i += (size_t)gridDim.x * blockDim.x) {
    float dW = p.dW[i], up = p.uprev[i];
    float chi1 = (dW * dW - fabsf(p.dt)) / (2.0f * p.sqdt);
    float chi2 = sosri_chi2(p, i);
    float chi3 = (dW * dW * dW - 3.0f * dW * p.dt) / (6.0f * p.dt);
    float k1 = p.k[0][i], k2 = p.k[1][i], k3 = p.k[2][i], k4 = p.k[3][i];
    float g1 = p.g[0][i], g2 = p.g[1][i], g3 = p.g[2][i], g4 = p.g[3][i];
    float E2 = chi2 * (c.be31 * g1 + c.be32 * g2 + c.be33 * g3 + c.be34 * g4) +
               chi3 * (c.be41 * g1 + c.be42 * g2 + c.be43 * g3 + c.be44 * g4);
    float u = up + p.dt * (c.al1 * k1 + c.al2 * k2 + c.al3 * k3 + c.al4 * k4) + E2 +
              dW * (c.be11 * g1 + c.be12 * g2 + c.be13 * g3 + c.be14 * g4) +
              chi1 * (c.be21 * g1 + c.be22 * g2 + c.be23 * g3 + c.be24 * g4);
    float E1 = p.dt * (k1 + k2 + k3 + k4);
    float r = (p.delta * E1 + E2) / (p.abstol + fmaxf(fabsf(up), fabsf(u)) * p.reltol);
    p.u[i] = u;
    acc += (double)(r * r);
  }
  double s = lr_block_sum(acc);
  if (threadIdx.x == 0) p.partials[blockIdx.x] = s;
}

__global__ void sosri_finish_kernel(const double* partials, double n, float dt, float* out) {
  double s = lr_sum_partials(partials);
  if (threadIdx.x == 0) out[0] = sqrtf((float)s / (float)n) * dt;
}

extern "C" int lrnde_sosri_step(lrnde_ctx* ctx, const lrnde_model* drift,
                                const lrnde_model* diffusion, const lrnde_opts* o,
                                const float* ps_drift, const float* ps_diffusion,
                                const float* uprev, const float* dW, const float* dZ, float t,
                                float dt, float delta, int64_t B, float* u, float* reg_val) {
  LR_API_BEGIN
  if (!ctx || !drift || !diffusion || !o || !ps_drift || !ps_diffusion || !uprev || !dW || !dZ ||
      !u || !reg_val || B < 1)
    lr_fail(LRNDE_EINVAL, "lrnde_sosri_step: bad args");
  if (drift->D != diffusion->D) lr_fail(LRNDE_EINVAL, "drift and diffusion state dims differ");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t DB = (size_t)drift->D * B;
  // owned copies throughout: the inputs sit together in one pooled buffer, u is a slice of the work buffer
  CallerBufs io(ctx, o->host_buffers);
  const float* psd = io.copy_in(ps_drift, drift->nparams);
  const float* psg = io.copy_in(ps_diffusion, diffusion->nparams);
  DevBuf in(ctx, 3 * DB), work(ctx, 11 * DB);
  DevBuf descs(ctx, 8 * (sizeof(LinComb) / 4 + 1));
  DevBuf red(ctx, 2 * LR_ERR_BLOCKS + 8);
  io.copy_in(in.p, uprev, DB);
  io.copy_in(in.p + DB, dW, DB);
  io.copy_in(in.p + 2 * DB, dZ, DB);
  SosriP p;
  p.c = lr_sosri_tab();
  p.uprev = in.p; p.dW = in.p + DB; p.dZ = in.p + 2 * DB;
  for (int i = 0; i < 4; ++i) { p.k[i] = work.p + (size_t)i * DB; p.g[i] = work.p + (size_t)(4 + i) * DB; }
  p.H0 = work.p + 8 * DB; p.H1 = work.p + 9 * DB; p.u = work.p + 10 * DB;
  p.t = t; p.dt = dt; p.sqdt = sqrtf(fabsf(dt)); p.abstol = o->abstol; p.reltol = o->reltol;
  p.delta = delta; p.n = DB; p.partials = (double*)red.p;
  const float c0[4] = {0.0f, p.c.c02, p.c.c03, p.c.c04};
  const float c1[4] = {p.c.c11, p.c.c12, p.c.c13, p.c.c14};
  std::vector<LinComb> hd(8);
  for (int s = 0; s < 4; ++s) {
    memset(&hd[2 * s], 0, sizeof(LinComb));
    memset(&hd[2 * s + 1], 0, sizeof(LinComb));
    hd[2 * s].base = (s == 0) ? p.uprev : p.H0;
    hd[2 * s].t = t + c0[s] * dt;
    hd[2 * s].dst = p.k[s];
    hd[2 * s + 1].base = (s == 0) ? p.uprev : p.H1;
    hd[2 * s + 1].t = t + c1[s] * dt;
    hd[2 * s + 1].dst = p.g[s];
  }
  LR_CUDA(cudaMemcpyAsync(descs.p, hd.data(), sizeof(LinComb) * 8, cudaMemcpyHostToDevice, st));
  const LinComb* dd = (const LinComb*)descs.p;
  MlpEval evf(ctx, drift, psd, B, lr_ode_route(ctx, drift, o, B), false);
  MlpEval evg(ctx, diffusion, psg, B, lr_ode_route(ctx, diffusion, o, B), false);
  evf.prepare();
  evg.prepare();
  for (int s = 0; s < 4; ++s) {
    if (s > 0) {
      sosri_stage_kernel<<<lr_ew_blocks(DB), 256, 0, st>>>(p, s);
      LR_COUNT(ctx);
    }
    evf.forward(dd + 2 * s, nullptr);
    evg.forward(dd + 2 * s + 1, nullptr);
  }
  sosri_final_kernel<<<LR_ERR_BLOCKS, 256, 0, st>>>(p);
  LR_COUNT(ctx);
  float* out_scalar = (float*)(p.partials + LR_ERR_BLOCKS);
  sosri_finish_kernel<<<1, 32, 0, st>>>(p.partials, (double)DB, dt, out_scalar);
  LR_COUNT(ctx);
  LR_CHECK_LAUNCH();
  io.copy_out(u, p.u, DB);
  io.finish();
  LR_CUDA(cudaMemcpyAsync(reg_val, out_scalar, 4, cudaMemcpyDeviceToHost, st));
  LR_CUDA(cudaStreamSynchronize(st));
  LR_API_END
}

// ------------------------------------------------------------------------------------------
// classifier head + logitcrossentropy:  loss = mean_b( -log softmax(W u_b + b)[y_b] )
// ------------------------------------------------------------------------------------------
__global__ void softmax_ce_kernel(const float* logits, const int* labels, int Cn, int B,
                                  float* dlogits, double* partials, int* bad_label) {
  double acc = 0.0;
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    const float* z = logits + (size_t)b * Cn;
    float mx = z[0];
    for (int c = 1; c < Cn; ++c) mx = fmaxf(mx, z[c]);
    float s = 0.0f;
    for (int c = 0; c < Cn; ++c) s += expf(z[c] - mx);
    float lse = mx + logf(s);
    int y = labels[b];
    if (y < 0 || y >= Cn) { *bad_label = 1; y = 0; }   // reported as LRNDE_EINVAL by the caller (labels are 0-based)
    acc += (double)(lse - z[y]);
    for (int c = 0; c < Cn; ++c)
      dlogits[(size_t)b * Cn + c] = (expf(z[c] - lse) - (c == y ? 1.0f : 0.0f)) / (float)B;
  }
  double r = lr_block_sum(acc);
  if (threadIdx.x == 0) partials[blockIdx.x] = r;
}
// Fused head for small class counts (Cn <= 16): one warp per sample reads u_b once, forms the Cn logits (weights in
// shared memory), the cross entropy, dlogits (kept for the weight gradient) and d_u[:, b] = W^T dlogits[:, b].
// Same arithmetic as dense_nn_kernel + softmax_ce_kernel + dense_nn_kernel, in 2 * 4 * D * B bytes of traffic.
constexpr int kHeadMaxC = 16;
__global__ void __launch_bounds__(256) head_fused_kernel(const float* __restrict__ Wc, const float* __restrict__ u,
                                                         const int* __restrict__ labels, int Cn, int D, int B,
                                                         float* __restrict__ dlogits, float* __restrict__ d_u,
                                                         double* partials, int* bad_label) {
  extern __shared__ float hw[];                 // W [Cn x D] column-major (as in ps), then the bias [Cn]
  for (int i = threadIdx.x; i < Cn * (D + 1); i += blockDim.x) hw[i] = Wc[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  double acc = 0.0;
  for (int b = blockIdx.x * nwarp + warp; b < B; b += gridDim.x * nwarp) {
    const float* ub = u + (size_t)b * D;
    float z[kHeadMaxC];
#pragma unroll
    for (int c = 0; c < kHeadMaxC; ++c) z[c] = 0.0f;
    for (int d = lane; d < D; d += 32) {
      const float x = __ldcg(ub + d);
#pragma unroll
      for (int c = 0; c < kHeadMaxC; ++c)
        if (c < Cn) z[c] = fmaf(hw[c + d * Cn], x, z[c]);
    }
#pragma unroll
    for (int c = 0; c < kHeadMaxC; ++c) {
      if (c < Cn) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) z[c] += __shfl_xor_sync(0xffffffffu, z[c], o);
        z[c] += hw[Cn * D + c];
      }
    }
    float mx = z[0];
#pragma unroll
    for (int c = 1; c < kHeadMaxC; ++c) if (c < Cn) mx = fmaxf(mx, z[c]);
    float sum = 0.0f;
#pragma unroll
    for (int c = 0; c < kHeadMaxC; ++c) if (c < Cn) sum += expf(z[c] - mx);
    const float lse = mx + logf(sum);
    int y = labels[b];
    if (y < 0 || y >= Cn) { if (lane == 0) *bad_label = 1; y = 0; }
    float zy = 0.0f;
    float dl[kHeadMaxC];
#pragma unroll
    for (int c = 0; c < kHeadMaxC; ++c) {
      dl[c] = 0.0f;
      if (c < Cn) {
        if (c == y) zy = z[c];
        dl[c] = (expf(z[c] - lse) - (c == y ? 1.0f : 0.0f)) / (float)B;
      }
    }
    if (lane == 0) {
      acc += (double)(lse - zy);
      for (int c = 0; c < Cn; ++c) dlogits[(size_t)b * Cn + c] = dl[c];
    }
    if (d_u) {
      float* out = d_u + (size_t)b * D;
      for (int d = lane; d < D; d += 32) {
        float v = 0.0f;
#pragma unroll
        for (int c = 0; c < kHeadMaxC; ++c)
          if (c < Cn) v = fmaf(hw[c + d * Cn], dl[c], v);
        out[d] = v;
      }
    }
  }
  double r = lr_block_sum(acc);
  if (threadIdx.x == 0) partials[blockIdx.x] = r;
}
__global__ void mean_finish_kernel(const double* partials, int nb, double n, float* out) {
  double s = 0.0;
  for (int i = threadIdx.x; i < nb; i += 32) s += partials[i];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if (threadIdx.x == 0) out[0] = (float)(s / n);
}

extern "C" int lrnde_head_ce(lrnde_ctx* ctx, const float* Wc, const float* u,
                             const int32_t* labels, int64_t B, int32_t D, int32_t Cn,
                             int32_t host_buffers, float* loss, float* d_u, float* d_Wc) {
  LR_API_BEGIN
  if (!ctx || !Wc || !u || !labels || !loss || B < 1 || D < 1 || Cn < 1)
    lr_fail(LRNDE_EINVAL, "lrnde_head_ce: bad args");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t DB = (size_t)D * B, CB = (size_t)Cn * B, PW = (size_t)Cn * (D + 1);
  DevBuf logits(ctx, CB), dlog(ctx, CB), wt(ctx, (size_t)D * Cn);
  const int nb = 296;
  DevBuf red(ctx, 2 * nb + 8);
  int* badd = (int*)(red.p + 2 * nb + 4);
  LR_CUDA(cudaMemsetAsync(badd, 0, sizeof(int), st));
  CallerBufs io(ctx, host_buffers);
  const float* Wd = io.in(Wc, PW);
  const float* ud = io.in(u, DB);
  const int* ld = io.in(labels, (size_t)B);
  float* dud = io.out(d_u, DB);
  float* dWd = io.out(d_Wc, PW);
  const size_t head_smem = sizeof(float) * (size_t)Cn * (D + 1);
  const bool fused_head = Cn <= kHeadMaxC && head_smem <= 160 * 1024 && !getenv("LRNDE_NO_FUSED_HEAD");
  float* lossd = (float*)((double*)red.p + nb);
  if (fused_head) {
    static size_t attr_bytes = 0;
    if (head_smem > attr_bytes) {
      LR_CUDA(cudaFuncSetAttribute(head_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)head_smem));
      attr_bytes = head_smem;
    }
    LR_CUDA(cudaMemsetAsync(red.p, 0, sizeof(double) * nb, st));
    const int hb = (int)std::min<int64_t>(nb, (B + 7) / 8);   // at most nb blocks (the partial sums), 8 warps each
    head_fused_kernel<<<hb, 256, head_smem, st>>>(Wd, ud, ld, Cn, D, (int)B, dlog.p, dud, (double*)red.p, badd);
    LR_COUNT(ctx);
    mean_finish_kernel<<<1, 32, 0, st>>>((double*)red.p, nb, (double)B, lossd);
    LR_COUNT(ctx);
  } else {
  DenseP p;
  memset(&p, 0, sizeof(p));
  p.A = Wd; p.lda = Cn; p.M = Cn; p.K = D; p.td = 0; p.bias = 1;
  p.X = ud; p.ldx = D; p.N = (int)B; p.Y = logits.p; p.ldy = Cn; p.act = ACT_IDENTITY; p.dact = -1;
  p.out_scale = 1.0f;
  dim3 g((Cn + DN_BM - 1) / DN_BM, (unsigned)((B + DN_BN - 1) / DN_BN));
  dense_nn_kernel<<<g, 256, 0, st>>>(p);
  LR_COUNT(ctx);
  softmax_ce_kernel<<<nb, 256, 0, st>>>(logits.p, ld, Cn, (int)B, dlog.p, (double*)red.p, badd);
  LR_COUNT(ctx);
  mean_finish_kernel<<<1, 32, 0, st>>>((double*)red.p, nb, (double)B, lossd);
  LR_COUNT(ctx);
  }
  if (d_u && !fused_head) {
    dim3 tg((Cn + 31) / 32, (D + 31) / 32), tb(32, 8);
    transpose_kernel<<<tg, tb, 0, st>>>(Wd, Cn, D, wt.p);
    LR_COUNT(ctx);
    DenseP q;
    memset(&q, 0, sizeof(q));
    q.A = wt.p; q.lda = D; q.M = D; q.K = Cn; q.X = dlog.p; q.ldx = Cn; q.N = (int)B;
    q.Y = dud; q.ldy = D; q.act = ACT_IDENTITY; q.dact = -1; q.out_scale = 1.0f;
    dim3 g2((D + DN_BM - 1) / DN_BM, (unsigned)((B + DN_BN - 1) / DN_BN));
    dense_nn_kernel<<<g2, 256, 0, st>>>(q);
    LR_COUNT(ctx);
  }
  if (d_Wc) {
    const int naug = D + 1;
    int tiles = ((Cn + DN_BM - 1) / DN_BM) * ((naug + DN_BN - 1) / DN_BN);
    int S = std::max(1, std::min(64, (2 * 148 + tiles - 1) / tiles));
    int chunk = (int)((B + S - 1) / S);
    chunk = std::max(16, ((chunk + 15) / 16) * 16);
    S = (int)((B + chunk - 1) / chunk);
    DevBuf part(ctx, (size_t)S * PW);
    WgradP wg;
    memset(&wg, 0, sizeof(wg));
    wg.Dl = dlog.p; wg.ldd = Cn; wg.M = Cn; wg.X = ud; wg.ldx = D; wg.Nin = D; wg.td = 0; wg.bias = 1;
    wg.B = (int)B; wg.chunk = chunk; wg.part = part.p;
    dim3 g3((Cn + DN_BM - 1) / DN_BM, (naug + DN_BN - 1) / DN_BN, S);
    wgrad_nt_kernel<<<g3, 256, 0, st>>>(wg);
    LR_COUNT(ctx);
    wgrad_reduce_kernel<<<lr_ew_blocks(PW), 256, 0, st>>>(part.p, S, PW, dWd, nullptr, 0, 1.0f, 0.0f, nullptr);
    LR_COUNT(ctx);
    LR_CHECK_LAUNCH();
    LR_CUDA(cudaStreamSynchronize(st));
  }
  LR_CHECK_LAUNCH();
  io.finish();
  int bad_host = 0;
  LR_CUDA(cudaMemcpyAsync(loss, lossd, 4, cudaMemcpyDeviceToHost, st));
  LR_CUDA(cudaMemcpyAsync(&bad_host, badd, sizeof(int), cudaMemcpyDeviceToHost, st));
  LR_CUDA(cudaStreamSynchronize(st));
  if (bad_host) lr_fail(LRNDE_EINVAL, "lrnde_head_ce: a label is outside [0, %d) (labels are 0-based class indices)", Cn);
  LR_API_END
}

// ------------------------------------------------------------------------------------------
// CUDA IPC plumbing (one process per GPU)
// ------------------------------------------------------------------------------------------
extern "C" int lrnde_ipc_export(lrnde_ctx* ctx, void* dev_ptr, void* handle64) {
  LR_API_BEGIN
  if (!ctx || !dev_ptr || !handle64) lr_fail(LRNDE_EINVAL, "lrnde_ipc_export: bad args");
  LR_CUDA(cudaSetDevice(ctx->device));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  cudaIpcMemHandle_t h;
  LR_CUDA(cudaIpcGetMemHandle(&h, dev_ptr));
  memcpy(handle64, &h, 64);
  LR_API_END
}
extern "C" int lrnde_ipc_open(lrnde_ctx* ctx, const void* handle64, void** dev_ptr) {
  LR_API_BEGIN
  if (!ctx || !handle64 || !dev_ptr) lr_fail(LRNDE_EINVAL, "lrnde_ipc_open: bad args");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  LR_CUDA(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  LR_API_END
}

// ------------------------------------------------------------------------------------------
// Adam (Optimisers.jl semantics: experiments/src/construct.jl:104-152 builds Adam(lr); the
// update is m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2; p -= lr * mhat / (sqrt(vhat) + eps))
// ------------------------------------------------------------------------------------------
__global__ void adam_kernel(float* p, const float* g, float* m, float* v, size_t n, float lr,
                            float b1, float b2, float eps, float c1, float c2) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    float gi = g[i];
    float mi = b1 * m[i] + (1.0f - b1) * gi;
    float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    p[i] -= lr * (mi / c1) / (sqrtf(vi / c2) + eps);
  }
}
extern "C" int lrnde_adam_step(lrnde_ctx* ctx, float* p, const float* g, float* m, float* v,
                               int64_t n, float lr, float beta1, float beta2, float eps,
                               int32_t step) {
  LR_API_BEGIN
  if (!ctx || !p || !g || !m || !v || n < 1 || step < 1) lr_fail(LRNDE_EINVAL, "lrnde_adam_step: bad args");
  LR_CUDA(cudaSetDevice(ctx->device));
  float c1 = 1.0f - powf(beta1, (float)step), c2 = 1.0f - powf(beta2, (float)step);
  adam_kernel<<<lr_ew_blocks((size_t)n), 256, 0, ctx->stream>>>(p, g, m, v, (size_t)n, lr, beta1, beta2,
                                                                 eps, c1, c2);
  LR_COUNT(ctx);
  LR_CHECK_LAUNCH();
  LR_API_END
}

// ------------------------------------------------------------------------------------------
// The other optimisers experiments/src/construct.jl:104-125 can build (Optimisers.jl rules): Descent, Momentum,
// Nesterov, Adam / AdamW (= Adam chained with WeightDecay(0)), AdaMax, each optionally chained with
// WeightDecay(wd) (OptimiserChain(opt, WeightDecay(wd)): the decay term wd * p is added to the rule's update,
// not scaled by the learning rate).  s1 / s2: state buffers (momentum / first moment; second moment / inf-norm).
// ------------------------------------------------------------------------------------------
__global__ void opt_kernel(int kind, float* p, const float* g, float* s1, float* s2, size_t n, float lr, float a,
                           float b, float eps, float wd, float c1, float c2) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float gi = g[i], pi = p[i];
    float dx;
    if (kind == LRNDE_OPT_DESCENT) dx = lr * gi;
    else if (kind == LRNDE_OPT_MOMENTUM) { const float v = a * s1[i] + lr * gi; s1[i] = v; dx = v; }
    else if (kind == LRNDE_OPT_NESTEROV) {
      const float v = s1[i];
      dx = -(a * a) * v + (1.0f + a) * lr * gi;
      s1[i] = a * v - lr * gi;
    } else if (kind == LRNDE_OPT_ADAMAX) {
      const float m = a * s1[i] + (1.0f - a) * gi;
      const float u = fmaxf(b * s2[i], fabsf(gi));
      s1[i] = m; s2[i] = u;
      dx = (lr / c1) * m / (u + eps);
    } else {   // LRNDE_OPT_ADAM
      const float m = a * s1[i] + (1.0f - a) * gi;
      const float v = b * s2[i] + (1.0f - b) * gi * gi;
      s1[i] = m; s2[i] = v;
      dx = lr * (m / c1) / (sqrtf(v / c2) + eps);
    }
    p[i] = pi - (dx + wd * pi);
  }
}
extern "C" int lrnde_opt_step(lrnde_ctx* ctx, int32_t kind, float* p, const float* g, float* s1, float* s2, int64_t n,
                              float lr, float a, float b, float eps, float weight_decay, int32_t step) {
  LR_API_BEGIN
  if (!ctx || !p || !g || n < 1 || step < 1) lr_fail(LRNDE_EINVAL, "lrnde_opt_step: bad args");
  if (kind < LRNDE_OPT_DESCENT || kind > LRNDE_OPT_ADAMAX) lr_fail(LRNDE_EINVAL, "lrnde_opt_step: unknown optimiser %d", kind);
  if (kind != LRNDE_OPT_DESCENT && !s1) lr_fail(LRNDE_EINVAL, "lrnde_opt_step: the rule needs state buffer s1");
  if ((kind == LRNDE_OPT_ADAM || kind == LRNDE_OPT_ADAMAX) && !s2) lr_fail(LRNDE_EINVAL, "lrnde_opt_step: the rule needs state buffer s2");
  LR_CUDA(cudaSetDevice(ctx->device));
  const float c1 = 1.0f - powf(a, (float)step), c2 = 1.0f - powf(b, (float)step);
  opt_kernel<<<lr_ew_blocks((size_t)n), 256, 0, ctx->stream>>>(kind, p, g, s1, s2, (size_t)n, lr, a, b, eps, weight_decay, c1, c2);
  LR_COUNT(ctx);
  LR_CHECK_LAUNCH();
  LR_API_END
}

// ------------------------------------------------------------------------------------------
// Sum of a device vector over the data-parallel group (the once-per-iteration all-reduce of the parameter
// gradients, SURVEY 8e (2)) through the peer-mapped mailboxes set by lrnde_ctx_set_dist: every rank publishes its
// chunk in its own staging area, raises a flag on every peer, and adds all ranks' chunks in rank order over
// NVLink peer loads -- identical bits on every rank, no host round trip, no NCCL dependency.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ar_publish_kernel(LrMailbox* mine, LrMailbox* const* peers, int rank, int nranks,
                                                         const float* v, size_t n, unsigned long long seq,
                                                         unsigned int* counter) {
  const int par = (int)(seq & 1ull);
  float* stage = lr_mbox_stage(mine, par, 2);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) stage[i] = v[i];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int prev = atomicAdd(counter, 1u);
    if (prev == gridDim.x - 1) {
      *counter = 0;
      __threadfence_system();
      for (int r = 0; r < nranks; ++r) {
        volatile unsigned long long* f = &peers[r]->mflag[par][rank];
        *f = seq + 1;
      }
    }
  }
}
__global__ void __launch_bounds__(256) ar_gather_kernel(LrMailbox* mine, LrMailbox* const* peers, int nranks, float* v,
                                                        size_t n, unsigned long long seq, int* timed_out) {
  const int par = (int)(seq & 1ull);
  if (threadIdx.x == 0) {
    long long spins = 0;
    for (int r = 0; r < nranks; ++r) {
      volatile unsigned long long* f = &mine->mflag[par][r];
      while (*f != seq + 1) {
        __nanosleep(40);
        if (++spins > (1ll << 26)) { *timed_out = 1; break; }
      }
    }
    __threadfence_system();
  }
  __syncthreads();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float s = 0.0f;
    for (int r = 0; r < nranks; ++r) s += ((const volatile float*)lr_mbox_stage(peers[r], par, 2))[i];
    v[i] = s;
  }
}
extern "C" int lrnde_allreduce_sum(lrnde_ctx* ctx, float* v, int64_t n) {
  LR_API_BEGIN
  if (!ctx || !v || n < 0) lr_fail(LRNDE_EINVAL, "lrnde_allreduce_sum: bad args");
  if (ctx->nranks <= 1 || n == 0) return LRNDE_OK;
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  DevBuf aux(ctx, 8 + 2 * LR_MAX_RANKS);
  unsigned int* counter = (unsigned int*)aux.p;
  int* timed_out = (int*)(aux.p + 1);
  LrMailbox** peers = (LrMailbox**)(aux.p + 4);
  LR_CUDA(cudaMemsetAsync(aux.p, 0, 16, st));
  LR_CUDA(cudaMemcpyAsync(peers, ctx->peer_mbox, sizeof(LrMailbox*) * LR_MAX_RANKS, cudaMemcpyHostToDevice, st));
  for (int64_t off = 0; off < n; off += LR_MU_MAX) {
    const size_t cnt = (size_t)std::min<int64_t>(LR_MU_MAX, n - off);
    ar_publish_kernel<<<64, 256, 0, st>>>(ctx->peer_mbox[ctx->rank], peers, ctx->rank, ctx->nranks, v + off, cnt, ctx->mseq, counter);
    LR_COUNT(ctx);
    ar_gather_kernel<<<64, 256, 0, st>>>(ctx->peer_mbox[ctx->rank], peers, ctx->nranks, v + off, cnt, ctx->mseq, timed_out);
    LR_COUNT(ctx);
    ctx->mseq += 1;
  }
  LR_CHECK_LAUNCH();
  int to = 0;
  LR_CUDA(cudaMemcpyAsync(&to, timed_out, sizeof(int), cudaMemcpyDeviceToHost, st));
  LR_CUDA(cudaStreamSynchronize(st));
  if (to) lr_fail(LRNDE_ESTATE, "lrnde_allreduce_sum: a peer rank never published its vector (timed out)");
  LR_API_END
}

// ------------------------------------------------------------------------------------------
// Roofline probe: `iters` back-to-back evaluations of f(u, ps, t) (the unit of work SURVEY 8d
// counts flops for) between two CUDA events on the ctx stream.  Device pointers only.
// ------------------------------------------------------------------------------------------
extern "C" int lrnde_profile_feval(lrnde_ctx* ctx, const lrnde_model* m, const lrnde_opts* o,
                                   const float* ps, const float* u, int64_t B, int32_t iters,
                                   float* du, float* ms_per_eval, int32_t* launches_per_eval) {
  LR_API_BEGIN
  if (!ctx || !m || !ps || !u || !du || !ms_per_eval || B < 1 || iters < 1)
    lr_fail(LRNDE_EINVAL, "lrnde_profile_feval: bad args");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  DevBuf ddesc(ctx, sizeof(LinComb) / 4 + 1);
  LinComb d;
  memset(&d, 0, sizeof(d));
  d.base = u; d.t = 0.5f; d.dst = du;
  // LRNDE_PROFILE_NSRC=n: time the evaluation with an n-source stage combination in the operand
  // prologue (the HBM-bound shape of the later Tsit5 stages) instead of a plain input
  const char* ns_env = getenv("LRNDE_PROFILE_NSRC");
  const int nsrc = ns_env ? std::max(0, std::min(7, atoi(ns_env))) : 0;
  const size_t len = (size_t)m->D * (size_t)B;
  DevBuf srcs(ctx, nsrc ? len * (size_t)nsrc : 1);
  if (nsrc) {
    LR_CUDA(cudaMemsetAsync(srcs.p, 0, len * (size_t)nsrc * sizeof(float), st));
    d.n = nsrc; d.scale = 0.01f;
    for (int i = 0; i < nsrc; ++i) { d.src[i] = srcs.p + (size_t)i * len; d.coef[i] = 0.1f * (float)(i + 1); }
  }
  LR_CUDA(cudaMemcpyAsync(ddesc.p, &d, sizeof(d), cudaMemcpyHostToDevice, st));
  MlpEval ev(ctx, m, ps, B, lr_ode_route(ctx, m, o, B), false);
  ev.prepare();
  // LRNDE_PROFILE_LAYERS=k: only the first k layers (k = 1 isolates the layer-1 kernel with the
  // stage combination in its operand prologue)
  if (const char* nl_env = getenv("LRNDE_PROFILE_LAYERS")) ev.max_layers = std::max(1, atoi(nl_env));
  long l0 = ctx->launches;
  ev.forward((const LinComb*)ddesc.p, nullptr);  // warm
  long per = ctx->launches - l0;
  cudaEvent_t e0, e1;
  LR_CUDA(cudaEventCreate(&e0));
  LR_CUDA(cudaEventCreate(&e1));
  LR_CUDA(cudaEventRecord(e0, st));
  for (int i = 0; i < iters; ++i) ev.forward((const LinComb*)ddesc.p, nullptr);
  LR_CUDA(cudaEventRecord(e1, st));
  LR_CUDA(cudaEventSynchronize(e1));
  float ms = 0.0f;
  LR_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *ms_per_eval = ms / (float)iters;
  if (launches_per_eval) *launches_per_eval = (int32_t)per;
  LR_API_END
}

#ifdef LRNDE_UMMA_TRACE
extern "C" int lrnde_debug_trace(long long* out, int n) {
  cudaMemcpyFromSymbol(out, g_umma_trace, sizeof(long long) * (size_t)n);
  return 0;
}
#endif
