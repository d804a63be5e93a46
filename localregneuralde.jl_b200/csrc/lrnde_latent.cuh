// Latent-ODE encoder (SURVEY 8f, row n2): Recurrence(LatentGRUCell(in, h, latent)) of the physionet config,
//   LatentGRUCell   src/layers/latent_ode.jl:1-48   (quirks kept: new_y_mean is built from new_state_std, :37;
//                                                    the observation mask sums rows F div 2 .. F-1, i.e. the mask
//                                                    rows AND the trailing dt row, :40)
//   Recurrence      experiments/src/construct.jl:231 (cell applied along the time dimension, last output returned)
// and its reverse pass (back-propagation through time w.r.t. the parameters; the inputs are data).
//
// Same B200 mapping as the SDE path (lrnde_sde.cuh): samples are independent, the three gate networks
// (6.6 K .. 17 K parameters) live in shared memory, each CTA walks the whole time series of its tile of
// samples in ONE launch (T sequential cells, no launch per step), the reverse pass accumulates the parameter
// gradients in shared memory and they are reduced in a fixed order.
#pragma once

struct GruP {
  SdeNet nu, nr, nn;  // update gate, reset gate, new state
  const float* ps;
  const float* x;     // [F, T, B] column-major
  int F, T, B, L, S, SP, tiles_per_cta;
  int g_global;       // reverse pass: gradient accumulators in global memory (gpart) instead of shared memory
  float* carry;       // [T][B][2L]: (y_mean, y_std) before step t
  float* y;           // [2L, B]
  const float* d_y;   // [2L, B]
  float* gpart;       // [grid][nu.wfloats + nr.wfloats + nn.wfloats]
};

struct GruBufs {
  float *Wu, *Wr, *Wn, *Gu, *Gr, *Gn;
  float *yc, *c2, *ug, *rg, *ns, *ym, *ys, *mask, *pre, *post;
  float *mb, *sb, *nsb, *ugb, *rgb, *c2b, *ycb, *scr, *dA, *dB;
};

__device__ void gru_carve(float* sm, const GruP& p, bool bwd, GruBufs& b) {
  float* q = sm;
  b.Wu = q; q += p.nu.wfloats; b.Wr = q; q += p.nr.wfloats; b.Wn = q; q += p.nn.wfloats;
  b.Gu = b.Gr = b.Gn = nullptr;
  if (bwd && !p.g_global) { b.Gu = q; q += p.nu.wfloats; b.Gr = q; q += p.nr.wfloats; b.Gn = q; q += p.nn.wfloats; }
  const int SP = p.SP, I = 2 * p.L + p.F, L = p.L;
  auto take = [&](int rows) { float* r = q; q += rows * SP; return r; };
  b.yc = take(I); b.c2 = take(I); b.ug = take(L); b.rg = take(L); b.ns = take(2 * L); b.ym = take(L); b.ys = take(L);
  b.mask = take(1);
  const int hid = max(p.nu.hid_rows, p.nn.hid_rows);
  b.pre = take(hid); b.post = take(hid);
  if (bwd) {
    const int md = max(p.nu.maxdim, p.nn.maxdim);
    b.mb = take(L); b.sb = take(L); b.nsb = take(2 * L); b.ugb = take(L); b.rgb = take(L);
    b.c2b = take(I); b.ycb = take(I); b.scr = take(2 * L); b.dA = take(md); b.dB = take(md);
  }
}
static size_t gru_smem_bytes(const GruP& p, bool bwd) {
  const int I = 2 * p.L + p.F, L = p.L;
  size_t f = (size_t)(p.nu.wfloats + p.nr.wfloats + p.nn.wfloats) * ((bwd && !p.g_global) ? 2 : 1);
  int rows = 2 * I + 6 * L + 1 + 2 * std::max(p.nu.hid_rows, p.nn.hid_rows);
  if (bwd) rows += 8 * L + 2 * I + 2 * std::max(p.nu.maxdim, p.nn.maxdim);
  return (f + (size_t)rows * p.SP) * sizeof(float) + 16;
}

// one cell evaluation on the tile: fills yc, ug, rg, c2, ns, mask from (ym, ys, x_t)
__device__ void gru_cell_fwd(const GruP& p, const GruBufs& b, int t, int b0, const SdeTile& T) {
  const int L = p.L, F = p.F, SP = p.SP;
  for (int idx = T.tid; idx < (2 * L + F) * T.S; idx += T.nthr) {
    const int s = idx / (2 * L + F), r = idx % (2 * L + F);
    float v;
    if (r < L) v = b.ym[r * SP + s];
    else if (r < 2 * L) v = b.ys[(r - L) * SP + s];
    else v = (s < T.nvalid) ? p.x[((size_t)(b0 + s) * p.T + t) * F + (r - 2 * L)] : 0.0f;
    b.yc[r * SP + s] = v;
  }
  __syncthreads();
  if (T.tid < T.S) {   // mask = sum(x[F div 2 + 1 : end]) > 0   (latent_ode.jl:40)
    float acc = 0.0f;
    for (int r = F / 2; r < F; ++r) acc += b.yc[(2 * L + r) * SP + T.tid];
    b.mask[T.tid] = acc > 0.0f ? 1.0f : 0.0f;
  }
  sde_mlp_fwd(p.nu, b.Wu, b.yc, 0.0f, b.ug, b.pre, b.post, T);
  sde_mlp_fwd(p.nr, b.Wr, b.yc, 0.0f, b.rg, b.pre, b.post, T);
  for (int idx = T.tid; idx < (2 * L + F) * T.S; idx += T.nthr) {
    const int s = idx % T.S, r = idx / T.S;
    float v = b.yc[r * SP + s];
    if (r < 2 * L) v *= b.rg[(r < L ? r : r - L) * SP + s];
    b.c2[r * SP + s] = v;
  }
  __syncthreads();
  sde_mlp_fwd(p.nn, b.Wn, b.c2, 0.0f, b.ns, b.pre, b.post, T);
}

__global__ void __launch_bounds__(SDE_THREADS, 1) gru_forward_kernel(GruP p) {
  extern __shared__ __align__(16) float sde_sm[];
  GruBufs b;
  gru_carve(sde_sm, p, false, b);
  const int tid = threadIdx.x, nthr = blockDim.x, L = p.L, SP = p.SP;
  sde_load_weights(p.nu, p.ps, b.Wu, tid, nthr);
  sde_load_weights(p.nr, p.ps, b.Wr, tid, nthr);
  sde_load_weights(p.nn, p.ps, b.Wn, tid, nthr);
  __syncthreads();
  SdeTile T{p.S, SP, L, 0, nthr, tid};
  for (int ti = 0; ti < p.tiles_per_cta; ++ti) {
    const int b0 = (blockIdx.x * p.tiles_per_cta + ti) * p.S;
    if (b0 >= p.B) break;
    T.nvalid = min(p.S, p.B - b0);
    for (int idx = tid; idx < L * T.S; idx += nthr) {   // latent_ode.jl:20-24
      const int a = (idx / T.S) * SP + (idx % T.S);
      b.ym[a] = 0.0f; b.ys[a] = 1.0f;
    }
    __syncthreads();
    for (int t = 0; t < p.T; ++t) {
      if (p.carry)
        for (int idx = tid; idx < 2 * L * T.S; idx += nthr) {
          const int s = idx / (2 * L), j = idx % (2 * L);
          if (s < T.nvalid)
            p.carry[((size_t)t * p.B + b0 + s) * 2 * L + j] = (j < L) ? b.ym[j * SP + s] : b.ys[(j - L) * SP + s];
        }
      gru_cell_fwd(p, b, t, b0, T);
      for (int idx = tid; idx < L * T.S; idx += nthr) {
        const int s = idx % T.S, a = (idx / T.S) * SP + s;
        const float ug = b.ug[a], nss = b.ns[(L + idx / T.S) * SP + s], m = b.mask[s];
        const float ym = b.ym[a], ys = b.ys[a];
        const float nm = (1.0f - ug) * nss + ug * ym;      // :37 (new_state_std on purpose)
        const float nsd = (1.0f - ug) * nss + ug * ys;
        b.ym[a] = m * nm + (1.0f - m) * ym;
        b.ys[a] = m * nsd + (1.0f - m) * ys;
      }
      __syncthreads();
    }
    for (int idx = tid; idx < 2 * L * T.S; idx += nthr) {
      const int s = idx / (2 * L), j = idx % (2 * L);
      if (s < T.nvalid) p.y[(size_t)(b0 + s) * 2 * L + j] = (j < L) ? b.ym[j * SP + s] : b.ys[(j - L) * SP + s];
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(SDE_THREADS, 1) gru_backward_kernel(GruP p) {
  extern __shared__ __align__(16) float sde_sm[];
  GruBufs b;
  gru_carve(sde_sm, p, true, b);
  const int tid = threadIdx.x, nthr = blockDim.x, L = p.L, SP = p.SP, I = 2 * p.L + p.F;
  sde_load_weights(p.nu, p.ps, b.Wu, tid, nthr);
  sde_load_weights(p.nr, p.ps, b.Wr, tid, nthr);
  sde_load_weights(p.nn, p.ps, b.Wn, tid, nthr);
  const int gstride = p.nu.wfloats + p.nr.wfloats + p.nn.wfloats;
  if (p.g_global) {   // networks too large for weights + accumulators in shared memory: accumulate in this CTA's
    b.Gu = p.gpart + (size_t)blockIdx.x * gstride;   // slice of gpart (L2 resident)
    b.Gr = b.Gu + p.nu.wfloats;
    b.Gn = b.Gr + p.nr.wfloats;
  }
  for (int e = tid; e < p.nu.wfloats; e += nthr) b.Gu[e] = 0.0f;
  for (int e = tid; e < p.nr.wfloats; e += nthr) b.Gr[e] = 0.0f;
  for (int e = tid; e < p.nn.wfloats; e += nthr) b.Gn[e] = 0.0f;
  __syncthreads();
  SdeTile T{p.S, SP, L, 0, nthr, tid};
  for (int ti = 0; ti < p.tiles_per_cta; ++ti) {
    const int b0 = (blockIdx.x * p.tiles_per_cta + ti) * p.S;
    if (b0 >= p.B) break;
    T.nvalid = min(p.S, p.B - b0);
    for (int idx = tid; idx < L * T.S; idx += nthr) {
      const int s = idx % T.S, j = idx / T.S, a = j * SP + s;
      b.mb[a] = (s < T.nvalid) ? p.d_y[(size_t)(b0 + s) * 2 * L + j] : 0.0f;
      b.sb[a] = (s < T.nvalid) ? p.d_y[(size_t)(b0 + s) * 2 * L + L + j] : 0.0f;
    }
    __syncthreads();
    for (int t = p.T - 1; t >= 0; --t) {
      for (int idx = tid; idx < L * T.S; idx += nthr) {
        const int s = idx % T.S, j = idx / T.S, a = j * SP + s;
        const size_t g = ((size_t)t * p.B + b0 + s) * 2 * L;
        b.ym[a] = (s < T.nvalid) ? p.carry[g + j] : 0.0f;
        b.ys[a] = (s < T.nvalid) ? p.carry[g + L + j] : 1.0f;
      }
      __syncthreads();
      gru_cell_fwd(p, b, t, b0, T);
      for (int idx = tid; idx < L * T.S; idx += nthr) {
        const int s = idx % T.S, j = idx / T.S, a = j * SP + s;
        const float m = b.mask[s], ug = b.ug[a], nss = b.ns[(L + j) * SP + s], ym = b.ym[a], ys = b.ys[a];
        const float me = m * b.mb[a], se = m * b.sb[a];
        b.nsb[j * SP + s] = 0.0f;
        b.nsb[(L + j) * SP + s] = (1.0f - ug) * (me + se);
        b.ugb[a] = (ym - nss) * me + (ys - nss) * se;
        b.mb[a] = (1.0f - m) * b.mb[a] + ug * me;     // becomes the cotangent of the previous carry
        b.sb[a] = (1.0f - m) * b.sb[a] + ug * se;
      }
      for (int idx = tid; idx < I * T.S; idx += nthr) {
        const int a = (idx / T.S) * SP + (idx % T.S);
        b.c2b[a] = 0.0f; b.ycb[a] = 0.0f;
      }
      __syncthreads();
      sde_mlp_vjp(p.nn, b.Wn, b.Gn, b.c2, 0.0f, b.nsb, b.c2b, b.scr, b.pre, b.post, b.dA, b.dB, T);
      for (int idx = tid; idx < L * T.S; idx += nthr) {
        const int s = idx % T.S, j = idx / T.S, a = j * SP + s;
        const float rg = b.rg[a], cm = b.c2b[a], cs = b.c2b[(L + j) * SP + s];
        b.mb[a] += rg * cm;
        b.sb[a] += rg * cs;
        b.rgb[a] = b.ym[a] * cm + b.ys[a] * cs;
      }
      __syncthreads();
      sde_mlp_vjp(p.nr, b.Wr, b.Gr, b.yc, 0.0f, b.rgb, b.ycb, b.scr, b.pre, b.post, b.dA, b.dB, T);
      sde_mlp_vjp(p.nu, b.Wu, b.Gu, b.yc, 0.0f, b.ugb, b.ycb, b.scr, b.pre, b.post, b.dA, b.dB, T);
      for (int idx = tid; idx < L * T.S; idx += nthr) {
        const int s = idx % T.S, j = idx / T.S, a = j * SP + s;
        b.mb[a] += b.ycb[a];
        b.sb[a] += b.ycb[(L + j) * SP + s];
      }
      __syncthreads();
    }
  }
  if (p.g_global) return;
  const int stride = gstride;
  float* mine = p.gpart + (size_t)blockIdx.x * stride;
  for (int e = tid; e < p.nu.wfloats; e += nthr) mine[e] = b.Gu[e];
  for (int e = tid; e < p.nr.wfloats; e += nthr) mine[p.nu.wfloats + e] = b.Gr[e];
  for (int e = tid; e < p.nn.wfloats; e += nthr) mine[p.nu.wfloats + p.nr.wfloats + e] = b.Gn[e];
}

// ---------------------------------------------------------------- host side
struct lrnde_gru_tape {
  lrnde_ctx* ctx = nullptr;
  GruP p;
  int grid = 1;
  int host = 0;
  std::vector<void*> owned;
  ~lrnde_gru_tape() { for (void* q : owned) ctx->release(q); }
};

static SdeNet gru_make_net(int I, int H, int O, int act2, long long& off) {
  SdeNet n;
  memset(&n, 0, sizeof(n));
  n.nl = 2; n.td = 0; n.D = O;
  const int ins[2] = {I, H}, outs[2] = {H, O}, acts[2] = {ACT_TANH, act2};
  int woff = 0, hoff = 0, md = std::max(I, O);
  for (int l = 0; l < 2; ++l) {
    n.in[l] = ins[l]; n.out[l] = outs[l]; n.outp[l] = (outs[l] + 3) & ~3; n.act[l] = acts[l];
    n.ps_w[l] = off; off += (long long)outs[l] * ins[l];
    n.ps_b[l] = off; off += outs[l];
    n.w_off[l] = woff; woff += (ins[l] + 1) * n.outp[l];
    n.hid_off[l] = hoff; hoff += n.outp[l];
    md = std::max(md, std::max(ins[l], n.outp[l]));
  }
  n.wfloats = woff; n.hid_rows = hoff; n.maxdim = md; n.nparams = 0;
  return n;
}

static void gru_setup(lrnde_ctx* ctx, GruP& p, int F, int H, int L, int T, int64_t B, int* grid) {
  memset(&p, 0, sizeof(p));
  if (F < 2 || H < 1 || L < 1 || T < 1 || B < 1) lr_fail(LRNDE_EINVAL, "lrnde_gru: bad dims");
  long long off = 0;
  const int I = 2 * L + F;
  p.nu = gru_make_net(I, H, L, ACT_SIGMOID, off);
  p.nr = gru_make_net(I, H, L, ACT_SIGMOID, off);
  p.nn = gru_make_net(I, H, 2 * L, ACT_TANH, off);
  p.F = F; p.T = T; p.B = (int)B; p.L = L;
  int n_sm = 0;
  size_t smem_optin = 0;
  sde_device_limits(ctx->device, &n_sm, &smem_optin);
  int S = 32;
  while (S > 8 && ((B + S - 1) / S) < n_sm / 2) S >>= 1;
  p.g_global = ((size_t)(p.nu.wfloats + p.nr.wfloats + p.nn.wfloats) * 2 * sizeof(float) > smem_optin / 2) ? 1 : 0;
  for (;; S >>= 1) {
    p.S = S; p.SP = S + 1;
    if (gru_smem_bytes(p, true) <= smem_optin) break;
    if (S <= 4) lr_fail(LRNDE_EINVAL, "GRU cell too large for the shared-memory resident path");
  }
  const int ntiles = (int)((B + S - 1) / S);
  p.tiles_per_cta = (ntiles + 4 * n_sm - 1) / (4 * n_sm);
  *grid = (ntiles + p.tiles_per_cta - 1) / p.tiles_per_cta;
}

extern "C" int64_t lrnde_gru_nparams(int32_t F, int32_t H, int32_t L) {
  const int64_t I = 2 * (int64_t)L + F;
  return 2 * ((I + 1) * H + (int64_t)(H + 1) * L) + (I + 1) * H + (int64_t)(H + 1) * 2 * L;
}

extern "C" int lrnde_gru_forward(lrnde_ctx* ctx, int32_t F, int32_t H, int32_t L, const float* ps, const float* x,
                                 int32_t T, int64_t B, int32_t host_buffers, int32_t keep_tape, float* y,
                                 lrnde_gru_tape** tape_out) {
  LR_API_BEGIN
  if (!ctx || !ps || !x || !y) lr_fail(LRNDE_EINVAL, "lrnde_gru_forward: bad args");
  if (keep_tape && !tape_out) lr_fail(LRNDE_EINVAL, "keep_tape set but tape is NULL");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  auto Tp = std::make_unique<lrnde_gru_tape>();
  Tp->ctx = ctx; Tp->host = host_buffers;
  GruP& p = Tp->p;
  gru_setup(ctx, p, F, H, L, T, B, &Tp->grid);
  auto take = [&](size_t nfloat) { float* q = (float*)ctx->alloc(sizeof(float) * std::max<size_t>(nfloat, 1)); Tp->owned.push_back(q); return q; };
  const int64_t P = lrnde_gru_nparams(F, H, L);
  const size_t nx = (size_t)F * T * B, ny = (size_t)2 * L * B;
  CallerBufs io(ctx, host_buffers);
  float* psd = take(P); float* xd = take(nx); float* yd = take(ny);
  io.copy_in(psd, ps, P);   // ps and x: kept by the tape for the backward
  io.copy_in(xd, x, nx);
  io.copy_out(y, yd, ny);
  p.ps = psd; p.x = xd; p.y = yd;
  p.carry = keep_tape ? take((size_t)T * ny) : nullptr;
  const size_t smem = gru_smem_bytes(p, false);
  LR_CUDA(cudaFuncSetAttribute(gru_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  gru_forward_kernel<<<Tp->grid, SDE_THREADS, smem, st>>>(p);
  LR_COUNT(ctx);
  LR_CUDA(cudaGetLastError());
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  if (keep_tape) *tape_out = Tp.release();
  LR_API_END
}

extern "C" int lrnde_gru_backward(lrnde_ctx* ctx, lrnde_gru_tape* Tp, const float* d_y, float* d_ps) {
  LR_API_BEGIN
  if (!ctx || !Tp || !d_y || !d_ps) lr_fail(LRNDE_EINVAL, "lrnde_gru_backward: bad args");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  GruP p = Tp->p;
  const size_t ny = (size_t)2 * p.L * p.B;
  const int64_t P = lrnde_gru_nparams(p.F, p.nu.out[0], p.L);
  CallerBufs io(ctx, Tp->host);   // owned copies: pooled (256-byte aligned) arrays that alias no argument
  p.d_y = io.copy_in(d_y, ny);
  float* dps = io.copy_out(d_ps, P);
  const int stride = p.nu.wfloats + p.nr.wfloats + p.nn.wfloats;
  DevBuf gpart(ctx, (size_t)Tp->grid * stride);
  p.gpart = gpart.p;
  const size_t smem = gru_smem_bytes(p, true);
  LR_CUDA(cudaFuncSetAttribute(gru_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  gru_backward_kernel<<<Tp->grid, SDE_THREADS, smem, st>>>(p);
  LR_COUNT(ctx);
  sde_grad_reduce_kernel<<<64, 256, 0, st>>>(p.nu, gpart.p, stride, 0, Tp->grid, dps);
  sde_grad_reduce_kernel<<<64, 256, 0, st>>>(p.nr, gpart.p, stride, p.nu.wfloats, Tp->grid, dps);
  sde_grad_reduce_kernel<<<64, 256, 0, st>>>(p.nn, gpart.p, stride, p.nu.wfloats + p.nr.wfloats, Tp->grid, dps);
  LR_COUNT(ctx); LR_COUNT(ctx); LR_COUNT(ctx);
  LR_CUDA(cudaGetLastError());
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  LR_API_END
}

extern "C" int lrnde_gru_tape_free(lrnde_gru_tape* Tp) {
  LR_API_BEGIN
  delete Tp;
  LR_API_END
}

// ==========================================================================================
// The small layers either side of the latent ODE (physionet model, experiments/src/construct.jl:229-247):
//   rec_to_gen  Chain(Dense(2L => L, tanh), Dense(L => 2N))      -> lrnde_mlp_forward / backward
//   gen_to_data Dense(N => in) applied to every saved time point -> lrnde_mlp_forward / backward
//   ReparameterizeLayer (src/layers/common.jl:48-77)             -> lrnde_reparameterize (+ _backward)
//   log_likelihood_loss / kl_divergence / the latent-ODE loss (experiments/src/utils.jl:94-101,
//   construct.jl:36-70)                                          -> lrnde_latent_loss
// ==========================================================================================
struct MlpOpP {
  SdeNet n;
  const float* ps; const float* x; float* y;   // x [in, N], y [out, N] column-major
  const float* d_y; float* d_x; float* gpart;
  int N, S, SP, tiles_per_cta, in0, outL;
};

__device__ void mlpop_carve(float* sm, const MlpOpP& p, bool bwd, float*& W, float*& G, float*& xin, float*& yout,
                            float*& pre, float*& post, float*& cot, float*& xbar, float*& dA, float*& dB) {
  float* q = sm;
  W = q; q += p.n.wfloats;
  G = nullptr;
  if (bwd) { G = q; q += p.n.wfloats; }
  auto take = [&](int rows) { float* r = q; q += rows * p.SP; return r; };
  xin = take(p.in0); yout = take(p.outL); pre = take(p.n.hid_rows); post = take(p.n.hid_rows);
  cot = xbar = dA = dB = nullptr;
  if (bwd) { cot = take(p.outL); xbar = take(p.in0); dA = take(p.n.maxdim); dB = take(p.n.maxdim); }
}
static size_t mlpop_smem(const MlpOpP& p, bool bwd) {
  size_t f = (size_t)p.n.wfloats * (bwd ? 2 : 1);
  int rows = p.in0 + p.outL + 2 * p.n.hid_rows + (bwd ? p.outL + p.in0 + 2 * p.n.maxdim : 0);
  return (f + (size_t)rows * p.SP) * sizeof(float) + 16;
}

template <bool BWD>
__global__ void __launch_bounds__(SDE_THREADS, 1) mlpop_kernel(MlpOpP p) {
  extern __shared__ __align__(16) float sde_sm[];
  float *W, *G, *xin, *yout, *pre, *post, *cot, *xbar, *dA, *dB;
  mlpop_carve(sde_sm, p, BWD, W, G, xin, yout, pre, post, cot, xbar, dA, dB);
  const int tid = threadIdx.x, nthr = blockDim.x, SP = p.SP;
  sde_load_weights(p.n, p.ps, W, tid, nthr);
  if (BWD) for (int e = tid; e < p.n.wfloats; e += nthr) G[e] = 0.0f;
  __syncthreads();
  SdeTile T{p.S, SP, p.in0, 0, nthr, tid};
  for (int ti = 0; ti < p.tiles_per_cta; ++ti) {
    const int b0 = (blockIdx.x * p.tiles_per_cta + ti) * p.S;
    if (b0 >= p.N) break;
    T.nvalid = min(p.S, p.N - b0);
    for (int idx = tid; idx < p.in0 * T.S; idx += nthr) {
      const int s = idx / p.in0, r = idx % p.in0;
      xin[r * SP + s] = (s < T.nvalid) ? p.x[(size_t)(b0 + s) * p.in0 + r] : 0.0f;
    }
    if (BWD)
      for (int idx = tid; idx < p.outL * T.S; idx += nthr) {
        const int s = idx / p.outL, r = idx % p.outL;
        cot[r * SP + s] = (s < T.nvalid) ? p.d_y[(size_t)(b0 + s) * p.outL + r] : 0.0f;
      }
    if (BWD) for (int idx = tid; idx < p.in0 * T.S; idx += nthr) xbar[(idx / T.S) * SP + (idx % T.S)] = 0.0f;
    __syncthreads();
    if (!BWD) {
      sde_mlp_fwd(p.n, W, xin, 0.0f, yout, pre, post, T);
      for (int idx = tid; idx < p.outL * T.S; idx += nthr) {
        const int s = idx / p.outL, r = idx % p.outL;
        if (s < T.nvalid) p.y[(size_t)(b0 + s) * p.outL + r] = yout[r * SP + s];
      }
    } else {
      sde_mlp_vjp(p.n, W, G, xin, 0.0f, cot, xbar, yout, pre, post, dA, dB, T);
      if (p.d_x)
        for (int idx = tid; idx < p.in0 * T.S; idx += nthr) {
          const int s = idx / p.in0, r = idx % p.in0;
          if (s < T.nvalid) p.d_x[(size_t)(b0 + s) * p.in0 + r] = xbar[r * SP + s];
        }
    }
    __syncthreads();
  }
  if (BWD) {
    float* mine = p.gpart + (size_t)blockIdx.x * p.n.wfloats;
    for (int e = tid; e < p.n.wfloats; e += nthr) mine[e] = G[e];
  }
}

static void mlpop_setup(lrnde_ctx* ctx, MlpOpP& p, const lrnde_layer_desc* layers, int nlayers, int64_t N, int* grid) {
  memset(&p, 0, sizeof(p));
  if (!layers || nlayers < 1 || nlayers > SDE_MAXL || N < 1) lr_fail(LRNDE_EINVAL, "lrnde_mlp: bad args");
  SdeNet& n = p.n;
  n.nl = nlayers; n.td = 0;
  long long off = 0;
  int woff = 0, hoff = 0, md = layers[0].in_dims;
  for (int l = 0; l < nlayers; ++l) {
    const int in = layers[l].in_dims, out = layers[l].out_dims;
    if (in < 1 || out < 1 || (l > 0 && in != layers[l - 1].out_dims)) lr_fail(LRNDE_EINVAL, "lrnde_mlp: layer %d dims", l);
    n.in[l] = in; n.out[l] = out; n.outp[l] = (out + 3) & ~3; n.act[l] = lr_map_act(layers[l].act);
    n.ps_w[l] = off; off += (long long)out * in;
    n.ps_b[l] = off; off += out;
    n.w_off[l] = woff; woff += (in + 1) * n.outp[l];
    n.hid_off[l] = hoff; hoff += n.outp[l];
    md = std::max(md, std::max(in, n.outp[l]));
  }
  n.wfloats = woff; n.hid_rows = hoff; n.maxdim = md; n.nparams = (int)off; n.D = layers[0].in_dims;
  p.in0 = layers[0].in_dims; p.outL = layers[nlayers - 1].out_dims; p.N = (int)N;
  int n_sm = 0;
  size_t smem_optin = 0;
  sde_device_limits(ctx->device, &n_sm, &smem_optin);
  int S = 32;
  for (;; S >>= 1) {
    p.S = S; p.SP = S + 1;
    if (mlpop_smem(p, true) <= smem_optin) break;
    if (S <= 4) lr_fail(LRNDE_EINVAL, "lrnde_mlp: network too large for the shared-memory resident path");
  }
  const int ntiles = (int)((N + S - 1) / S);
  p.tiles_per_cta = (ntiles + 4 * n_sm - 1) / (4 * n_sm);
  *grid = (ntiles + p.tiles_per_cta - 1) / p.tiles_per_cta;
}

extern "C" int lrnde_mlp_forward(lrnde_ctx* ctx, const lrnde_layer_desc* layers, int32_t nlayers, const float* ps,
                                 const float* x, int64_t N, int32_t host_buffers, float* y) {
  LR_API_BEGIN
  if (!ctx || !ps || !x || !y) lr_fail(LRNDE_EINVAL, "lrnde_mlp_forward: bad args");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  MlpOpP p; int grid = 1;
  mlpop_setup(ctx, p, layers, nlayers, N, &grid);
  CallerBufs io(ctx, host_buffers);   // owned copies: pooled (256-byte aligned) arrays that alias no argument
  p.ps = io.copy_in(ps, p.n.nparams);
  p.x = io.copy_in(x, (size_t)p.in0 * N);
  p.y = io.copy_out(y, (size_t)p.outL * N);
  const size_t smem = mlpop_smem(p, false);
  LR_CUDA(cudaFuncSetAttribute(mlpop_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mlpop_kernel<false><<<grid, SDE_THREADS, smem, st>>>(p);
  LR_COUNT(ctx);
  LR_CUDA(cudaGetLastError());
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  LR_API_END
}

extern "C" int lrnde_mlp_backward(lrnde_ctx* ctx, const lrnde_layer_desc* layers, int32_t nlayers, const float* ps,
                                  const float* x, const float* d_y, int64_t N, int32_t host_buffers, float* d_x,
                                  float* d_ps) {
  LR_API_BEGIN
  if (!ctx || !ps || !x || !d_y || !d_ps) lr_fail(LRNDE_EINVAL, "lrnde_mlp_backward: bad args");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  MlpOpP p; int grid = 1;
  mlpop_setup(ctx, p, layers, nlayers, N, &grid);
  CallerBufs io(ctx, host_buffers);   // owned copies: pooled (256-byte aligned) arrays that alias no argument
  p.ps = io.copy_in(ps, p.n.nparams);
  p.x = io.copy_in(x, (size_t)p.in0 * N);
  p.d_y = io.copy_in(d_y, (size_t)p.outL * N);
  DevBuf dxd(ctx, (size_t)p.in0 * N);   // the kernel always writes d_x
  io.copy_out(d_x, dxd.p, (size_t)p.in0 * N);
  DevBuf gpart(ctx, (size_t)grid * p.n.wfloats);
  float* dpsd = io.copy_out(d_ps, p.n.nparams);
  p.d_x = dxd.p; p.gpart = gpart.p;
  const size_t smem = mlpop_smem(p, true);
  LR_CUDA(cudaFuncSetAttribute(mlpop_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mlpop_kernel<true><<<grid, SDE_THREADS, smem, st>>>(p);
  LR_COUNT(ctx);
  sde_grad_reduce_kernel<<<64, 256, 0, st>>>(p.n, gpart.p, p.n.wfloats, 0, grid, dpsd);
  LR_COUNT(ctx);
  LR_CUDA(cudaGetLastError());
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  LR_API_END
}

// ---- ReparameterizeLayer: y = mu + exp(logsigma2 / 2) * eps, eps ~ N(0,1) from Philox(seed, stream 2)
__global__ void reparam_kernel(const float* x, int L, int B, unsigned long long seed, int training, float* y,
                               const float* d_y, const float* d_mu, const float* d_ls, float* d_x) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < (size_t)L * B; i += (size_t)gridDim.x * blockDim.x) {
    const size_t b = i / L, l = i % L;
    const float mu = x[b * 2 * L + l], ls = x[b * 2 * L + L + l];
    const float eps = training ? sde_normal(seed, 2u, 0u, i) : 0.0f;
    const float sd = training ? expf(ls / 2.0f) : 0.0f;
    if (y) y[i] = mu + sd * eps;
    if (d_x) {
      const float g = d_y ? d_y[i] : 0.0f;
      d_x[b * 2 * L + l] = g + (d_mu ? d_mu[i] : 0.0f);
      d_x[b * 2 * L + L + l] = g * eps * sd * 0.5f + (d_ls ? d_ls[i] : 0.0f);
    }
  }
}

// x [2L,B] -> y [L,B]; d_x (optional pass: give d_y and/or the KL cotangents d_mu, d_ls) [2L,B]
extern "C" int lrnde_reparameterize(lrnde_ctx* ctx, const float* x, int32_t L, int64_t B, uint64_t seed, int32_t training,
                                    int32_t host_buffers, float* y, const float* d_y, const float* d_mu,
                                    const float* d_ls, float* d_x) {
  LR_API_BEGIN
  if (!ctx || !x || L < 1 || B < 1) lr_fail(LRNDE_EINVAL, "lrnde_reparameterize: bad args");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t n = (size_t)L * B;
  CallerBufs io(ctx, host_buffers);   // owned copies: pooled (256-byte aligned) arrays that alias no argument
  const float* xd = io.copy_in(x, 2 * n);
  float* yd = io.copy_out(y, n);
  const float* dyd = io.copy_in(d_y, n);
  const float* dmd = io.copy_in(d_mu, n);
  const float* dld = io.copy_in(d_ls, n);
  float* dxd = io.copy_out(d_x, 2 * n);
  reparam_kernel<<<lr_ew_blocks(n), 256, 0, st>>>(xd, L, (int)B, seed, training, yd, dyd, dmd, dld, dxd);
  LR_COUNT(ctx);
  LR_CUDA(cudaGetLastError());
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  LR_API_END
}

// ---- latent-ODE loss: -mean_b(ll_b - w_kl * kl_b) with the reference's formulas
// (experiments/src/utils.jl:94-101: the Gaussian normaliser is summed over ALL entries, observed or not, and
// divided by the number of observed ones).  One CTA per sample; sums in double, fixed order.
__global__ void __launch_bounds__(256) latent_loss_kernel(const float* pred, const float* data, const float* mask,
                                                          const float* mu, const float* ls, int FT, int L, int B,
                                                          float w_kl, double* per_sample, float* d_pred, float* d_mu,
                                                          float* d_ls) {
  const int b = blockIdx.x;
  const float sig = 0.01f;
  const float cst = -logf(sig) - logf(6.283185307179586f) / 2.0f;
  double lik = 0.0, msum = 0.0;
  for (int i = threadIdx.x; i < FT; i += blockDim.x) {
    const size_t g = (size_t)b * FT + i;
    const float m = mask[g];
    const float r = pred[g] * m - data[g] * m;
    lik += (double)(-(r * r) / (2.0f * sig * sig) + cst);
    msum += (double)m;
  }
  __shared__ double s_bc[2];
  lik = lr_block_sum(lik);       // valid in thread 0 only
  msum = lr_block_sum(msum);
  if (threadIdx.x == 0) { s_bc[0] = lik; s_bc[1] = msum; }
  __syncthreads();
  lik = s_bc[0]; msum = s_bc[1];
  double kl = 0.0;
  for (int i = threadIdx.x; i < L; i += blockDim.x) {
    const float m_ = mu[(size_t)b * L + i], l_ = ls[(size_t)b * L + i];
    kl += (double)(expf(l_) + m_ * m_ - 1.0f - l_);
  }
  kl = lr_block_sum(kl) / (2.0 * L);
  if (threadIdx.x == 0) { per_sample[2 * b] = lik / msum; per_sample[2 * b + 1] = kl; }
  const float inv = (float)(1.0 / msum) / (float)B;
  if (d_pred)
    for (int i = threadIdx.x; i < FT; i += blockDim.x) {
      const size_t g = (size_t)b * FT + i;
      const float m = mask[g];
      d_pred[g] = ((pred[g] * m - data[g] * m) * m / (sig * sig)) * inv;
    }
  if (d_mu)
    for (int i = threadIdx.x; i < L; i += blockDim.x) {
      d_mu[(size_t)b * L + i] = w_kl * mu[(size_t)b * L + i] / ((float)L * (float)B);
      d_ls[(size_t)b * L + i] = w_kl * (expf(ls[(size_t)b * L + i]) - 1.0f) / (2.0f * (float)L * (float)B);
    }
}

// pred / data / mask: [F,T,B]; mu / logsigma2: [L,B].  out3 (HOST) = {loss, -mean(ll), mean(kl)}.
extern "C" int lrnde_latent_loss(lrnde_ctx* ctx, const float* pred, const float* data, const float* mask, const float* mu,
                                 const float* logsigma2, int32_t F, int32_t T, int32_t L, int64_t B, float w_kl,
                                 int32_t host_buffers, float* out3, float* d_pred, float* d_mu, float* d_logsigma2) {
  LR_API_BEGIN
  if (!ctx || !pred || !data || !mask || !mu || !logsigma2 || !out3) lr_fail(LRNDE_EINVAL, "lrnde_latent_loss: bad args");
  if ((d_mu == nullptr) != (d_logsigma2 == nullptr)) lr_fail(LRNDE_EINVAL, "d_mu and d_logsigma2 go together");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t n = (size_t)F * T * B, nl = (size_t)L * B;
  CallerBufs io(ctx, host_buffers);   // owned copies: pooled (256-byte aligned) arrays that alias no argument
  const float* pd = io.copy_in(pred, n);
  const float* dd = io.copy_in(data, n);
  const float* md = io.copy_in(mask, n);
  const float* mud = io.copy_in(mu, nl);
  const float* lsd = io.copy_in(logsigma2, nl);
  float* dpd = io.copy_out(d_pred, n);
  float* dmu = io.copy_out(d_mu, nl);
  float* dls = io.copy_out(d_logsigma2, nl);
  DevBuf per(ctx, 4 * (size_t)B + 4);
  latent_loss_kernel<<<(unsigned)B, 256, 0, st>>>(pd, dd, md, mud, lsd, F * T, L, (int)B, w_kl, (double*)per.p, dpd, dmu,
                                                  dls);
  LR_COUNT(ctx);
  LR_CUDA(cudaGetLastError());
  std::vector<double> h(2 * (size_t)B);
  LR_CUDA(cudaMemcpyAsync(h.data(), per.p, sizeof(double) * 2 * B, cudaMemcpyDeviceToHost, st));
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  double ll = 0.0, kl = 0.0;
  for (int64_t b = 0; b < B; ++b) { ll += h[2 * b]; kl += h[2 * b + 1]; }
  ll /= (double)B; kl /= (double)B;
  out3[0] = (float)(-(ll - (double)w_kl * kl));
  out3[1] = (float)(-ll);
  out3[2] = (float)kl;
  LR_API_END
}
