// Neural SDE side of the hot path (included at the end of lrnde_api.cu, single translation unit):
//
//   lrnde_sde_forward   replaces (n::NeuralDSDE)(x, ps, st)           src/layers/neural_sde.jl:82-123
//                       = _solve_neuraldsde_generic (:44-72: solve(SDEProblem(dudt, g, x, tspan, ps),
//                         SOSRI(); saveat, maxiters, abstol, reltol)) + _get_dsde_integrator (:35-40)
//                         + _perform_step(::FourStageSRIConstantCache) (src/perform_step.jl:49-106)
//   lrnde_sde_backward  replaces the TrackerAdjoint pullback (neural_sde.jl:12): reverse mode through
//                       every accepted SOSRI step (dt, EEst and the noise are constants) and through the
//                       linear interpolation of each saved state; reg_val w.r.t. the parameters only
//                       (_get_dsde_integrator is @non_differentiable, neural_sde.jl:42)
//
// The SOSRI solve loop, the RSwM3 rejection sampling of the Wiener increments, sde_determine_initdt
// and the PI controller live in un-vendored StochasticDiffEq / DiffEqNoiseProcess; they follow
// SURVEY App. A.6 exactly as restated in oracle/lrnde_sde_oracle.py (same constants, same order of
// noise draws).  Noise: counter-based Philox4x32-10, counter = (element, draw, stream), key = seed.
//
// B200 mapping.  The SDE states of the reference configs are small (mnist_sde: 32 x 128, drift
// 32-64-32, diffusion 32-32: 6.3 K parameters), so the whole adaptive solve is ONE persistent
// cooperative kernel: every CTA owns a fixed slice of the batch, keeps both networks in shared
// memory, evaluates the 4 drift + 4 diffusion stages of an attempt out of shared memory, and the
// grid meets once per attempt (grid.sync) to sum the error norm; the PI controller, accept/reject
// and the RSwM3 stack bookkeeping are then recomputed identically by every CTA, and the stack /
// bridge arithmetic is element-wise on the CTA's own slice.  No host round trip inside a solve, no
// launch per stage.  The reverse pass is one ordinary launch over the same slices with the
// parameter gradients accumulated in shared memory and reduced in a fixed order.
#pragma once
#include <cooperative_groups.h>

namespace cg = cooperative_groups;

#include "lrnde_smem_mlp.cuh"

// ---------------------------------------------------------------- Philox4x32-10
__device__ __forceinline__ float sde_normal(unsigned long long seed, unsigned stream, unsigned draw,
                                            unsigned long long elem) {
  unsigned c0 = (unsigned)elem, c1 = (unsigned)(elem >> 32), c2 = draw, c3 = stream;
  unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  const double u1 = ((double)c0 + 0.5) * 2.3283064365386963e-10;
  const double u2 = ((double)c1 + 0.5) * 2.3283064365386963e-10;
  return (float)(sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2));
}

// ---------------------------------------------------------------- SOSRI step on a tile
struct SdeBufs {
  float *U, *dW, *dZ, *k[4], *g[4], *H0, *H1, *un;
  float *pre, *post, *dA, *dB;  // network scratch
  // reverse pass only
  float *kb[4], *gb[4], *Ub, *hb0, *hb1, *cot, *E1b, *E2b;
};

__device__ __forceinline__ void sde_chi(float dW, float dZ, float dt, float sqdt, float& chi1, float& chi2,
                                        float& chi3) {
  chi1 = (dW * dW - fabsf(dt)) / (2.0f * sqdt);
  chi2 = (dW + dZ / sqrtf(3.0f)) / 2.0f;
  chi3 = (dW * dW * dW - 3.0f * dW * dt) / (6.0f * dt);
}

// H0_stage / H1_stage of stage = 2..4 from k1..k_{stage-1}, g1..g_{stage-1} (perform_step.jl:65-82)
__device__ void sde_stage_inputs(const SosriTab& c, const SdeBufs& b, int stage, float dt, float sqdt,
                                 const SdeTile& T) {
  for (int idx = T.tid; idx < T.D * T.S; idx += T.nthr) {
    const int a = (idx / T.S) * T.SP + (idx % T.S);
    float chi1, chi2, chi3;
    sde_chi(b.dW[a], b.dZ[a], dt, sqdt, chi1, chi2, chi3);
    const float up = b.U[a];
    float h0, h1;
    if (stage == 2) {
      h0 = up + dt * c.a021 * b.k[0][a] + c.b021 * chi2 * b.g[0][a];
      h1 = up + dt * c.a121 * b.k[0][a] + sqdt * c.b121 * b.g[0][a];
    } else if (stage == 3) {
      h0 = up + dt * (c.a031 * b.k[0][a] + c.a032 * b.k[1][a]) + chi2 * (c.b031 * b.g[0][a] + c.b032 * b.g[1][a]);
      h1 = up + dt * (c.a131 * b.k[0][a] + c.a132 * b.k[1][a]) + sqdt * (c.b131 * b.g[0][a] + c.b132 * b.g[1][a]);
    } else {
      h0 = up + dt * (c.a041 * b.k[0][a] + c.a042 * b.k[1][a] + c.a043 * b.k[2][a]) +
           chi2 * (c.b041 * b.g[0][a] + c.b042 * b.g[1][a] + c.b043 * b.g[2][a]);
      h1 = up + dt * (c.a141 * b.k[0][a] + c.a142 * b.k[1][a] + c.a143 * b.k[2][a]) +
           sqdt * (c.b141 * b.g[0][a] + c.b142 * b.g[1][a] + c.b143 * b.g[2][a]);
    }
    b.H0[a] = h0;
    b.H1[a] = h1;
  }
  __syncthreads();
}

__device__ __forceinline__ float sde_stage_t(const SosriTab& c, int stage, int which, float t, float dt) {
  const float c0[4] = {0.0f, c.c02, c.c03, c.c04};
  const float c1[4] = {c.c11, c.c12, c.c13, c.c14};
  return t + (which ? c1[stage - 1] : c0[stage - 1]) * dt;
}

// k1..k4, g1..g4, u_new for the tile; returns this thread's partial sum of resid^2 (valid samples)
__device__ double sde_sosri_fwd(const SosriTab& c, const SdeNet& nf, const SdeNet& ng, const float* Wf,
                                const float* Wg, const SdeBufs& b, float t, float dt, float abstol,
                                float reltol, float delta, const SdeTile& T) {
  const float sqdt = sqrtf(fabsf(dt));
  sde_mlp_fwd(nf, Wf, b.U, t, b.k[0], b.pre, b.post, T);
  sde_mlp_fwd(ng, Wg, b.U, sde_stage_t(c, 1, 1, t, dt), b.g[0], b.pre, b.post, T);
  for (int st = 2; st <= 4; ++st) {
    sde_stage_inputs(c, b, st, dt, sqdt, T);
    sde_mlp_fwd(nf, Wf, b.H0, sde_stage_t(c, st, 0, t, dt), b.k[st - 1], b.pre, b.post, T);
    sde_mlp_fwd(ng, Wg, b.H1, sde_stage_t(c, st, 1, t, dt), b.g[st - 1], b.pre, b.post, T);
  }
  double part = 0.0;
  for (int idx = T.tid; idx < T.D * T.S; idx += T.nthr) {
    const int s = idx % T.S, a = (idx / T.S) * T.SP + s;
    float chi1, chi2, chi3;
    sde_chi(b.dW[a], b.dZ[a], dt, sqdt, chi1, chi2, chi3);
    const float k1 = b.k[0][a], k2 = b.k[1][a], k3 = b.k[2][a], k4 = b.k[3][a];
    const float g1 = b.g[0][a], g2 = b.g[1][a], g3 = b.g[2][a], g4 = b.g[3][a];
    const float E2 = chi2 * (c.be31 * g1 + c.be32 * g2 + c.be33 * g3 + c.be34 * g4) +
                     chi3 * (c.be41 * g1 + c.be42 * g2 + c.be43 * g3 + c.be44 * g4);
    const float up = b.U[a];
    const float u = up + dt * (c.al1 * k1 + c.al2 * k2 + c.al3 * k3 + c.al4 * k4) + E2 +
                    b.dW[a] * (c.be11 * g1 + c.be12 * g2 + c.be13 * g3 + c.be14 * g4) +
                    chi1 * (c.be21 * g1 + c.be22 * g2 + c.be23 * g3 + c.be24 * g4);
    const float E1 = dt * (k1 + k2 + k3 + k4);
    b.un[a] = u;
    if (s < T.nvalid) {
      const float r = (delta * E1 + E2) / (abstol + fmaxf(fabsf(up), fabsf(u)) * reltol);
      part += (double)r * (double)r;
    }
  }
  __syncthreads();
  return part;
}

// Reverse mode through the step (oracle sosri_step_backward).  In: b.cot = cotangent of u_new,
// optional b.E1b / b.E2b (regulariser; nullptr = zero).  Out: b.Ub = cotangent of uprev, G += param grads.
__device__ void sde_sosri_bwd(const SosriTab& c, const SdeNet& nf, const SdeNet& ng, const float* Wf,
                              const float* Wg, float* Gf, float* Gg, const SdeBufs& b, float t, float dt,
                              bool use_E, const SdeTile& T) {
  const float sqdt = sqrtf(fabsf(dt));
  // forward internals (k, g) are recomputed; un is scratch here
  sde_mlp_fwd(nf, Wf, b.U, t, b.k[0], b.pre, b.post, T);
  sde_mlp_fwd(ng, Wg, b.U, sde_stage_t(c, 1, 1, t, dt), b.g[0], b.pre, b.post, T);
  for (int st = 2; st <= 4; ++st) {
    sde_stage_inputs(c, b, st, dt, sqdt, T);
    sde_mlp_fwd(nf, Wf, b.H0, sde_stage_t(c, st, 0, t, dt), b.k[st - 1], b.pre, b.post, T);
    sde_mlp_fwd(ng, Wg, b.H1, sde_stage_t(c, st, 1, t, dt), b.g[st - 1], b.pre, b.post, T);
  }
  const float al[4] = {c.al1, c.al2, c.al3, c.al4};
  const float b1[4] = {c.be11, c.be12, c.be13, c.be14}, b2[4] = {c.be21, c.be22, c.be23, c.be24};
  const float b3[4] = {c.be31, c.be32, c.be33, c.be34}, b4[4] = {c.be41, c.be42, c.be43, c.be44};
  for (int idx = T.tid; idx < T.D * T.S; idx += T.nthr) {
    const int a = (idx / T.S) * T.SP + (idx % T.S);
    float chi1, chi2, chi3;
    sde_chi(b.dW[a], b.dZ[a], dt, sqdt, chi1, chi2, chi3);
    const float ub = b.cot[a];
    const float e1 = use_E ? b.E1b[a] : 0.0f;
    const float e2t = ub + (use_E ? b.E2b[a] : 0.0f);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      b.kb[i][a] = dt * al[i] * ub + dt * e1;
      b.gb[i][a] = (chi2 * b3[i] + chi3 * b4[i]) * e2t + (b.dW[a] * b1[i] + chi1 * b2[i]) * ub;
    }
    b.Ub[a] = ub;
  }
  __syncthreads();
  const float a0[4][3] = {{0, 0, 0}, {c.a021, 0, 0}, {c.a031, c.a032, 0}, {c.a041, c.a042, c.a043}};
  const float a1[4][3] = {{0, 0, 0}, {c.a121, 0, 0}, {c.a131, c.a132, 0}, {c.a141, c.a142, c.a143}};
  const float bb0[4][3] = {{0, 0, 0}, {c.b021, 0, 0}, {c.b031, c.b032, 0}, {c.b041, c.b042, c.b043}};
  const float bb1[4][3] = {{0, 0, 0}, {c.b121, 0, 0}, {c.b131, c.b132, 0}, {c.b141, c.b142, c.b143}};
  for (int st = 4; st >= 1; --st) {
    const float* x0 = b.U;
    const float* x1 = b.U;
    if (st > 1) {
      sde_stage_inputs(c, b, st, dt, sqdt, T);
      x0 = b.H0; x1 = b.H1;
    }
    for (int idx = T.tid; idx < T.D * T.S; idx += T.nthr) {
      const int a = (idx / T.S) * T.SP + (idx % T.S);
      b.hb0[a] = 0.0f; b.hb1[a] = 0.0f;
    }
    __syncthreads();
    sde_mlp_vjp(nf, Wf, Gf, x0, sde_stage_t(c, st, 0, t, dt), b.kb[st - 1], b.hb0, b.un, b.pre, b.post, b.dA, b.dB, T);
    sde_mlp_vjp(ng, Wg, Gg, x1, sde_stage_t(c, st, 1, t, dt), b.gb[st - 1], b.hb1, b.un, b.pre, b.post, b.dA, b.dB, T);
    for (int idx = T.tid; idx < T.D * T.S; idx += T.nthr) {
      const int a = (idx / T.S) * T.SP + (idx % T.S);
      const float h0 = b.hb0[a], h1 = b.hb1[a];
      b.Ub[a] += h0 + h1;
      if (st > 1) {
        float chi1, chi2, chi3;
        sde_chi(b.dW[a], b.dZ[a], dt, sqdt, chi1, chi2, chi3);
        for (int j = 0; j < st - 1; ++j) {
          b.kb[j][a] += dt * (a0[st - 1][j] * h0 + a1[st - 1][j] * h1);
          b.gb[j][a] += chi2 * bb0[st - 1][j] * h0 + sqdt * bb1[st - 1][j] * h1;
        }
      }
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------- tile <-> global ([D, B] column-major)
__device__ __forceinline__ void sde_tile_load(float* dst, const float* __restrict__ g, int b0, const SdeTile& T) {
  for (int idx = T.tid; idx < T.D * T.S; idx += T.nthr) {
    const int s = idx / T.D, d = idx % T.D;
    dst[d * T.SP + s] = (s < T.nvalid) ? g[(size_t)(b0 + s) * T.D + d] : 0.0f;
  }
}
__device__ __forceinline__ void sde_tile_store(float* __restrict__ g, const float* src, int b0, const SdeTile& T) {
  for (int idx = T.tid; idx < T.D * T.S; idx += T.nthr) {
    const int s = idx / T.D, d = idx % T.D;
    if (s < T.nvalid) g[(size_t)(b0 + s) * T.D + d] = src[d * T.SP + s];
  }
}

__device__ double sde_block_sum(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  double tot = 0.0;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += red[i];
  __syncthreads();
  return tot;
}


// Sum of slot `k` of every CTA's partial record, identical on every CTA: lane l adds the records
// l, l + 32, ... in order, then a fixed shuffle tree.  Call from all threads of warp 0.
__device__ __forceinline__ double sde_partials_sum(const double* base, int nblk, int k) {
  double v = 0.0;
  for (int i = threadIdx.x & 31; i < nblk; i += 32) v += base[(size_t)i * 4 + k];
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------- kernel parameters
struct SdeShared {  // controller state, identical in every CTA
  float t, dt, qold, tnew;
  int iter, nacc, nrej, retcode, n1, n2, ndraw, next_save, natt;
  float L1[SDE_STK], L2[SDE_STK];
  // plan of the element-wise phase
  int accept;
  int npop, split, push_rem, fresh, draw_split, draw_fresh, sv_first, sv_count;
  float q_split, L_split, left;
  int nmove, push_cut, draw_rej, n2_before;
  float qK, dtK;
  float dt0;  // initdt
  int stk_overflow;
};

struct SdeSolveP {
  SdeNet nf, ng;
  SdeConsts k;
  SosriTab tab;
  const float* psf; const float* psg;
  int B, S, SP, tiles_per_cta;
  float t0, t2, abstol, reltol;
  int maxiters;
  unsigned long long seed;
  unsigned first_draw;
  // tape: states [cap + 1][D*B], increments [cap + 1][D*B] (slot n = attempt in flight after n accepts)
  float* tape_u; float* tape_w; float* tape_z; float* tape_t; float* tape_dt;
  int cap;
  float* S1w; float* S1z; float* S2w; float* S2z;  // [SDE_STK][D*B]
  const float* save_t; int nsave; float* u_save; int* save_step; float* save_theta;
  double* partials;  // [2][grid][4]
  float* log_t; float* log_dt; float* log_e; unsigned char* log_a; int log_cap;
  int* out_i;    // [0] nacc [1] nrej [2] retcode [3] ndraw [4] natt [5] nf_drift [6] nf_diffusion [7] overflow
  float* out_f;  // [0] t_final [1] dt_reg [2] eest_reg
  // regulariser step (sde_reg_kernel)
  const float* u1; float t1; float* reg_w; float* reg_z;
};

struct SdeSmemLayout { int W_f, W_g, G_f, G_g, bufs, total_floats; };

// carve the dynamic shared memory: weights (+ gradient accumulators), then nbuf [D][SP] tiles, then
// the network scratch
__device__ void sde_carve(float* sm, const SdeNet& nf, const SdeNet& ng, int D, int SP, bool bwd, float*& Wf,
                          float*& Wg, float*& Gf, float*& Gg, SdeBufs& b) {
  float* p = sm;
  Wf = p; p += nf.wfloats;
  Wg = p; p += ng.wfloats;
  Gf = Gg = nullptr;
  if (bwd) { Gf = p; p += nf.wfloats; Gg = p; p += ng.wfloats; }
  const int tile = D * SP;
  auto take = [&]() { float* r = p; p += tile; return r; };
  b.U = take(); b.dW = take(); b.dZ = take();
  for (int i = 0; i < 4; ++i) b.k[i] = take();
  for (int i = 0; i < 4; ++i) b.g[i] = take();
  b.H0 = take(); b.H1 = take(); b.un = take();
  const int hid = max(nf.hid_rows, ng.hid_rows), md = max(nf.maxdim, ng.maxdim);
  b.pre = p; p += hid * SP;
  b.post = p; p += hid * SP;
  b.dA = b.dB = nullptr;
  if (bwd) {
    b.dA = p; p += md * SP;
    b.dB = p; p += md * SP;
    for (int i = 0; i < 4; ++i) b.kb[i] = take();
    for (int i = 0; i < 4; ++i) b.gb[i] = take();
    b.Ub = take(); b.hb0 = take(); b.hb1 = take(); b.cot = take(); b.E1b = take(); b.E2b = take();
  }
}
static size_t sde_smem_bytes(const SdeNet& nf, const SdeNet& ng, int D, int SP, bool bwd) {
  size_t f = (size_t)(nf.wfloats + ng.wfloats) * (bwd ? 2 : 1);
  const int hid = std::max(nf.hid_rows, ng.hid_rows), md = std::max(nf.maxdim, ng.maxdim);
  f += (size_t)D * SP * (bwd ? 28 : 14) + (size_t)hid * SP * 2 + (bwd ? (size_t)md * SP * 2 : 0);
  return f * sizeof(float) + 16;
}

// sde_determine_initdt (SURVEY A.6 / oracle sde_initdt) for the CTA's tiles of `u` at time t;
// two grid-wide sums.  Every CTA returns the same dt.
__device__ float sde_initdt_coop(const SdeSolveP& p, const float* Wf, const float* Wg, const SdeBufs& b,
                                 const float* u, float t, float dtmax, int parity_base, double* red,
                                 cg::grid_group& grid) {
  SdeTile T{p.S, p.SP, p.nf.D, 0, (int)blockDim.x, (int)threadIdx.x};
  const size_t n_total = (size_t)p.B * p.nf.D;
  double s0 = 0.0, s1 = 0.0;
  for (int ti = 0; ti < p.tiles_per_cta; ++ti) {
    const int b0 = (blockIdx.x * p.tiles_per_cta + ti) * p.S;
    if (b0 >= p.B) break;
    T.nvalid = min(p.S, p.B - b0);
    sde_tile_load(b.U, u, b0, T);
    __syncthreads();
    sde_mlp_fwd(p.nf, Wf, b.U, t, b.k[0], b.pre, b.post, T);
    sde_mlp_fwd(p.ng, Wg, b.U, t, b.g[0], b.pre, b.post, T);
    for (int idx = T.tid; idx < T.D * T.S; idx += T.nthr) {
      const int s = idx % T.S, a = (idx / T.S) * T.SP + s;
      if (s < T.nvalid) {
        const float u0 = b.U[a], sk = p.abstol + fabsf(u0) * p.reltol;
        const float f0 = b.k[0][a], g0 = 3.0f * b.g[0][a];
        const float r0 = u0 / sk, r1 = fmaxf(fabsf(f0 + g0), fabsf(f0 - g0)) / sk;
        s0 += (double)r0 * r0; s1 += (double)r1 * r1;
      }
    }
    __syncthreads();
  }
  s0 = sde_block_sum(s0, red);
  s1 = sde_block_sum(s1, red);
  double* mine = p.partials + ((size_t)(parity_base & 1) * gridDim.x + blockIdx.x) * 4;
  if (threadIdx.x == 0) { mine[0] = s0; mine[1] = s1; }
  grid.sync();
  __shared__ double s_tot[2];
  if (threadIdx.x < 32) {
    const double* q = p.partials + (size_t)(parity_base & 1) * gridDim.x * 4;
    const double a = sde_partials_sum(q, gridDim.x, 0), c = sde_partials_sum(q, gridDim.x, 1);
    if (threadIdx.x == 0) { s_tot[0] = a; s_tot[1] = c; }
  }
  __syncthreads();
  const double t0s = s_tot[0], t1s = s_tot[1];
  __syncthreads();
  const float d0 = sqrtf((float)(t0s / (double)n_total)), d1 = sqrtf((float)(t1s / (double)n_total));
  float dt0 = (d0 < 1e-5f || d1 < 1e-5f) ? 1e-6f : 0.01f * (d0 / d1);
  dt0 = fminf(dt0, dtmax);
  double s2 = 0.0;
  for (int ti = 0; ti < p.tiles_per_cta; ++ti) {
    const int b0 = (blockIdx.x * p.tiles_per_cta + ti) * p.S;
    if (b0 >= p.B) break;
    T.nvalid = min(p.S, p.B - b0);
    sde_tile_load(b.U, u, b0, T);
    __syncthreads();
    sde_mlp_fwd(p.nf, Wf, b.U, t, b.k[0], b.pre, b.post, T);
    sde_mlp_fwd(p.ng, Wg, b.U, t, b.g[0], b.pre, b.post, T);
    for (int idx = T.tid; idx < T.D * T.S; idx += T.nthr) {
      const int a = (idx / T.S) * T.SP + (idx % T.S);
      b.H0[a] = b.U[a] + dt0 * b.k[0][a];
    }
    __syncthreads();
    sde_mlp_fwd(p.nf, Wf, b.H0, t + dt0, b.k[1], b.pre, b.post, T);
    sde_mlp_fwd(p.ng, Wg, b.H0, t + dt0, b.g[1], b.pre, b.post, T);
    for (int idx = T.tid; idx < T.D * T.S; idx += T.nthr) {
      const int s = idx % T.S, a = (idx / T.S) * T.SP + s;
      if (s < T.nvalid) {
        const float sk = p.abstol + fabsf(b.U[a]) * p.reltol;
        const float f0 = b.k[0][a], g0 = 3.0f * b.g[0][a], f1 = b.k[1][a], g1 = 3.0f * b.g[1][a];
        const float dg = fmaxf(fabsf(g0 - g1), fabsf(g0 + g1));
        const float r = fmaxf(fabsf(f1 - f0 + dg), fabsf(f1 - f0 - dg)) / sk;
        s2 += (double)r * r;
      }
    }
    __syncthreads();
  }
  s2 = sde_block_sum(s2, red);
  double* mine2 = p.partials + ((size_t)((parity_base + 1) & 1) * gridDim.x + blockIdx.x) * 4;
  if (threadIdx.x == 0) mine2[0] = s2;
  grid.sync();
  if (threadIdx.x < 32) {
    const double a = sde_partials_sum(p.partials + (size_t)((parity_base + 1) & 1) * gridDim.x * 4, gridDim.x, 0);
    if (threadIdx.x == 0) s_tot[0] = a;
  }
  __syncthreads();
  const double t2s = s_tot[0];
  __syncthreads();
  const float d2 = sqrtf((float)(t2s / (double)n_total)) / dt0;
  const float mx = fmaxf(d1, d2);
  float dt1;
  if (mx <= 1e-15f) dt1 = fmaxf(1e-6f, dt0 * 1e-3f);
  else dt1 = powf(10.0f, -(2.0f + log10f(mx)) / (p.k.order + 0.5f));
  return fminf(fminf(100.0f * dt0, dt1), dtmax);
}

// ---------------------------------------------------------------- the adaptive solve
__global__ void __launch_bounds__(SDE_THREADS, 1) sde_solve_kernel(SdeSolveP p) {
  cg::grid_group grid = cg::this_grid();
  extern __shared__ __align__(16) float sde_sm[];
  __shared__ SdeShared C;
  __shared__ double red[32];
  float *Wf, *Wg, *Gf, *Gg;
  SdeBufs b;
  const int D = p.nf.D;
  sde_carve(sde_sm, p.nf, p.ng, D, p.SP, false, Wf, Wg, Gf, Gg, b);
  const int tid = threadIdx.x, nthr = blockDim.x;
  sde_load_weights(p.nf, p.psf, Wf, tid, nthr);
  sde_load_weights(p.ng, p.psg, Wg, tid, nthr);
  __syncthreads();
  const size_t DB = (size_t)D * p.B;
  const float dtmax = fabsf(p.t2 - p.t0);
  const float dtmin = fmaxf(lr_spacing(p.t0), lr_spacing(p.t2));
  // this CTA's slice of the flat [D*B] arrays
  const size_t e_begin = (size_t)blockIdx.x * p.tiles_per_cta * p.S * D;
  const size_t e_end = min(DB, e_begin + (size_t)p.tiles_per_cta * p.S * D);

  float dt_init = sde_initdt_coop(p, Wf, Wg, b, p.tape_u, p.t0, dtmax, 0, red, grid);
  if (tid == 0) {
    C.t = p.t0; C.qold = p.k.qoldinit; C.iter = 0; C.nacc = 0; C.nrej = 0; C.retcode = 0;
    C.n1 = 0; C.n2 = 0; C.ndraw = p.first_draw; C.next_save = 0; C.natt = 0; C.stk_overflow = 0;
    float dt = fminf(fmaxf(dt_init, dtmin), dtmax);
    dt = fminf(dt, p.t2 - p.t0);
    C.dt = dt;
  }
  __syncthreads();
  // first increments: sqrt(dt) * N  (draw C.ndraw)
  {
    const float sq = sqrtf(C.dt);
    const unsigned dr = C.ndraw;
    for (size_t e = e_begin + tid; e < e_end; e += nthr) {
      p.tape_w[e] = sq * sde_normal(p.seed, 0u, dr, e);
      p.tape_z[e] = sq * sde_normal(p.seed, 1u, dr, e);
    }
    __syncthreads();
    if (tid == 0) C.ndraw++;
    __syncthreads();
  }
  // saves at (or before) t0: the initial state (save_start); save_step = -1
  while (C.next_save < p.nsave && p.save_t[C.next_save] <= p.t0) {
    float* dst = p.u_save + (size_t)C.next_save * DB;
    for (size_t e = e_begin + tid; e < e_end; e += nthr) dst[e] = p.tape_u[e];
    __syncthreads();
    if (tid == 0) {
      if (blockIdx.x == 0) { p.save_step[C.next_save] = -1; p.save_theta[C.next_save] = 0.0f; }
      C.next_save++;
    }
    __syncthreads();
  }
  SdeTile T{p.S, p.SP, D, 0, nthr, tid};
  int parity = 0;
  while (true) {
    // ---- loop header (uniform over the grid: every CTA holds the same C)
    if (!(C.t < p.t2) || C.retcode != 0) break;
    if (C.iter + 1 > p.maxiters) { if (tid == 0) C.retcode = LRNDE_RET_MAXITERS; __syncthreads(); break; }
    if (C.dt <= dtmin && !(C.t + C.dt >= p.t2)) { if (tid == 0) C.retcode = LRNDE_RET_DTMIN; __syncthreads(); break; }
    if (C.nacc >= p.cap) { if (tid == 0) C.retcode = LRNDE_RET_TAPEFULL; __syncthreads(); break; }
    const int n = C.nacc;
    const float t = C.t, dt = C.dt;
    float* ucur = p.tape_u + (size_t)n * DB;
    float* unew = p.tape_u + (size_t)(n + 1) * DB;
    float* dWg = p.tape_w + (size_t)n * DB;
    float* dZg = p.tape_z + (size_t)n * DB;
    // ---- the attempt
    double part = 0.0;
    for (int ti = 0; ti < p.tiles_per_cta; ++ti) {
      const int b0 = (blockIdx.x * p.tiles_per_cta + ti) * p.S;
      if (b0 >= p.B) break;
      T.nvalid = min(p.S, p.B - b0);
      sde_tile_load(b.U, ucur, b0, T);
      sde_tile_load(b.dW, dWg, b0, T);
      sde_tile_load(b.dZ, dZg, b0, T);
      __syncthreads();
      part += sde_sosri_fwd(p.tab, p.nf, p.ng, Wf, Wg, b, t, dt, p.abstol, p.reltol, p.k.delta, T);
      sde_tile_store(unew, b.un, b0, T);
      __syncthreads();
    }
    part = sde_block_sum(part, red);
    if (tid == 0) p.partials[((size_t)parity * gridDim.x + blockIdx.x) * 4] = part;
    grid.sync();
    // ---- controller (thread 0 of every CTA, identical arithmetic)
    if (tid < 32) {
      const double a = sde_partials_sum(p.partials + (size_t)parity * gridDim.x * 4, gridDim.x, 0);
      if (tid == 0) red[0] = a;
    }
    __syncthreads();
    if (tid == 0) {
      const double tot = red[0];
      const float eest = sqrtf((float)(tot / (double)DB));
      C.iter++;
      const int li = C.natt++;
      C.accept = 0; C.npop = 0; C.split = 0; C.push_rem = 0; C.fresh = 0; C.sv_count = 0; C.nmove = 0; C.push_cut = 0;
      if (!isfinite(eest)) {
        C.retcode = LRNDE_RET_UNSTABLE;
        if (blockIdx.x == 0 && li < p.log_cap) { p.log_t[li] = t; p.log_dt[li] = dt; p.log_e[li] = eest; p.log_a[li] = 0; }
        C.accept = -1;
      } else {
        const float q11 = lr_fastpow(eest, p.k.beta1, p.k.pow_mode);
        float q = q11 / lr_fastpow(C.qold, p.k.beta2, p.k.pow_mode);
        q = lr_pymax(1.0f / p.k.qmax, lr_pymin(1.0f / p.k.qmin, q / p.k.gamma));
        const bool acc = eest <= 1.0f;
        if (blockIdx.x == 0 && li < p.log_cap) { p.log_t[li] = t; p.log_dt[li] = dt; p.log_e[li] = eest; p.log_a[li] = acc ? 1 : 0; }
        if (acc) {
          C.accept = 1;
          const float dtnew = dt / q;
          C.qold = lr_pymax(eest, p.k.qoldinit);
          float tnew = t + dt;
          if (fabsf(tnew - p.t2) < 100.0f * lr_spacing(fmaxf(fabsf(t), fabsf(p.t2)))) tnew = p.t2;
          C.tnew = tnew;
          if (blockIdx.x == 0) { p.tape_t[n] = t; p.tape_dt[n] = dt; p.tape_t[n + 1] = tnew; }
          // saves inside (t, tnew]
          C.sv_first = C.next_save;
          while (C.next_save < p.nsave && p.save_t[C.next_save] <= tnew) {
            if (blockIdx.x == 0) {
              const float s = p.save_t[C.next_save];
              p.save_step[C.next_save] = n;
              p.save_theta[C.next_save] = (s == tnew) ? 1.0f : (s - t) / (tnew - t);
            }
            C.next_save++;
          }
          C.sv_count = C.next_save - C.sv_first;
          C.nacc = n + 1;
          C.t = tnew;
          if (tnew < p.t2) {
            float dtn = lr_pymin(lr_pymin(lr_pymax(dtnew, dtmin), dtmax), p.t2 - tnew);
            // RSwM3 accept: plan the pops off the future stack
            C.n2 = 0;
            float dttmp = 0.0f;
            bool done = false;
            while (C.n1 > 0 && !done) {
              const float L = C.L1[C.n1 - 1];
              const float qtmp = (dtn - dttmp) / L;
              if (qtmp > 1.0f) {
                dttmp += L;
                C.n1--; C.npop++;
                if (C.n2 < SDE_STK) C.L2[C.n2] = L; else C.stk_overflow = 1;
                C.n2++;
              } else {
                C.split = 1; C.q_split = qtmp; C.L_split = L; C.draw_split = C.ndraw++;
                C.n1--;
                if ((1.0f - qtmp) * L > p.k.discard) { C.push_rem = 1; C.L1[C.n1] = (1.0f - qtmp) * L; C.n1++; }
                if (C.n2 < SDE_STK) C.L2[C.n2] = qtmp * L; else C.stk_overflow = 1;
                C.n2++;
                dttmp = dtn;
                done = true;
              }
            }
            if (!done) {
              const float left = dtn - dttmp;
              if (left > 0.0f) {
                C.fresh = 1; C.left = left; C.draw_fresh = C.ndraw++;
                if (C.n2 < SDE_STK) C.L2[C.n2] = left; else C.stk_overflow = 1;
                C.n2++;
              }
            }
            C.dt = dtn;
          }
        } else {
          C.nrej++;
          float dtnew = dt / lr_pymin(1.0f / p.k.qmin, q11 / p.k.gamma);
          dtnew = lr_pymin(lr_pymax(dtnew, dtmin), dtmax);
          const float qr = dtnew / dt;
          float dttmp = 0.0f;
          C.n2_before = C.n2;
          while (C.n2 > 0) {
            const float L = C.L2[C.n2 - 1];
            if (dttmp + L < (1.0f - qr) * dt) {
              dttmp += L;
              C.n2--; C.nmove++;
              if (C.n1 < SDE_STK) C.L1[C.n1] = L; else C.stk_overflow = 1;
              C.n1++;
            } else break;
          }
          C.dtK = dt - dttmp;
          C.qK = qr * dt / C.dtK;
          C.draw_rej = C.ndraw++;
          const float cut = (1.0f - C.qK) * C.dtK;
          if (cut > p.k.discard) {
            C.push_cut = 1;
            if (C.n1 < SDE_STK) C.L1[C.n1] = cut; else C.stk_overflow = 1;
            C.n1++;
          }
          C.n2 = 1; C.L2[0] = dtnew;
          C.dt = dtnew;
        }
        if (C.stk_overflow) C.retcode = LRNDE_RET_TAPEFULL;
      }
    }
    __syncthreads();
    parity ^= 1;
    if (C.accept < 0 || C.stk_overflow) break;
    // ---- element-wise phase on the CTA's own slice
    if (C.accept == 1) {
      for (int k = 0; k < C.sv_count; ++k) {
        const int sv = C.sv_first + k;
        const float s = p.save_t[sv];
        float* dst = p.u_save + (size_t)sv * DB;
        if (s == C.tnew) {
          for (size_t e = e_begin + tid; e < e_end; e += nthr) dst[e] = unew[e];
        } else {
          const float th = (s - t) / (C.tnew - t);
          for (size_t e = e_begin + tid; e < e_end; e += nthr) dst[e] = (1.0f - th) * ucur[e] + th * unew[e];
        }
      }
      if (C.t < p.t2) {
        float* nW = p.tape_w + (size_t)(n + 1) * DB;
        float* nZ = p.tape_z + (size_t)(n + 1) * DB;
        // stack indices before this accept: the popped entries were n1_old-1 ... ; reconstruct
        const int n1_after = C.n1;
        const int n1_old = n1_after - C.push_rem + C.split + C.npop;
        for (size_t e = e_begin + tid; e < e_end; e += nthr) {
          float w = 0.0f, z = 0.0f;
          int pos2 = 0;
          for (int j = 0; j < C.npop; ++j) {
            const size_t src = (size_t)(n1_old - 1 - j) * DB + e;
            const float lw = p.S1w[src], lz = p.S1z[src];
            w += lw; z += lz;
            p.S2w[(size_t)pos2 * DB + e] = lw; p.S2z[(size_t)pos2 * DB + e] = lz;
            pos2++;
          }
          if (C.split) {
            const int si = n1_old - 1 - C.npop;
            const size_t src = (size_t)si * DB + e;
            const float lw = p.S1w[src], lz = p.S1z[src];
            const float sd = sqrtf(fmaxf((1.0f - C.q_split) * C.q_split * C.L_split, 0.0f));
            const float bw = C.q_split * lw + sd * sde_normal(p.seed, 0u, (unsigned)C.draw_split, e);
            const float bz = C.q_split * lz + sd * sde_normal(p.seed, 1u, (unsigned)C.draw_split, e);
            w += bw; z += bz;
            if (C.push_rem) { p.S1w[src] = lw - bw; p.S1z[src] = lz - bz; }
            p.S2w[(size_t)pos2 * DB + e] = bw; p.S2z[(size_t)pos2 * DB + e] = bz;
            pos2++;
          }
          if (C.fresh) {
            const float sq = sqrtf(C.left);
            const float bw = sq * sde_normal(p.seed, 0u, (unsigned)C.draw_fresh, e);
            const float bz = sq * sde_normal(p.seed, 1u, (unsigned)C.draw_fresh, e);
            w += bw; z += bz;
            p.S2w[(size_t)pos2 * DB + e] = bw; p.S2z[(size_t)pos2 * DB + e] = bz;
          }
          nW[e] = w; nZ[e] = z;
        }
      }
    } else {
      // reject: S2 tops -> S1, bridge the straddling piece
      const int n1_after = C.n1;
      const int n1_base = n1_after - C.push_cut - C.nmove;  // first S1 slot receiving a moved piece
      const int n2_before = C.n2_before;
      for (size_t e = e_begin + tid; e < e_end; e += nthr) {
        float wt = 0.0f, zt = 0.0f;
        for (int j = 0; j < C.nmove; ++j) {
          const size_t src = (size_t)(n2_before - 1 - j) * DB + e;
          const float lw = p.S2w[src], lz = p.S2z[src];
          wt += lw; zt += lz;
          p.S1w[(size_t)(n1_base + j) * DB + e] = lw; p.S1z[(size_t)(n1_base + j) * DB + e] = lz;
        }
        const float Kw = dWg[e] - wt, Kz = dZg[e] - zt;
        const float sd = sqrtf(fmaxf((1.0f - C.qK) * C.qK * C.dtK, 0.0f));
        const float bw = C.qK * Kw + sd * sde_normal(p.seed, 0u, (unsigned)C.draw_rej, e);
        const float bz = C.qK * Kz + sd * sde_normal(p.seed, 1u, (unsigned)C.draw_rej, e);
        if (C.push_cut) {
          p.S1w[(size_t)(n1_base + C.nmove) * DB + e] = Kw - bw;
          p.S1z[(size_t)(n1_base + C.nmove) * DB + e] = Kz - bz;
        }
        p.S2w[e] = bw; p.S2z[e] = bz;
        dWg[e] = bw; dZg[e] = bz;
      }
    }
    __syncthreads();
  }
  // ---- saves past the end of a failed solve: the last state (oracle: min(s, ts[-1]))
  {
    const float* ulast = p.tape_u + (size_t)C.nacc * DB;
    for (int sv = C.next_save; sv < p.nsave; ++sv) {
      float* dst = p.u_save + (size_t)sv * DB;
      for (size_t e = e_begin + tid; e < e_end; e += nthr) dst[e] = ulast[e];
      if (blockIdx.x == 0 && tid == 0) { p.save_step[sv] = C.nacc - 1; p.save_theta[sv] = 1.0f; }
    }
  }
  if (blockIdx.x == 0 && tid == 0) {
    p.out_i[0] = C.nacc; p.out_i[1] = C.nrej; p.out_i[2] = C.retcode; p.out_i[3] = C.ndraw; p.out_i[4] = C.natt;
    p.out_i[5] = 2 + 4 * C.natt; p.out_i[6] = 2 + 4 * C.natt; p.out_i[7] = C.stk_overflow;
    p.out_f[0] = C.t;
  }
}

// _get_dsde_integrator + _perform_step: auto dt at (u1, t1), fresh increments, one SOSRI step;
// writes dt_reg, EEst and the increments (for the pullback)
__global__ void __launch_bounds__(SDE_THREADS, 1) sde_reg_kernel(SdeSolveP p) {
  cg::grid_group grid = cg::this_grid();
  extern __shared__ __align__(16) float sde_sm[];
  __shared__ double red[32];
  __shared__ float s_dt;
  float *Wf, *Wg, *Gf, *Gg;
  SdeBufs b;
  const int D = p.nf.D;
  sde_carve(sde_sm, p.nf, p.ng, D, p.SP, false, Wf, Wg, Gf, Gg, b);
  const int tid = threadIdx.x, nthr = blockDim.x;
  sde_load_weights(p.nf, p.psf, Wf, tid, nthr);
  sde_load_weights(p.ng, p.psg, Wg, tid, nthr);
  __syncthreads();
  const size_t DB = (size_t)D * p.B;
  const float span = fabsf(p.t2 - p.t1);
  const float dtmin = fmaxf(lr_spacing(p.t1), lr_spacing(p.t2));
  float dt = sde_initdt_coop(p, Wf, Wg, b, p.u1, p.t1, span, 0, red, grid);
  dt = (p.t2 > p.t1) ? fminf(fmaxf(dt, dtmin), span) : dtmin;
  const size_t e_begin = (size_t)blockIdx.x * p.tiles_per_cta * p.S * D;
  const size_t e_end = min(DB, e_begin + (size_t)p.tiles_per_cta * p.S * D);
  const float sq = sqrtf(dt);
  for (size_t e = e_begin + tid; e < e_end; e += nthr) {
    p.reg_w[e] = sq * sde_normal(p.seed, 0u, p.first_draw, e);
    p.reg_z[e] = sq * sde_normal(p.seed, 1u, p.first_draw, e);
  }
  __syncthreads();
  SdeTile T{p.S, p.SP, D, 0, nthr, tid};
  double part = 0.0;
  for (int ti = 0; ti < p.tiles_per_cta; ++ti) {
    const int b0 = (blockIdx.x * p.tiles_per_cta + ti) * p.S;
    if (b0 >= p.B) break;
    T.nvalid = min(p.S, p.B - b0);
    sde_tile_load(b.U, p.u1, b0, T);
    sde_tile_load(b.dW, p.reg_w, b0, T);
    sde_tile_load(b.dZ, p.reg_z, b0, T);
    __syncthreads();
    part += sde_sosri_fwd(p.tab, p.nf, p.ng, Wf, Wg, b, p.t1, dt, p.abstol, p.reltol, p.k.delta, T);
  }
  part = sde_block_sum(part, red);
  // sde_initdt_coop used parities 0 and 1 once each; parity 0 again is safe after its two grid syncs
  if (tid == 0) p.partials[((size_t)0 * gridDim.x + blockIdx.x) * 4 + 2] = part;
  grid.sync();
  if (blockIdx.x == 0 && tid == 0) {
    double tot = 0.0;
    for (unsigned i = 0; i < gridDim.x; ++i) tot += p.partials[(size_t)i * 4 + 2];
    p.out_f[1] = dt;
    p.out_f[2] = sqrtf((float)(tot / (double)DB));
  }
  (void)s_dt;
}

// ---------------------------------------------------------------- reverse pass
struct SdeBwdP {
  SdeNet nf, ng;
  SosriTab tab;
  const float* psf; const float* psg;
  int B, S, SP, tiles_per_cta;
  float abstol, reltol, delta;
  const float* tape_u; const float* tape_w; const float* tape_z; const float* tape_t; const float* tape_dt;
  int nacc;
  const float* d_save; int nsave; const int* save_step; const float* save_theta;  // cotangent blocks
  float* d_x;
  float* gpart;  // [grid][nf.wfloats + ng.wfloats]
  // regulariser
  int with_reg; const float* u1; const float* reg_w; const float* reg_z; float t1, dt_reg, eest_reg, d_reg;
};

__global__ void __launch_bounds__(SDE_THREADS, 1) sde_backward_kernel(SdeBwdP p) {
  extern __shared__ __align__(16) float sde_sm[];
  float *Wf, *Wg, *Gf, *Gg;
  SdeBufs b;
  const int D = p.nf.D;
  sde_carve(sde_sm, p.nf, p.ng, D, p.SP, true, Wf, Wg, Gf, Gg, b);
  const int tid = threadIdx.x, nthr = blockDim.x;
  sde_load_weights(p.nf, p.psf, Wf, tid, nthr);
  sde_load_weights(p.ng, p.psg, Wg, tid, nthr);
  for (int e = tid; e < p.nf.wfloats; e += nthr) Gf[e] = 0.0f;
  for (int e = tid; e < p.ng.wfloats; e += nthr) Gg[e] = 0.0f;
  __syncthreads();
  const size_t DB = (size_t)D * p.B;
  SdeTile T{p.S, p.SP, D, 0, nthr, tid};
  for (int ti = 0; ti < p.tiles_per_cta; ++ti) {
    const int b0 = (blockIdx.x * p.tiles_per_cta + ti) * p.S;
    if (b0 >= p.B) break;
    T.nvalid = min(p.S, p.B - b0);
    // b.cot carries the cotangent of state n+1 while step n is reversed
    for (int idx = tid; idx < D * T.S; idx += nthr) b.cot[(idx / T.S) * T.SP + (idx % T.S)] = 0.0f;
    __syncthreads();
    for (int n = p.nacc - 1; n >= 0; --n) {
      // saves interpolated inside step n: theta to state n+1
      for (int k = 0; k < p.nsave; ++k)
        if (p.save_step[k] == n) {
          const float th = p.save_theta[k];
          const float* dk = p.d_save + (size_t)k * DB;
          for (int idx = tid; idx < D * T.S; idx += nthr) {
            const int s = idx / D, d = idx % D;
            if (s < T.nvalid) b.cot[d * T.SP + s] += th * dk[(size_t)(b0 + s) * D + d];
          }
        }
      sde_tile_load(b.U, p.tape_u + (size_t)n * DB, b0, T);
      sde_tile_load(b.dW, p.tape_w + (size_t)n * DB, b0, T);
      sde_tile_load(b.dZ, p.tape_z + (size_t)n * DB, b0, T);
      __syncthreads();
      sde_sosri_bwd(p.tab, p.nf, p.ng, Wf, Wg, Gf, Gg, b, p.tape_t[n], p.tape_dt[n], false, T);
      // cotangent of state n: from the step + (1 - theta) shares of the saves inside step n
      for (int idx = tid; idx < D * T.S; idx += nthr) {
        const int a = (idx / T.S) * T.SP + (idx % T.S);
        b.cot[a] = b.Ub[a];
      }
      __syncthreads();
      for (int k = 0; k < p.nsave; ++k)
        if (p.save_step[k] == n && p.save_theta[k] != 1.0f) {
          const float th = 1.0f - p.save_theta[k];
          const float* dk = p.d_save + (size_t)k * DB;
          for (int idx = tid; idx < D * T.S; idx += nthr) {
            const int s = idx / D, d = idx % D;
            if (s < T.nvalid) b.cot[d * T.SP + s] += th * dk[(size_t)(b0 + s) * D + d];
          }
        }
      __syncthreads();
    }
    // saves at t0 (save_step == -1)
    for (int k = 0; k < p.nsave; ++k)
      if (p.save_step[k] < 0) {
        const float* dk = p.d_save + (size_t)k * DB;
        for (int idx = tid; idx < D * T.S; idx += nthr) {
          const int s = idx / D, d = idx % D;
          if (s < T.nvalid) b.cot[d * T.SP + s] += dk[(size_t)(b0 + s) * D + d];
        }
      }
    __syncthreads();
    if (p.d_x) sde_tile_store(p.d_x, b.cot, b0, T);
    __syncthreads();
    // ---- regulariser pullback (parameters only)
    if (p.with_reg) {
      sde_tile_load(b.U, p.u1, b0, T);
      sde_tile_load(b.dW, p.reg_w, b0, T);
      sde_tile_load(b.dZ, p.reg_z, b0, T);
      __syncthreads();
      (void)sde_sosri_fwd(p.tab, p.nf, p.ng, Wf, Wg, b, p.t1, p.dt_reg, p.abstol, p.reltol, p.delta, T);
      const float dt = p.dt_reg, sqdt = sqrtf(fabsf(dt));
      const float nn = (float)DB;
      for (int idx = tid; idx < D * T.S; idx += nthr) {
        const int s = idx % T.S, a = (idx / T.S) * T.SP + s;
        float chi1, chi2, chi3;
        sde_chi(b.dW[a], b.dZ[a], dt, sqdt, chi1, chi2, chi3);
        const SosriTab& c = p.tab;
        const float g1 = b.g[0][a], g2 = b.g[1][a], g3 = b.g[2][a], g4 = b.g[3][a];
        const float E2 = chi2 * (c.be31 * g1 + c.be32 * g2 + c.be33 * g3 + c.be34 * g4) +
                         chi3 * (c.be41 * g1 + c.be42 * g2 + c.be43 * g3 + c.be44 * g4);
        const float E1 = dt * (b.k[0][a] + b.k[1][a] + b.k[2][a] + b.k[3][a]);
        const float up = b.U[a], u = b.un[a];
        const float sc = p.abstol + fmaxf(fabsf(up), fabsf(u)) * p.reltol;
        const float r = (p.delta * E1 + E2) / sc;
        float rbar = 0.0f;
        if (s < T.nvalid && p.eest_reg > 0.0f) rbar = (p.d_reg * dt) * r / (nn * p.eest_reg);
        b.E1b[a] = p.delta * rbar / sc;
        b.E2b[a] = rbar / sc;
        const float scbar = -rbar * r / sc;
        const float sg = (u > 0.0f) ? 1.0f : ((u < 0.0f) ? -1.0f : 0.0f);
        b.cot[a] = (fabsf(u) > fabsf(up)) ? scbar * p.reltol * sg : 0.0f;
      }
      __syncthreads();
      sde_sosri_bwd(p.tab, p.nf, p.ng, Wf, Wg, Gf, Gg, b, p.t1, dt, true, T);
    }
  }
  float* mine = p.gpart + (size_t)blockIdx.x * (p.nf.wfloats + p.ng.wfloats);
  for (int e = tid; e < p.nf.wfloats; e += nthr) mine[e] = Gf[e];
  for (int e = tid; e < p.ng.wfloats; e += nthr) mine[p.nf.wfloats + e] = Gg[e];
}

// fixed-order sum of the per-CTA partial gradients, un-padded into the flat parameter layout (one thread per
// padded element; `stride` = floats per CTA record, `base` = offset of this network inside the record)
__global__ void sde_grad_reduce_kernel(SdeNet n, const float* gpart, int stride, int base, int nblk, float* d_ps) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n.wfloats; e += gridDim.x * blockDim.x) {
    int l = 0;
    while (l + 1 < n.nl && e >= n.w_off[l + 1]) ++l;
    const int loc = e - n.w_off[l];
    const int rows = n.in[l] + n.td + 1, outp = n.outp[l], out = n.out[l];
    const int i = loc / outp, r = loc % outp;
    if (r >= out) continue;
    float acc = 0.0f;
#pragma unroll 8
    for (int bb = 0; bb < nblk; ++bb) acc += gpart[(size_t)bb * stride + base + e];
    if (i < rows - 1) d_ps[n.ps_w[l] + (long long)i * out + r] = acc;
    else d_ps[n.ps_b[l] + r] = acc;
  }
}

// ---------------------------------------------------------------- the other in-tree SDE steps
// _perform_step(::RKMilCommuteConstantCache) (perform_step.jl:108-170) and
// _perform_step(::LambaEulerHeunConstantCache) (:172-206), diagonal noise, Ito, injected dW.
// kind 0 = RKMilCommute (quirk kept: the drift/noise error of :162-163 is overwritten at :165 and
// EEst is the RMS of the relative CHANGE), kind 1 = LambaEulerHeun.
struct SdeAuxP {
  SdeNet nf, ng;
  const float* psf; const float* psg;
  int B, S, SP, tiles_per_cta, kind;
  float t, dt, abstol, reltol, delta;
  const float* uprev; const float* dW; float* u; double* partials;
};

__global__ void __launch_bounds__(SDE_THREADS, 1) sde_aux_step_kernel(SdeAuxP p) {
  extern __shared__ __align__(16) float sde_sm[];
  __shared__ double red[32];
  float *Wf, *Wg, *Gf, *Gg;
  SdeBufs b;
  const int D = p.nf.D;
  sde_carve(sde_sm, p.nf, p.ng, D, p.SP, false, Wf, Wg, Gf, Gg, b);
  const int tid = threadIdx.x, nthr = blockDim.x;
  sde_load_weights(p.nf, p.psf, Wf, tid, nthr);
  sde_load_weights(p.ng, p.psg, Wg, tid, nthr);
  __syncthreads();
  SdeTile T{p.S, p.SP, D, 0, nthr, tid};
  const float t = p.t, dt = p.dt, sqdt = sqrtf(fabsf(dt));
  double part = 0.0;
  for (int ti = 0; ti < p.tiles_per_cta; ++ti) {
    const int b0 = (blockIdx.x * p.tiles_per_cta + ti) * p.S;
    if (b0 >= p.B) break;
    T.nvalid = min(p.S, p.B - b0);
    sde_tile_load(b.U, p.uprev, b0, T);
    sde_tile_load(b.dW, p.dW, b0, T);
    __syncthreads();
    sde_mlp_fwd(p.nf, Wf, b.U, t, b.k[0], b.pre, b.post, T);   // du1
    sde_mlp_fwd(p.ng, Wg, b.U, t, b.g[0], b.pre, b.post, T);   // L
    for (int idx = tid; idx < D * T.S; idx += nthr) {
      const int a = (idx / T.S) * T.SP + (idx % T.S);
      const float K = b.U[a] + dt * b.k[0][a];
      b.H0[a] = K;
      b.H1[a] = (p.kind == 0) ? K + sqdt * b.g[0][a] : K + b.g[0][a] * b.dW[a];
    }
    __syncthreads();
    if (p.kind == 0) {
      sde_mlp_fwd(p.ng, Wg, b.H1, t, b.g[1], b.pre, b.post, T);        // gtmp
      sde_mlp_fwd(p.nf, Wf, b.H0, t + dt, b.k[1], b.pre, b.post, T);   // du2 (evaluated, unused: quirk)
      for (int idx = tid; idx < D * T.S; idx += nthr) {
        const int s = idx % T.S, a = (idx / T.S) * T.SP + s;
        const float dW = b.dW[a], L = b.g[0][a];
        const float J = dW * dW / 2.0f - 0.5f * fabsf(dt);
        const float Dgj = (b.g[1][a] - L) / sqdt;
        const float u = b.H0[a] + L * dW + Dgj * J;
        b.un[a] = u;
        if (s < T.nvalid) {
          const float up = b.U[a];
          const float r = (u - up) / (p.abstol + fmaxf(fabsf(up), fabsf(u)) * p.reltol);
          part += (double)r * r;
        }
      }
    } else {
      sde_mlp_fwd(p.ng, Wg, b.H1, t + dt, b.g[1], b.pre, b.post, T);   // g(tmp, t+dt)
      sde_mlp_fwd(p.nf, Wf, b.H1, t + dt, b.k[1], b.pre, b.post, T);   // f(tmp, t+dt)
      sde_mlp_fwd(p.nf, Wf, b.H0, t + dt, b.k[2], b.pre, b.post, T);   // du2
      for (int idx = tid; idx < D * T.S; idx += nthr) {
        const int a = (idx / T.S) * T.SP + (idx % T.S);
        b.H1[a] = b.U[a] + b.g[0][a] * sqdt;                           // utilde
      }
      __syncthreads();
      sde_mlp_fwd(p.ng, Wg, b.H1, t, b.g[2], b.pre, b.post, T);
      for (int idx = tid; idx < D * T.S; idx += nthr) {
        const int s = idx % T.S, a = (idx / T.S) * T.SP + s;
        const float dW = b.dW[a], L = b.g[0][a], up = b.U[a];
        const float gtmp2 = 0.5f * (L + b.g[1][a]);
        const float u = up + (dt / 2.0f) * (b.k[0][a] + b.k[1][a]) + gtmp2 * dW;
        b.un[a] = u;
        if (s < T.nvalid) {
          const float Ed = dt * (b.k[2][a] - b.k[0][a]) / 2.0f;
          const float En = ((b.g[2][a] - L) / sqdt) * (dW * dW) / 2.0f;
          const float r = (p.delta * Ed + En) / (p.abstol + fmaxf(fabsf(up), fabsf(u)) * p.reltol);
          part += (double)r * r;
        }
      }
    }
    __syncthreads();
    sde_tile_store(p.u, b.un, b0, T);
    __syncthreads();
  }
  part = sde_block_sum(part, red);
  if (tid == 0) p.partials[blockIdx.x] = part;
}

// ==========================================================================================
// Host side: C ABI (include/lrnde.h, "Neural SDE" section)
// ==========================================================================================
struct lrnde_sde_tape {
  lrnde_ctx* ctx = nullptr;
  SdeNet nf, ng;
  SdeConsts k;
  SosriTab tab;
  lrnde_sde_opts opts;
  int64_t B = 0;
  int S = 32, SP = 33, tiles_per_cta = 1, grid = 1;
  float *psf = nullptr, *psg = nullptr;
  float *tape_u = nullptr, *tape_w = nullptr, *tape_z = nullptr, *tape_t = nullptr, *tape_dt = nullptr;
  float *S1w = nullptr, *S1z = nullptr, *S2w = nullptr, *S2z = nullptr;
  float *save_t = nullptr, *save_theta = nullptr, *u_save_dev = nullptr, *u1 = nullptr, *reg_w = nullptr,
        *reg_z = nullptr, *log_t = nullptr, *log_dt = nullptr, *log_e = nullptr, *out_f = nullptr;
  int *save_step = nullptr, *out_i = nullptr;
  unsigned char* log_a = nullptr;
  double* partials = nullptr;
  int cap = 0, nacc = 0, natt = 0, nsave_dev = 0, log_cap = 0;
  bool all_steps = false, with_reg = false;
  float t1 = 0.f, dt_reg = 0.f, eest_reg = 0.f;
  std::vector<float> step_t;  // host copy of the accepted step times (nacc + 1)
  std::vector<void*> owned;
  template <typename Tp> Tp* take(size_t n) {
    Tp* p = (Tp*)ctx->alloc(sizeof(Tp) * std::max<size_t>(n, 1));
    owned.push_back(p);
    return p;
  }
  ~lrnde_sde_tape() { for (void* p : owned) ctx->release(p); }
};

static SdeNet sde_make_net(const lrnde_model* m, const char* what) {
  SdeNet n;
  memset(&n, 0, sizeof(n));
  if ((int)m->layers.size() > SDE_MAXL) lr_fail(LRNDE_EINVAL, "%s: at most %d layers on the SDE path", what, SDE_MAXL);
  if (m->input_act != ACT_IDENTITY) lr_fail(LRNDE_EINVAL, "%s: input activation is not supported on the SDE path", what);
  n.nl = (int)m->layers.size(); n.td = m->td; n.D = m->D; n.nparams = (int)m->nparams;
  int woff = 0, hoff = 0, md = m->D;
  for (int l = 0; l < n.nl; ++l) {
    const LayerInfo& L = m->layers[l];
    n.in[l] = L.in; n.out[l] = L.out; n.outp[l] = (L.out + 3) & ~3; n.act[l] = L.act;
    n.ps_w[l] = L.w_off; n.ps_b[l] = L.b_off;
    n.w_off[l] = woff; woff += (L.in + m->td + 1) * n.outp[l];
    n.hid_off[l] = hoff; hoff += n.outp[l];
    md = std::max(md, std::max(L.in, n.outp[l]));
  }
  n.wfloats = woff; n.hid_rows = hoff; n.maxdim = md;
  return n;
}

static SdeConsts sde_make_consts(const lrnde_sde_opts* o) {
  SdeConsts k;
  k.order = 1.5f;
  k.beta1 = (float)(7.0 / (10.0 * 1.5)); k.beta2 = (float)(2.0 / (5.0 * 1.5));
  k.gamma = o->gamma > 0.f ? o->gamma : 0.9f;
  k.qmin = o->qmin > 0.f ? o->qmin : 0.2f;
  k.qmax = o->qmax > 0.f ? o->qmax : 1.125f;
  k.qoldinit = 1e-4f;
  k.delta = o->delta > 0.f ? o->delta : (float)(1.0 / 6.0);
  k.discard = 1e-15f;
  k.pow_mode = o->pow_mode;
  return k;
}

static void sde_fill_solve_params(SdeSolveP& p, lrnde_sde_tape& T) {
  memset(&p, 0, sizeof(p));
  p.nf = T.nf; p.ng = T.ng; p.k = T.k; p.tab = T.tab;
  p.psf = T.psf; p.psg = T.psg;
  p.B = (int)T.B; p.S = T.S; p.SP = T.SP; p.tiles_per_cta = T.tiles_per_cta;
  p.t0 = T.opts.t0; p.t2 = T.opts.t2; p.abstol = T.opts.abstol; p.reltol = T.opts.reltol;
  p.maxiters = T.opts.maxiters; p.seed = T.opts.seed; p.first_draw = 0;
  p.tape_u = T.tape_u; p.tape_w = T.tape_w; p.tape_z = T.tape_z; p.tape_t = T.tape_t; p.tape_dt = T.tape_dt;
  p.cap = T.cap;
  p.S1w = T.S1w; p.S1z = T.S1z; p.S2w = T.S2w; p.S2z = T.S2z;
  p.save_t = T.save_t; p.nsave = T.nsave_dev; p.u_save = T.u_save_dev; p.save_step = T.save_step;
  p.save_theta = T.save_theta;
  p.partials = T.partials;
  p.log_t = T.log_t; p.log_dt = T.log_dt; p.log_e = T.log_e; p.log_a = T.log_a; p.log_cap = T.log_cap;
  p.out_i = T.out_i; p.out_f = T.out_f;
  p.u1 = T.u1; p.t1 = T.t1; p.reg_w = T.reg_w; p.reg_z = T.reg_z;
}

extern "C" int lrnde_sde_forward(lrnde_ctx* ctx, const lrnde_model* drift, const lrnde_model* diffusion,
                                 const lrnde_sde_opts* o, const float* ps_drift, const float* ps_diffusion,
                                 const float* x, int64_t B, float* u_save, lrnde_sde_stats* stats,
                                 lrnde_sde_tape** tape_out) {
  LR_API_BEGIN
  if (!ctx || !drift || !diffusion || !o || !ps_drift || !ps_diffusion || !x || !stats || B < 1)
    lr_fail(LRNDE_EINVAL, "lrnde_sde_forward: bad args");
  if (o->reg_mode < LRNDE_REG_NONE || o->reg_mode > LRNDE_REG_BIASED)
    lr_fail(LRNDE_EINVAL, "regularize must be one of (:none, :unbiased, :biased)");  // utils.jl:53-58
  if (drift->D != diffusion->D) lr_fail(LRNDE_EINVAL, "drift and diffusion act on different state sizes");
  if (!(o->t2 > o->t0)) lr_fail(LRNDE_EINVAL, "tspan must be increasing");
  if (o->keep_tape && !tape_out) lr_fail(LRNDE_EINVAL, "keep_tape set but tape is NULL");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  memset(stats, 0, sizeof(*stats));
  const long launches0 = ctx->launches;
  auto T = std::make_unique<lrnde_sde_tape>();
  T->ctx = ctx;
  T->nf = sde_make_net(drift, "drift");
  T->ng = sde_make_net(diffusion, "diffusion");
  T->k = sde_make_consts(o);
  T->tab = lr_sosri_tab();
  T->opts = *o;
  T->opts.saveat = nullptr;
  T->B = B;
  const int D = drift->D;
  const size_t DB = (size_t)D * (size_t)B;
  CallerBufs io(ctx, o->host_buffers);

  // ---- launch shape: S samples per tile, one CTA per SM at most (cooperative launch)
  int n_sm = 0;
  size_t smem_optin = 0;
  sde_device_limits(ctx->device, &n_sm, &smem_optin);
  int S = 32;
  while (S > 8 && ((B + S - 1) / S) < n_sm / 2) S >>= 1;
  size_t smem_f = 0, smem_b = 0;
  for (;; S >>= 1) {
    smem_f = sde_smem_bytes(T->nf, T->ng, D, S + 1, false);
    smem_b = sde_smem_bytes(T->nf, T->ng, D, S + 1, true);
    if (smem_b <= smem_optin) break;
    if (S <= 4) lr_fail(LRNDE_EINVAL, "SDE networks / state too large for the shared-memory resident path (%zu bytes)", smem_b);
  }
  T->S = S; T->SP = S + 1;
  const int ntiles = (int)((B + S - 1) / S);
  LR_CUDA(cudaFuncSetAttribute(sde_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_f));
  LR_CUDA(cudaFuncSetAttribute(sde_reg_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_f));
  const int max_grid = n_sm;   // __launch_bounds__(SDE_THREADS, 1): one CTA per SM is always co-resident
  T->tiles_per_cta = (ntiles + max_grid - 1) / max_grid;
  T->grid = (ntiles + T->tiles_per_cta - 1) / T->tiles_per_cta;

  // ---- buffers
  const int64_t Pf = drift->nparams, Pg = diffusion->nparams;
  T->psf = T->take<float>(Pf);
  T->psg = T->take<float>(Pg);
  io.copy_in(T->psf, ps_drift, Pf);   // kept by the tape
  io.copy_in(T->psg, ps_diffusion, Pg);
  size_t budget = (size_t)8 << 30;
  int cap = (int)std::min<size_t>((size_t)o->maxiters, std::max<size_t>(64, budget / (3 * DB * sizeof(float))));
  cap = std::max(cap, 1);
  T->cap = cap;
  T->tape_u = T->take<float>((size_t)(cap + 1) * DB);
  T->tape_w = T->take<float>((size_t)(cap + 1) * DB);
  T->tape_z = T->take<float>((size_t)(cap + 1) * DB);
  T->tape_t = T->take<float>(cap + 2);
  T->tape_dt = T->take<float>(cap + 2);
  T->S1w = T->take<float>((size_t)SDE_STK * DB); T->S1z = T->take<float>((size_t)SDE_STK * DB);
  T->S2w = T->take<float>((size_t)SDE_STK * DB); T->S2z = T->take<float>((size_t)SDE_STK * DB);
  T->partials = T->take<double>((size_t)2 * T->grid * 4);
  T->log_cap = o->maxiters + 1;
  T->log_t = T->take<float>(T->log_cap); T->log_dt = T->take<float>(T->log_cap);
  T->log_e = T->take<float>(T->log_cap); T->log_a = T->take<unsigned char>(T->log_cap);
  T->out_i = T->take<int>(8); T->out_f = T->take<float>(4);
  LR_CUDA(cudaMemsetAsync(T->out_i, 0, sizeof(int) * 8, st));
  io.copy_in(T->tape_u, x, DB);   // u_0, the first state of the tape

  // ---- save times
  std::vector<float> times;
  T->all_steps = (o->nsave < 0);
  if (o->nsave > 0) {
    if (!o->saveat) lr_fail(LRNDE_EINVAL, "nsave > 0 but saveat is NULL");
    times.assign(o->saveat, o->saveat + o->nsave);
    for (size_t i = 1; i < times.size(); ++i)
      if (!(times[i] >= times[i - 1])) lr_fail(LRNDE_EINVAL, "saveat must be sorted");
  } else if (o->nsave == 0) times.push_back(o->t2);
  T->nsave_dev = (int)times.size();
  T->save_t = T->take<float>(times.size());
  T->save_step = T->take<int>(times.size());
  T->save_theta = T->take<float>(times.size());
  T->u_save_dev = T->take<float>(times.size() * DB);
  if (!times.empty()) LR_CUDA(cudaMemcpyAsync(T->save_t, times.data(), sizeof(float) * times.size(), cudaMemcpyHostToDevice, st));

  // ---- the solve: one cooperative launch
  SdeSolveP p;
  sde_fill_solve_params(p, *T);
  {
    void* args[] = {&p};
    LR_CUDA(cudaLaunchCooperativeKernel((void*)sde_solve_kernel, dim3(T->grid), dim3(SDE_THREADS), args, smem_f, st));
    LR_COUNT(ctx);
  }
  int oi[8]; float of[4];
  LR_CUDA(cudaMemcpyAsync(oi, T->out_i, sizeof(oi), cudaMemcpyDeviceToHost, st));
  LR_CUDA(cudaMemcpyAsync(of, T->out_f, sizeof(of), cudaMemcpyDeviceToHost, st));
  LR_CUDA(cudaStreamSynchronize(st));
  T->nacc = oi[0]; T->natt = oi[4];
  stats->naccept = oi[0]; stats->nreject = oi[1]; stats->retcode = oi[2]; stats->ndraws = oi[3];
  stats->nfe_drift = oi[5]; stats->nfe_diffusion = oi[6];
  T->step_t.assign(T->nacc + 1, o->t0);
  if (T->nacc > 0)
    LR_CUDA(cudaMemcpy(T->step_t.data(), T->tape_t, sizeof(float) * (T->nacc + 1), cudaMemcpyDeviceToHost));
  T->step_t[0] = o->t0;

  // ---- regulariser (training only; the caller passes LRNDE_REG_NONE in eval mode)
  stats->t1_used = o->t0;
  if (o->reg_mode != LRNDE_REG_NONE) {
    float t1 = o->t1;
    const float* u1src = nullptr;
    if (o->reg_mode == LRNDE_REG_UNBIASED) {
      int k1 = -1;
      for (size_t i = 0; i < times.size(); ++i) if (times[i] == t1) { k1 = (int)i; break; }
      if (k1 < 0) lr_fail(LRNDE_EINVAL, "unbiased: t1 must be one of the saveat times (neural_sde.jl:90-91)");
      u1src = T->u_save_dev + (size_t)k1 * DB;
    } else {
      // t1 = rand(rng, sol.t[1:end-1]) (neural_sde.jl:112): index = floor(u01 * ncand)
      if (T->all_steps) {
        const int start = o->save_start ? 0 : 1;
        const int ncand = T->nacc + 1 - start - 1;
        if (ncand > 0) {
          const int idx = start + std::min(ncand - 1, std::max(0, (int)std::floor(o->u01 * (float)ncand)));
          t1 = T->step_t[idx];
          u1src = T->tape_u + (size_t)idx * DB;
        } else { t1 = o->t0; u1src = T->tape_u; }
      } else {
        const int ncand = (int)times.size() - 1;
        if (ncand > 0) {
          const int idx = std::min(ncand - 1, std::max(0, (int)std::floor(o->u01 * (float)ncand)));
          t1 = times[idx];
          u1src = T->u_save_dev + (size_t)idx * DB;
        } else { t1 = o->t0; u1src = T->tape_u; }
      }
    }
    T->u1 = T->take<float>(DB);
    T->reg_w = T->take<float>(DB);
    T->reg_z = T->take<float>(DB);
    LR_CUDA(cudaMemcpyAsync(T->u1, u1src, sizeof(float) * DB, cudaMemcpyDeviceToDevice, st));
    T->t1 = t1;
    sde_fill_solve_params(p, *T);
    p.first_draw = (unsigned)stats->ndraws;
    void* args[] = {&p};
    LR_CUDA(cudaLaunchCooperativeKernel((void*)sde_reg_kernel, dim3(T->grid), dim3(SDE_THREADS), args, smem_f, st));
    LR_COUNT(ctx);
    LR_CUDA(cudaMemcpyAsync(of, T->out_f, sizeof(of), cudaMemcpyDeviceToHost, st));
    LR_CUDA(cudaStreamSynchronize(st));
    T->dt_reg = of[1]; T->eest_reg = of[2];
    T->with_reg = true;
    stats->reg_val = T->eest_reg * T->dt_reg;   // perform_step.jl:105: EEst * dt
    stats->dt_reg = T->dt_reg;
    stats->t1_used = t1;
    stats->ndraws += 1;
    stats->nfe_drift += 2 + 4; stats->nfe_diffusion += 2 + 4;  // the closures count the integrator's calls too
  }

  // ---- outputs
  stats->nsave_out = T->all_steps ? (T->nacc + (o->save_start ? 1 : 0)) : (int)times.size();
  if (!times.empty()) io.copy_out(u_save, T->u_save_dev, times.size() * DB);
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  stats->gpu_launches = (int32_t)(ctx->launches - launches0);
  if (o->keep_tape) *tape_out = T.release();
  LR_API_END
}

extern "C" int lrnde_sde_states(lrnde_ctx* ctx, const lrnde_sde_tape* T, int32_t first, int32_t count,
                                int32_t host_buffers, float* u_out, float* t_out) {
  LR_API_BEGIN
  if (!ctx || !T || first < 0 || count < 0 || first + count > T->nacc + 1)
    lr_fail(LRNDE_EINVAL, "lrnde_sde_states: range outside the %d stored states", T ? T->nacc + 1 : 0);
  const size_t DB = (size_t)T->nf.D * (size_t)T->B;
  CallerBufs io(ctx, host_buffers);
  if (count) io.copy_out(u_out, T->tape_u + (size_t)first * DB, DB * count);
  io.finish();
  if (t_out) for (int i = 0; i < count; ++i) t_out[i] = T->step_t[first + i];
  LR_CUDA(cudaStreamSynchronize(ctx->stream));
  LR_API_END
}

extern "C" int lrnde_sde_step_log(const lrnde_sde_tape* T, float* t, float* dt, float* eest, uint8_t* accepted,
                                  int32_t cap, int32_t* n) {
  LR_API_BEGIN
  if (!T || !n) lr_fail(LRNDE_EINVAL, "lrnde_sde_step_log: bad args");
  *n = T->natt;
  const int k = std::min<int>(cap, std::min(T->natt, T->log_cap));
  if (k > 0 && t) LR_CUDA(cudaMemcpy(t, T->log_t, sizeof(float) * k, cudaMemcpyDeviceToHost));
  if (k > 0 && dt) LR_CUDA(cudaMemcpy(dt, T->log_dt, sizeof(float) * k, cudaMemcpyDeviceToHost));
  if (k > 0 && eest) LR_CUDA(cudaMemcpy(eest, T->log_e, sizeof(float) * k, cudaMemcpyDeviceToHost));
  if (k > 0 && accepted) LR_CUDA(cudaMemcpy(accepted, T->log_a, k, cudaMemcpyDeviceToHost));
  LR_API_END
}

extern "C" int lrnde_sde_backward(lrnde_ctx* ctx, lrnde_sde_tape* T, const float* d_u_save, float d_reg,
                                  float* d_ps_drift, float* d_ps_diffusion, float* d_x) {
  LR_API_BEGIN
  if (!ctx || !T || !d_ps_drift || !d_ps_diffusion) lr_fail(LRNDE_EINVAL, "lrnde_sde_backward: bad args");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int D = T->nf.D;
  const size_t DB = (size_t)D * (size_t)T->B;
  CallerBufs io(ctx, T->opts.host_buffers);
  // cotangent blocks: one per saved state (all-steps mode: one per returned state, in order)
  int nblk = T->all_steps ? (T->nacc + (T->opts.save_start ? 1 : 0)) : T->nsave_dev;
  std::vector<int> step(std::max(nblk, 1));
  std::vector<float> theta(std::max(nblk, 1), 1.0f);
  const int* step_dev = T->save_step;
  const float* theta_dev = T->save_theta;
  DevBuf dsave(ctx, std::max<size_t>(1, (size_t)nblk * DB));   // the kernel reads a zero block for a NULL d_u_save
  if (d_u_save && nblk) io.copy_in(dsave.p, d_u_save, (size_t)nblk * DB);
  else if (nblk) LR_CUDA(cudaMemsetAsync(dsave.p, 0, sizeof(float) * nblk * DB, st));
  DevBuf stepb(ctx, nblk + 1), thetab(ctx, nblk + 1);
  if (T->all_steps) {
    const int off = T->opts.save_start ? 1 : 0;   // block k is state k + 1 - off = end of step k - off
    for (int k = 0; k < nblk; ++k) step[k] = k - off;
    LR_CUDA(cudaMemcpyAsync(stepb.p, step.data(), sizeof(int) * nblk, cudaMemcpyHostToDevice, st));
    LR_CUDA(cudaMemcpyAsync(thetab.p, theta.data(), sizeof(float) * nblk, cudaMemcpyHostToDevice, st));
    step_dev = (const int*)stepb.p;
    theta_dev = thetab.p;
  }
  const size_t smem_b = sde_smem_bytes(T->nf, T->ng, D, T->SP, true);
  LR_CUDA(cudaFuncSetAttribute(sde_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
  const int gstride = T->nf.wfloats + T->ng.wfloats;
  DevBuf gpart(ctx, (size_t)T->grid * gstride);
  DevBuf dx(ctx, DB);   // the kernel always writes d_x
  float* dpf = io.copy_out(d_ps_drift, T->nf.nparams);
  float* dpg = io.copy_out(d_ps_diffusion, T->ng.nparams);
  io.copy_out(d_x, dx.p, DB);
  SdeBwdP q;
  memset(&q, 0, sizeof(q));
  q.nf = T->nf; q.ng = T->ng; q.tab = T->tab; q.psf = T->psf; q.psg = T->psg;
  q.B = (int)T->B; q.S = T->S; q.SP = T->SP; q.tiles_per_cta = T->tiles_per_cta;
  q.abstol = T->opts.abstol; q.reltol = T->opts.reltol; q.delta = T->k.delta;
  q.tape_u = T->tape_u; q.tape_w = T->tape_w; q.tape_z = T->tape_z; q.tape_t = T->tape_t; q.tape_dt = T->tape_dt;
  q.nacc = T->nacc;
  q.d_save = dsave.p; q.nsave = nblk; q.save_step = step_dev; q.save_theta = theta_dev;
  q.d_x = dx.p; q.gpart = gpart.p;
  q.with_reg = (T->with_reg && d_reg != 0.0f) ? 1 : 0;
  q.u1 = T->u1; q.reg_w = T->reg_w; q.reg_z = T->reg_z; q.t1 = T->t1; q.dt_reg = T->dt_reg;
  q.eest_reg = T->eest_reg; q.d_reg = d_reg;
  sde_backward_kernel<<<T->grid, SDE_THREADS, smem_b, st>>>(q);
  LR_COUNT(ctx);
  sde_grad_reduce_kernel<<<64, 256, 0, st>>>(T->nf, gpart.p, gstride, 0, T->grid, dpf);
  LR_COUNT(ctx);
  sde_grad_reduce_kernel<<<64, 256, 0, st>>>(T->ng, gpart.p, gstride, T->nf.wfloats, T->grid, dpg);
  LR_COUNT(ctx);
  LR_CUDA(cudaGetLastError());
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  LR_API_END
}

extern "C" int lrnde_sde_tape_free(lrnde_sde_tape* T) {
  LR_API_BEGIN
  delete T;
  LR_API_END
}

extern "C" int lrnde_sde_aux_step(lrnde_ctx* ctx, const lrnde_model* drift, const lrnde_model* diffusion,
                                  int32_t kind, const float* ps_drift, const float* ps_diffusion,
                                  const float* uprev, const float* dW, float t, float dt, float abstol,
                                  float reltol, float delta, int64_t B, int32_t host_buffers, float* u,
                                  float* reg_val) {
  LR_API_BEGIN
  if (!ctx || !drift || !diffusion || !ps_drift || !ps_diffusion || !uprev || !dW || !u || !reg_val || B < 1)
    lr_fail(LRNDE_EINVAL, "lrnde_sde_aux_step: bad args");
  if (kind != LRNDE_SDESTEP_RKMIL && kind != LRNDE_SDESTEP_LAMBA_EULER_HEUN)
    lr_fail(LRNDE_EINVAL, "kind must be LRNDE_SDESTEP_RKMIL or LRNDE_SDESTEP_LAMBA_EULER_HEUN");
  if (drift->D != diffusion->D) lr_fail(LRNDE_EINVAL, "drift and diffusion act on different state sizes");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  SdeAuxP p;
  memset(&p, 0, sizeof(p));
  p.nf = sde_make_net(drift, "drift");
  p.ng = sde_make_net(diffusion, "diffusion");
  const int D = drift->D;
  const size_t DB = (size_t)D * (size_t)B;
  int n_sm = 0;
  size_t smem_optin = 0;
  sde_device_limits(ctx->device, &n_sm, &smem_optin);
  int S = 32;
  while (S > 8 && ((B + S - 1) / S) < n_sm / 2) S >>= 1;
  size_t smem = 0;
  for (;; S >>= 1) {
    smem = sde_smem_bytes(p.nf, p.ng, D, S + 1, false);
    if (smem <= smem_optin) break;
    if (S <= 4) lr_fail(LRNDE_EINVAL, "SDE networks / state too large for the shared-memory resident path");
  }
  const int ntiles = (int)((B + S - 1) / S);
  const int max_grid = 4 * n_sm;
  p.S = S; p.SP = S + 1; p.B = (int)B; p.kind = kind;
  p.tiles_per_cta = (ntiles + max_grid - 1) / max_grid;
  const int grid = (ntiles + p.tiles_per_cta - 1) / p.tiles_per_cta;
  p.t = t; p.dt = dt; p.abstol = abstol; p.reltol = reltol; p.delta = delta;
  CallerBufs io(ctx, host_buffers);   // owned copies: pooled (256-byte aligned) arrays that alias no argument
  p.psf = io.copy_in(ps_drift, drift->nparams);
  p.psg = io.copy_in(ps_diffusion, diffusion->nparams);
  p.uprev = io.copy_in(uprev, DB);
  p.dW = io.copy_in(dW, DB);
  p.u = io.copy_out(u, DB);
  DevBuf parts(ctx, 2 * (size_t)grid + 2);
  p.partials = (double*)parts.p;
  LR_CUDA(cudaFuncSetAttribute(sde_aux_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  sde_aux_step_kernel<<<grid, SDE_THREADS, smem, st>>>(p);
  LR_COUNT(ctx);
  LR_CUDA(cudaGetLastError());
  std::vector<double> hp(grid);
  LR_CUDA(cudaMemcpyAsync(hp.data(), parts.p, sizeof(double) * grid, cudaMemcpyDeviceToHost, st));
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  double tot = 0.0;
  for (double v : hp) tot += v;
  const float eest = sqrtf((float)(tot / (double)DB));
  *reg_val = eest * dt;   // perform_step.jl:169,205: EEst * dt
  LR_API_END
}
