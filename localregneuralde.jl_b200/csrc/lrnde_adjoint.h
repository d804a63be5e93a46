// Latent-space adjoint engine for TDChain(Dense(D(+1) => H, act), Dense(H(+1) => D)) dynamics: the continuous adjoint
// (InterpolatingAdjoint + ZygoteVJP, src/layers/neural_ode.jl:11, experiments/src/construct.jl:197) integrated by Tsit5
// over z = [lambda ; mu] with every stage evaluated in the H-dimensional hidden space.
//
// With W1 = layer-1 weight [H x D], W2a = [W2 | w2t | b2] ([D x Kaug]), Mz = W1 W2a, Mh = Mz[:, :H]:
//   forward state     y(tau) = x + W2a c(tau),  c(tau) = C_n + dt_n sum_i b_i(theta) [h_i ; t_i ; 1]   (hidden tape of
//                     the forward solve: C_n = cumulative image of u_n, lrnde_fused.cu)
//   pre-activation    p_j = W1 y_j + w1t tau_j + b1 = Zx + Mz c_j + w1t tau_j + b1,   h_j = act(p_j), s_j = act'(p_j)
//   adjoint stage     lambda_j = lambda_n + dt sum_i a_ji kappa_i,  kappa_i = -W1^T delta_i
//                     alpha_j := W2^T lambda_j = alpha_n - dt Mh^T eps_j,  eps_j = sum_i a_ji delta_i,  delta_j = s_j .* alpha_j
//   lambda block      lambda_{n+1} = lambda_n - dt W1^T Delta_b,  utilde = -dt W1^T Delta_bt   (Delta_w = sum_j w_j delta_j)
//   mu block          mu' = -J_p^T lambda:  sum_j w_j dW1_j = Delta_w x^T + (sum_j w_j delta_j c_j^T) W2a^T,
//                     sum_j w_j dW2a_j = lambda_n (sum_j w_j [h_j;tau_j;1])^T - dt W1^T (sum_j w_j eps_j [h_j;tau_j;1]^T)
// so an attempt touches D-dimensional data only to read lambda_n and x and to write lambda_{n+1}:
//   (0) adj_interp_kernel  c_j of the six stages from the forward hidden tape (lambda-independent: one pass over the
//                          whole batch, one read of each forward interval's tape per attempt), stored for (1) and (4)
//   (1) adj_pre_kernel     the rest of the lambda-independent stage work over the whole batch: p_j = Zx + Mz c_j + ...
//                          (tcgen05, Mz as TMEM A operand), [h_j;tau_j;1], s_j and the sums sum_j w_j [h_j;tau_j;1]
//   (2) adj_chain_kernel   the lambda recurrence of the six stages in hidden space: one Mh^T eps_j MMA round trip per
//                          stage (tcgen05, Mh^T as TMEM A operand; s_j from (1))
//   (3) kgemm_kernel<2,1>  [W1^T Delta_b, W1^T Delta_bt] with the lambda_{n+1} / residual epilogue (lrnde_fused.cu)
//   (4) pairacc_kernel     every batch contraction of the mu block (tcgen05, MN-major operands, split over the batch)
//   (5) adj_reduce_kernel + adj_mu_kernel   fixed-order reduction, mu_{n+1}, residual of the mu block
//   (6) controller_kernel  (unchanged)
#pragma once
#include "lrnde_fused.h"

struct LatentAdjoint {
  lrnde_ctx* ctx;
  const lrnde_model* m;
  const float* ps;
  int64_t B;
  int passes;
  FusedShape sh;
  size_t zlen = 0;
  int ntiles = 0, nunits = 0, nclusters = 1;
  int pre_ctas = 1;           // adj_pre_kernel: CTAs (one per SM), each takes whole 64-sample tiles
  int ntile_d = 0;            // 128-row feature tiles of a [D, B] array
  int nP = 1, chunkP = 32;    // pairacc: CTAs / samples per CTA of the hidden-space terms
  int nD = 1, chunkD = 32;    // pairacc: batch splits / samples per split of the D-dimensional terms
  float* Mz = nullptr;        // [128][128] plain fp32 (zero padded)
  const float* Mz_ext = nullptr;   // the copy the forward call kept, when there is one
  float* ws = nullptr;        // LA_NARR hidden-space arrays of [B][LR_ZROW]
  float* alpha_in = nullptr;  // W2^T lambda of the current state (written by the caller's GEMM before begin())
  float* hbuf = nullptr;      // operand images of the lambda GEMM: units of 16 samples x {Delta_b, Delta_bt}
  size_t unit_bytes = 0;
  float* partP = nullptr; float* partX = nullptr; float* partL = nullptr;
  float* RP = nullptr; float* RX = nullptr; float* RL = nullptr;
  const float* W1T = nullptr; // [H][D]
  const float* Zx = nullptr;  // W1 x, [B][LR_ZROW]
  const float* x = nullptr;   // [D, B]

  static bool eligible(const lrnde_model* m);
  LatentAdjoint(lrnde_ctx* c, const lrnde_model* mm, const float* p, int64_t b, int npasses);
  ~LatentAdjoint();
  void prepare(const float* mz_plain = nullptr);
  // stage-1 quantities (delta_1, [h_1;t;1], c_1, alpha) of the current state from alpha_in and S->yint[0]: (0), (1)
  void begin(SolveDev* S);
  // one Tsit5 attempt of the adjoint from the descriptors of S (st, yint, err): launches (0) - (5)
  void attempt(SolveDev* S);
  // profiling: the launches of attempt() one by one (0 interpolant + pre + chain, 1 lambda GEMM, 2 pairacc,
  // 3 reduce + mu)
  void attempt_part(SolveDev* S, int which);
};
