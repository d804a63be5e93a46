// Latent-space adjoint engine (see lrnde_adjoint.h): hand-written tcgen05 / TMEM / bulk-copy code for sm_100a.
// Reference arithmetic: the Tsit5 stages / u / utilde / residual of src/perform_step.jl:10-27,34-38,208-212 applied to
// the augmented adjoint state z = [lambda ; mu] of InterpolatingAdjoint(ZygoteVJP) (SURVEY App. A.5), with the
// right-hand side (-J_u^T lambda, -J_p^T lambda) of TDChain(Dense, Dense) (src/layers/common.jl:19-33) evaluated
// through the identities in the header.
#include "lrnde_adjoint.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "lrnde_fused_dev.cuh"

// hidden-space work arrays ([B][LR_ZROW] each, padded to whole 64-sample tiles).  Written by: interp = (0), pre = (1),
// chain = (2); stage 7 of an attempt is stage 1 of the next ring slot.
enum {
  LA_ALPHA = 0,   // + slot: W2^T lambda of the ring slot (pre in single mode, chain)
  LA_S1 = 2,      // + 3 * slot + {0: delta_1 (pre single / chain), 1: [h_1;t;1] (pre), 2: c_1 (interp)}: stage 1 (FSAL)
  LA_DEL = 8,     // + j - 2, j = 2..6: delta_j (chain)
  LA_CC = 13,     // + j - 2: c_j (rows Kaug, Kaug + 1 = tau_j, 1) (interp)
  LA_HH = 18,     // + j - 2: [h_j ; tau_j ; 1] (pre)
  LA_EPS = 23,    // + j - 2, j = 2..7: eps_j = sum_i a_ji delta_i  (eps_7 = Delta_b) (chain)
  LA_DBT = 29,    // Delta_btilde (chain)
  LA_HBB = 30,    // sum_j b_j [h_j;tau_j;1] (pre)
  LA_HBT = 31,    // sum_j btilde_j [h_j;tau_j;1] (pre)
  LA_SS = 32,     // + j - 2, j = 2..7: s_j = act'(p_j), 0 in rows >= H (pre)
  LA_NARR = 38
};

#ifdef LRNDE_UMMA_TRACE
__device__ long long g_adj_trace[1024];
// CTA 1 only; rows of 16 stamps (row = event kind, column = stage)
#define ATRACE(row, it) do { if ((int)blockIdx.x == 1 && (it) < 16) g_adj_trace[(row) * 16 + (it)] = clock64(); } while (0)
extern "C" int lrnde_debug_trace_adj(long long* out, int n) {
  cudaMemcpyFromSymbol(out, g_adj_trace, sizeof(long long) * (size_t)n);
  return 0;
}
#else
#define ATRACE(row, it) do { } while (0)
#endif

namespace ladj {
using namespace umma;
using namespace fused;

template <int ACT>
__device__ __forceinline__ void act_pair(float x, float& h, float& s) {
  if (ACT == ACT_TANH) { h = tanhf(x); s = 1.0f - h * h; }
  else if (ACT == ACT_SIGMOID) { h = 1.0f / (1.0f + expf(-x)); s = h * (1.0f - h); }
  else { h = lr_act(ACT, x); s = lr_dact(ACT, x); }
}

// ---------------------------------------------------------------------------------------------------------
// (0) interpolant kernel: c_j = C_n + dt_n sum_i b_i(theta_j) H(k_i), the dense interpolant of the forward solution in
// hidden space at every stage time of the attempt, written as the stored copy of c_j (rows Kaug, Kaug + 1 = tau_j, 1,
// the rest 0).  It does not depend on lambda, so it runs over the whole batch ahead of the pre kernel, and the stages
// that fall in the same forward interval share one read of that interval's 8 tape arrays.
// Thread = 4 hidden rows of one sample (a warp reads one sample's row of 512 bytes).
// ---------------------------------------------------------------------------------------------------------
struct AInterpP {
  SolveDev* S;
  int single;            // 1: c_1 of the current state (time / interpolant yint[0])
  float* ws;
  size_t zlen;
  int B, Kaug, nunit;    // nunit = padded samples x LR_ZROW / 4
};

__global__ void __launch_bounds__(256) adj_interp_kernel(AInterpP p) {
  SolveDev* S = p.S;
  if (p.single ? S->failed : S->done) return;
  __shared__ float s_cf[6][8], s_sc[6][8], s_tau[6];
  __shared__ const float* s_hb[6];
  __shared__ float* s_dst[6];
  const int nst = p.single ? 1 : 6;
  if (threadIdx.x < nst) {
    const int j = threadIdx.x;
    const LinComb& yd = S->yint[p.single ? 0 : j + 1];
    const size_t slotn = (size_t)(yd.base - S->ftape) / ((size_t)7 * S->flen);
    s_hb[j] = S->fhtape + slotn * 7 * S->fzlen;
    for (int s = 0; s < 8; ++s) {
      s_cf[j][s] = (s < 7) ? yd.coef[s] : 1.0f;
      s_sc[j][s] = (s < 7) ? 1.0f : yd.scale;
    }
    s_tau[j] = yd.t;
    const int slot = S->slot, next = (S->slot + 1) % S->cap;
    const int arr = p.single ? LA_S1 + 3 * slot + 2 : (j == 5 ? LA_S1 + 3 * next + 2 : LA_CC + j);
    s_dst[j] = p.ws + (size_t)arr * p.zlen;
  }
  __syncthreads();
  const int u = blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= p.nunit) return;
  const int b = u / (LR_ZROW / 4), r0 = (u % (LR_ZROW / 4)) * 4;
  const size_t e = (size_t)b * LR_ZROW + r0;
  const bool any = (b < p.B) && (r0 < p.Kaug);
  float4 tp[8];
  const float* cur = nullptr;
  for (int j = 0; j < nst; ++j) {
    if (any && s_hb[j] != cur) {   // tiles in the order the coefficients take them: H(k_1..7), then C_n
      cur = s_hb[j];
#pragma unroll
      for (int s = 0; s < 8; ++s) {
        const float* src = (s == 7) ? cur : cur + (size_t)(s < 6 ? s + 1 : 8) * S->fzlen;   // H(k_7) = H(k_1) of the next slot
        tp[s] = __ldcg(reinterpret_cast<const float4*>(src + e));
      }
    }
    float c[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    if (any) {
#pragma unroll
      for (int s = 0; s < 8; ++s) {
        const float cf = s_cf[j][s], sc = s_sc[j][s];
        c[0] = fmaf(cf, tp[s].x, __fmul_rn(sc, c[0]));
        c[1] = fmaf(cf, tp[s].y, __fmul_rn(sc, c[1]));
        c[2] = fmaf(cf, tp[s].z, __fmul_rn(sc, c[2]));
        c[3] = fmaf(cf, tp[s].w, __fmul_rn(sc, c[3]));
      }
    }
    float o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int r = r0 + k;
      o[k] = (r < p.Kaug) ? c[k] : ((r == p.Kaug) ? s_tau[j] : ((r == p.Kaug + 1) ? 1.0f : 0.0f));
    }
    *reinterpret_cast<float4*>(s_dst[j] + e) = make_float4(o[0], o[1], o[2], o[3]);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Shared by the two tensor-core kernels below: one CTA works on 64 samples as two independent halves of 32 (while the
// tensor core works for one half the other half's warps do their element-wise arithmetic).  Thread of a compute warp =
// one hidden row x 16 samples; an [M = 128 rows] x [K = KS * 8] matrix sits in tensor memory as the A operand (hi and lo
// images, 8 KS columns each), the 32-sample B operand tile is formed in shared memory.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void issue_group(uint32_t d, uint32_t a_hi, uint32_t a_lo, uint32_t b0, int nfull, int ntail,
                                            int passes, uint32_t idesc) {
  uint32_t first = 0u;
  for (int pc = 0; pc < nfull; ++pc) {
    const uint32_t bh = desc_lo(b0 + pc * 8192), bl = desc_lo(b0 + pc * 8192 + 4096);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t ah = a_hi + (uint32_t)((pc * 4 + k) * 8), al = a_lo + (uint32_t)((pc * 4 + k) * 8);
      if (passes == 3) {
        mma_ts(d, al, bh + 2 * k, kHi128, idesc, first);
        mma_ts(d, ah, bl + 2 * k, kHi128, idesc, 1u);
        mma_ts(d, ah, bh + 2 * k, kHi128, idesc, 1u);
      } else mma_ts(d, ah, bh + 2 * k, kHi128, idesc, first);
      first = 1u;
    }
  }
  for (int t = 0; t < ntail; ++t) {
    const uint32_t bb = b0 + nfull * 8192 + t * 2048;
    const uint32_t bh = desc_lo(bb), bl = desc_lo(bb + 1024);
    const uint32_t ah = a_hi + (uint32_t)((nfull * 4 + t) * 8), al = a_lo + (uint32_t)((nfull * 4 + t) * 8);
    if (passes == 3) {
      mma_ts(d, al, bh, kHi32, idesc, first);
      mma_ts(d, ah, bl, kHi32, idesc, 1u);
      mma_ts(d, ah, bh, kHi32, idesc, 1u);
    } else mma_ts(d, ah, bh, kHi32, idesc, first);
    first = 1u;
  }
}

// The per-thread view of a compute warp (warps 2 .. 17): TMEM lane quarter q, hidden row hrow, half cg and the first of
// its 16 samples inside the tile; tile_put16 writes the thread's 16 values as (tile row = sample, k = hrow) of a [hi | lo]
// operand image: byte offset = oA + r * oS + ((osw ^ m(r)) << 4) with m(r) = r & 7 (SWIZZLE_128B chunks of 32 k) or
// (r >> 2) & 1 (SWIZZLE_32B K-steps of the tail); lo image at + oLo.
struct ComputeLane {
  int q, cg, hrow, rbase;
  bool rowv, rowc, in_full, in_img;
  uint32_t oA, osw;
  __device__ __forceinline__ ComputeLane(int warp, int lane, int H, int Kaug, int KS, int nfull) {
    q = warp & 3;
    const int sub = (warp - 2) >> 2;
    cg = sub >> 1;
    hrow = q * 32 + lane;
    rbase = (sub & 1) * 16;
    rowv = hrow < H;
    rowc = hrow < Kaug;
    in_full = hrow < nfull * 32;
    in_img = hrow < KS * 8;
    if (in_full) {
      osw = (uint32_t)(lane >> 2);
      oA = (uint32_t)(q * 8192 + (lane & 3) * 4) + (uint32_t)rbase * 128u;
    } else {
      const int kt = hrow - nfull * 32, t = kt >> 3, kk = kt & 7;
      osw = (uint32_t)((kk >> 2) & 1);
      oA = (uint32_t)(nfull * 8192 + t * 2048 + (kk & 3) * 4) + (uint32_t)rbase * 32u;
    }
  }
  __device__ __forceinline__ void tile_put16(uint8_t* tile, const float (&val)[16], int passes) const {
    if (!in_img) return;
    const uint32_t oS = in_full ? 128u : 32u, oLo = in_full ? 4096u : 1024u;
    // tf32 split without branches: passes == 1 keeps the value (no rounding, lo = 0)
    const uint32_t rnd = (passes == 3) ? 0x1000u : 0u, msk = (passes == 3) ? 0xFFFFE000u : 0xFFFFFFFFu;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const uint32_t m = in_full ? (uint32_t)(i & 7) : (uint32_t)((i >> 2) & 1);
      const uint32_t o = oA + (uint32_t)i * oS + ((osw ^ m) << 4);
      const float hi = __uint_as_float((__float_as_uint(val[i]) + rnd) & msk);
      const float lo = __uint_as_float((__float_as_uint(val[i] - hi) + rnd) & msk);
      *reinterpret_cast<float*>(tile + o) = hi;
      *reinterpret_cast<float*>(tile + o + oLo) = lo;
    }
  }
};

// A operand -> tensor memory: element (hrow, k) of a [128][128] fp32 matrix, k < KS * 8, as hi at column k and lo at
// column 8 KS + k (warp `sub` of a lane quarter writes the K-steps sub, sub + 4, ...).  transposed: Mh^T = Mz[:H, :H]^T.
__device__ __forceinline__ void a_operand_to_tmem(const float* Mz, bool transposed, int H, int KS, int passes, int warp,
                                                  int hrow, uint32_t tlane) {
  const int sub = (warp - 2) >> 2;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int ks = sub + 4 * j;
    if (ks < KS) {
      float a[8], hi[8], lo[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int k = ks * 8 + e;
        a[e] = transposed ? ((hrow < H && k < H) ? __ldg(Mz + k * 128 + hrow) : 0.0f)   // Mh^T[hrow][k] = Mz[k][hrow]
                          : __ldg(Mz + hrow * 128 + k);                                  // Mz[hrow][k]  (zero padded)
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        if (passes == 3) { hi[e] = tf32_rna(a[e]); lo[e] = tf32_rna(a[e] - hi[e]); }
        else { hi[e] = a[e]; lo[e] = 0.0f; }
      }
      tmem_st8(tlane + (uint32_t)(ks * 8), hi);
      tmem_st8(tlane + (uint32_t)(8 * KS + ks * 8), lo);
    }
  }
  tmem_st_wait();
}

// ---------------------------------------------------------------------------------------------------------
// (1) pre kernel: everything of a stage that does not depend on lambda, over the whole batch:
//       p_j = Zx + Mz c_j + w1t tau_j + b1,  [h_j ; tau_j ; 1],  s_j = act'(p_j)   (rows >= H of s_j are 0)
//     and, per sample, sum_j b_j [h_j;tau_j;1] and sum_j btilde_j [h_j;tau_j;1] over the seven stages of the attempt
//     (stage 1 from the ring slot).  A CTA takes whole 64-sample tiles (all their stages, so the two sums stay in
//     registers), tile = blockIdx.x + i * gridDim.x; the stages are independent, so the c tile of the next stage is
//     formed while the tensor core works on the current one (two [hi | lo] tiles and two accumulators per half).
//     TMEM: [Mz hi | Mz lo] (8 KS columns each), then four 32-column accumulators (half cg, buffer b at 32 (2 cg + b)).
//     SINGLE (stage 1 of the current state, c_1 from yint[0]): also delta_1 = s_1 .* alpha_in and alpha of the slot.
// ---------------------------------------------------------------------------------------------------------
struct APreP {
  SolveDev* S;
  const float* Mz;
  const float* w1t;      // layer-1 time column (nullptr without TDChain)
  const float* b1;
  const float* Zx;
  const float* alpha_in;
  float* ws;
  size_t zlen;
  int H, td, Kaug, KS, nfull, ntail, passes, ntiles;
};

template <int ACT, bool SINGLE>
__global__ void __launch_bounds__(kThreads, 1) adj_pre_kernel(APreP p) {
  SolveDev* S = p.S;
  if (SINGLE ? S->failed : S->done) return;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t a_ready, bfull[2][2], pdone[2][2];
  __shared__ uint32_t tmem_slot;
  __shared__ float s_tau[6], s_cb[7], s_ct[7];
  __shared__ int s_slot, s_next;

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int nst = SINGLE ? 1 : 6;
  const int nk = ((p.ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x) * nst;   // stages of this CTA
  const uint32_t tileB = (uint32_t)(p.nfull * 8192 + p.ntail * 2048);   // [hi | lo] images of a 32-sample operand tile
  auto tile = [&](int cg, int b) { return smem + (size_t)(2 * cg + b) * tileB; };

  if (threadIdx.x == 0) {
    mbar_init(&a_ready, (uint32_t)kEpiWarps);
    for (int c = 0; c < 2; ++c)
      for (int b = 0; b < 2; ++b) { mbar_init(&bfull[c][b], (uint32_t)(kEpiWarps / 2)); mbar_init(&pdone[c][b], 1u); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    s_slot = S->slot; s_next = (S->slot + 1) % S->cap;
  }
  if (threadIdx.x >= 32 && threadIdx.x < 32 + nst) s_tau[threadIdx.x - 32] = S->yint[SINGLE ? 0 : threadIdx.x - 31].t;
  if (threadIdx.x >= 64 && threadIdx.x < 71) {   // weights of stage s = 0..6 in the two sums (b_7 = 0)
    const int s = threadIdx.x - 64;
    s_cb[s] = (s < 6) ? S->st[5].coef[s] : 0.0f;
    s_ct[s] = S->err.coef[s];
  }
  if (warp == 1) {   // 16 KS + 128 <= 352 columns (KS <= 14)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  const uint32_t c_acc = tmem_base + (uint32_t)(16 * p.KS);
  auto arr = [&](int idx) -> float* { return p.ws + (size_t)idx * p.zlen; };

  if (warp == 1) {
    // ---------------- tcgen05.mma issue (M = 128 hidden rows x N = 32 samples, A from tensor memory): p = Mz c
    constexpr uint32_t idesc = make_idesc(128, kNT / 2);
    mbar_wait(&a_ready, 0);
    tc_fence_after();
    const uint32_t mz_hi = tmem_base, mz_lo = tmem_base + (uint32_t)(8 * p.KS);
    for (int k = 0; k < nk; ++k) {
      const int b = k & 1;
      for (int cg = 0; cg < 2; ++cg) {
        mbar_wait(&bfull[cg][b], (uint32_t)((k >> 1) & 1));
        tc_fence_after();
        if (elect_one_sync()) {
          issue_group(c_acc + (uint32_t)((2 * cg + b) * 32), mz_hi, mz_lo, smem_u32(tile(cg, b)), p.nfull, p.ntail, p.passes,
                      idesc);
          mma_commit(&pdone[cg][b]);
        }
        __syncwarp();
      }
    }
  } else if (warp >= 2) {
    const ComputeLane L(warp, lane, p.H, p.Kaug, p.KS, p.nfull);
    const uint32_t tlane = tmem_base + ((uint32_t)(L.q * 32) << 16);
    a_operand_to_tmem(p.Mz, false, p.H, p.KS, p.passes, warp, L.hrow, tlane);
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&a_ready);

    const float w1t = (p.td && L.rowv && p.w1t) ? p.w1t[L.hrow] : 0.0f;
    const float b1 = L.rowv ? p.b1[L.hrow] : 0.0f;
    const int slot = s_slot, next = s_next;
    // element of (first sample of this thread, this row) for the k-th stage of the CTA.  The work arrays are padded to
    // whole 64-sample tiles, so samples beyond B are computed and stored like the others (never read back)
    auto e0_of = [&](int k) -> size_t {
      const int t = (int)blockIdx.x + (k / nst) * (int)gridDim.x;
      return (size_t)(t * kNT + L.cg * 32 + L.rbase) * LR_ZROW + L.hrow;
    };
    // c_j: adj_interp_kernel's stored copy
    auto c_src = [&](int j) -> const float* {
      return SINGLE ? arr(LA_S1 + 3 * slot + 2) : (j == 5 ? arr(LA_S1 + 3 * next + 2) : arr(LA_CC + j));
    };
    float c[16], zx[16], v[16], hb[16], ht[16];
    auto put_stage = [&](int k) {   // c of the k-th stage -> operand tile, then hand it to the MMA warp
      const float* src = c_src(k % nst) + e0_of(k);
#pragma unroll
      for (int i = 0; i < 16; ++i) c[i] = L.rowc ? __ldcg(src + (size_t)i * LR_ZROW) : 0.0f;
      L.tile_put16(tile(L.cg, k & 1), c, p.passes);
      tc_fence_before();
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bfull[L.cg][k & 1]);
    };
    if (nk > 0) put_stage(0);
    for (int k = 0; k < nk; ++k) {
      const int j = k % nst;
      const size_t e0 = e0_of(k);
      if (!SINGLE && j == 0) {   // the two sums start with stage 1 (FSAL) of the ring slot
        const float* h1 = arr(LA_S1 + 3 * slot + 1) + e0;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float hv = L.rowc ? __ldcg(h1 + (size_t)i * LR_ZROW) : 0.0f;
          hb[i] = fmaf(s_cb[0], hv, 0.0f);
          ht[i] = fmaf(s_ct[0], hv, 0.0f);
        }
      }
      if (k + 1 < nk) put_stage(k + 1);   // the next stage's tile while the tensor core works on this one
#pragma unroll
      for (int i = 0; i < 16; ++i) zx[i] = L.rowv ? __ldcg(p.Zx + e0 + (size_t)i * LR_ZROW) : 0.0f;
      mbar_wait(&pdone[L.cg][k & 1], (uint32_t)((k >> 1) & 1));
      tc_fence_after();
      tmem_ld16(tlane + (uint32_t)(16 * p.KS + (2 * L.cg + (k & 1)) * 32 + L.rbase), v);
      tc_fence_before();
      const float tau = s_tau[j];
      const float hconst = (p.td && L.hrow == p.H) ? tau : ((L.hrow == p.H + p.td) ? 1.0f : 0.0f);
      const float pb = p.td ? fmaf(w1t, tau, b1) : b1;
      const bool last = (!SINGLE && j == 5);
      float* dst_hh = (SINGLE ? arr(LA_S1 + 3 * slot + 1) : (last ? arr(LA_S1 + 3 * next + 1) : arr(LA_HH + j))) + e0;
      float* dst_s = arr(LA_SS + j) + e0;
      float* dst_del = arr(LA_S1 + 3 * slot + 0) + e0;
      float* dst_alpha = arr(LA_ALPHA + slot) + e0;
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = v[i] + zx[i] + pb;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        float h, sg;
        act_pair<ACT>(v[i], h, sg);
        const float sj = L.rowv ? sg : 0.0f;
        const float hv = L.rowv ? h : hconst;
        dst_hh[(size_t)i * LR_ZROW] = hv;
        if (SINGLE) {   // alpha_1 = alpha_n ; delta_1 = s_1 .* alpha_1
          const float an = L.rowv ? __ldcg(p.alpha_in + e0 + (size_t)i * LR_ZROW) : 0.0f;
          dst_del[(size_t)i * LR_ZROW] = sj * an;
          dst_alpha[(size_t)i * LR_ZROW] = an;
        } else {
          dst_s[(size_t)i * LR_ZROW] = sj;
          hb[i] = fmaf(s_cb[j + 1], hv, hb[i]);
          ht[i] = fmaf(s_ct[j + 1], hv, ht[i]);
        }
      }
      if (last) {
        float* hbb = arr(LA_HBB) + e0;
        float* hbt = arr(LA_HBT) + e0;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          hbb[(size_t)i * LR_ZROW] = L.rowc ? hb[i] : 0.0f;
          hbt[(size_t)i * LR_ZROW] = L.rowc ? ht[i] : 0.0f;
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------------
// (2) chain kernel: the lambda recurrence of the six stages, one MMA round trip per stage and half:
//       eps_j = sum_i a_ji delta_i -> alpha_j = alpha_n - dt Mh^T eps_j -> delta_j = s_j .* alpha_j
//     s_j comes from (1) on a bulk-copy ring, the part of eps_{j+1} that is already known is formed while the tensor
//     core works.  TMEM: [Mh^T hi | Mh^T lo] (8 KS columns each), then one 32-column accumulator per half.
// ---------------------------------------------------------------------------------------------------------
constexpr int kTapeBufs = 3;                       // ring of [64 samples][LR_ZROW] tiles of s_j
constexpr int kTapeBufBytes = kNT * LR_ZROW * 4;   // 32 KB
struct AChainP {
  SolveDev* S;
  const float* Mz;
  float* ws;
  size_t zlen;
  float* hbuf;
  uint32_t unit_bytes;
  int H, Kaug, KS, nfull, ntail, passes;
};

__global__ void __launch_bounds__(kThreads, 1) adj_chain_kernel(AChainP p) {
  SolveDev* S = p.S;
  if (S->done) return;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t a_ready, bfull[2], xdone[2], out_full, tfull[kTapeBufs], tempty[kTapeBufs];
  __shared__ uint32_t tmem_slot;
  __shared__ LinComb sd[6];
  __shared__ float s_bt[7];
  __shared__ int s_slot, s_next;

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * kNT;
  constexpr int nst = 6;
  const uint32_t tileB = (uint32_t)(p.nfull * 8192 + p.ntail * 2048);   // [hi | lo] images of a 32-sample operand tile
  auto tC = [&](int cg) { return smem + (size_t)cg * tileB; };         // Delta_bt images of the two halves
  auto tE = [&](int cg) { return smem + (size_t)(2 + cg) * tileB; };   // eps_j images (eps_7 = Delta_b)
  uint8_t* tbuf = smem + 4 * (size_t)tileB;        // kTapeBufs s_j tiles (tileB is a multiple of 1024)

  if (threadIdx.x == 0) {
    mbar_init(&a_ready, (uint32_t)kEpiWarps);
    mbar_init(&out_full, (uint32_t)kEpiWarps);
    for (int b = 0; b < kTapeBufs; ++b) { mbar_init(&tfull[b], 1u); mbar_init(&tempty[b], (uint32_t)kEpiWarps); }
    for (int c = 0; c < 2; ++c) {
      mbar_init(&bfull[c], (uint32_t)(kEpiWarps / 2));
      mbar_init(&xdone[c], 1u);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    s_slot = S->slot; s_next = (S->slot + 1) % S->cap;
  }
  if (threadIdx.x >= 64 && threadIdx.x < 70) sd[threadIdx.x - 64] = S->st[threadIdx.x - 64];
  if (threadIdx.x >= 128 && threadIdx.x < 135) s_bt[threadIdx.x - 128] = S->err.coef[threadIdx.x - 128];
  if (warp == 1) {   // 16 KS + 64 <= 288 columns (KS <= 14)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  const uint32_t c_acc = tmem_base + (uint32_t)(16 * p.KS);
  auto arr = [&](int idx) -> float* { return p.ws + (size_t)idx * p.zlen; };
  const bool tr = (threadIdx.x == 64);
  if (tr) ATRACE(0, 0);

  if (warp == 0) {
    // ---------------- s_j in: one whole (padded) tile per stage, bulk-copied onto a ring
    {
      constexpr uint32_t bytes = (uint32_t)kTapeBufBytes;
      for (int it = 0; it < nst; ++it) {
        const int b = it % kTapeBufs;
        mbar_wait(&tempty[b], (uint32_t)(((it / kTapeBufs) & 1) ^ 1));
        if (elect_one_sync()) {
          mbar_arrive_expect_tx(&tfull[b], bytes);
          bulk_g2s(tbuf + (size_t)b * kTapeBufBytes, arr(LA_SS + it) + (size_t)n0 * LR_ZROW, bytes, &tfull[b]);
        }
        __syncwarp();
      }
    }
    // ---------------- Delta_b / Delta_bt operand images out (units of 16 samples for the lambda GEMM)
    mbar_wait(&out_full, 0);
    if (elect_one_sync()) {
      for (int sg = 0; sg < 4; ++sg) {
        uint8_t* g = reinterpret_cast<uint8_t*>(p.hbuf) + ((size_t)blockIdx.x * 4 + sg) * p.unit_bytes;
        const int cg = sg >> 1, half = sg & 1;
        for (int c = 0; c < p.nfull; ++c)
          for (int lo = 0; lo < 2; ++lo) {
            bulk_s2g(g + (size_t)c * 8192 + lo * 4096, tE(cg) + (size_t)c * 8192 + lo * 4096 + half * 2048, 2048);
            bulk_s2g(g + (size_t)c * 8192 + lo * 4096 + 2048, tC(cg) + (size_t)c * 8192 + lo * 4096 + half * 2048, 2048);
          }
        for (int t = 0; t < p.ntail; ++t)
          for (int lo = 0; lo < 2; ++lo) {
            const size_t o = (size_t)p.nfull * 8192 + (size_t)t * 2048 + lo * 1024;
            bulk_s2g(g + o, tE(cg) + o + half * 512, 512);
            bulk_s2g(g + o + 512, tC(cg) + o + half * 512, 512);
          }
      }
      bulk_commit();
      bulk_wait0();
    }
    __syncwarp();
  } else if (warp == 1) {
    // ---------------- tcgen05.mma issue (M = 128 hidden rows x N = 32 samples, A from tensor memory): Mh^T eps_j
    constexpr uint32_t idesc = make_idesc(128, kNT / 2);
    mbar_wait(&a_ready, 0);
    tc_fence_after();
    const uint32_t mt_hi = tmem_base, mt_lo = tmem_base + (uint32_t)(8 * p.KS);
    for (int st = 0; st < nst; ++st) {
      for (int cg = 0; cg < 2; ++cg) {
        mbar_wait(&bfull[cg], (uint32_t)(st & 1));
        tc_fence_after();
        if (elect_one_sync()) {
          if (cg == 0) ATRACE(7, st);
          issue_group(c_acc + (uint32_t)(cg * 32), mt_hi, mt_lo, smem_u32(tE(cg)), p.nfull, p.ntail, p.passes, idesc);
          mma_commit(&xdone[cg]);
          if (cg == 0) ATRACE(8, st);
        }
        __syncwarp();
      }
    }
  } else {
    // ---------------- compute warps: lane = hidden row, registers = 16 samples
    const ComputeLane L(warp, lane, p.H, p.Kaug, p.KS, p.nfull);
    const int cg = L.cg;
    const uint32_t tlane = tmem_base + ((uint32_t)(L.q * 32) << 16);
    a_operand_to_tmem(p.Mz, true, p.H, p.KS, p.passes, warp, L.hrow, tlane);
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&a_ready);
    if (tr) ATRACE(0, 1);

    const bool rowv = L.rowv;
    const int slot = s_slot, next = s_next;
    const float dt = sd[0].scale;
    // element of (first sample, this row) in a [Bpad][LR_ZROW] array (padded to whole tiles: no bounds tests below)
    const size_t e0 = (size_t)(n0 + cg * 32 + L.rbase) * LR_ZROW + L.hrow;
    const float* ring_row = reinterpret_cast<const float*>(tbuf) + (cg * 32 + L.rbase) * LR_ZROW + L.hrow;

    const float* alpha_n = arr(LA_ALPHA + slot) + e0;
    float ep[16], dprev[16], an[16], v[16], ss[16];
    {
      const float* d1 = arr(LA_S1 + 3 * slot + 0) + e0;     // delta_1 (FSAL) of the current state
#pragma unroll
      for (int i = 0; i < 16; ++i) { ep[i] = 0.0f; dprev[i] = rowv ? __ldcg(d1 + (size_t)i * LR_ZROW) : 0.0f; }
    }
    for (int jj = 0; jj < nst; ++jj) {
      const bool last = (jj == 5);
      if (tr) ATRACE(1, jj);
      // ---- operand tile: eps_j = (partial sum prefetched during the previous stage) + a_{j,j-1} delta_{j-1}
      {
        const float cl = sd[jj].coef[jj];
        float* dst_eps = arr(LA_EPS + jj) + e0;
#pragma unroll
        for (int i = 0; i < 16; ++i) { v[i] = fmaf(cl, dprev[i], ep[i]); dst_eps[(size_t)i * LR_ZROW] = v[i]; }
        L.tile_put16(tE(cg), v, p.passes);
        tc_fence_before();
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bfull[cg]);
      }
      if (tr) ATRACE(2, jj);
      if (jj + 1 < nst) {   // known part of eps_{j+1}: delta_1 .. delta_j (the newest one is in registers)
#pragma unroll
        for (int i = 0; i < 16; ++i) ep[i] = sd[jj + 1].coef[jj] * dprev[i];
        if (rowv) {
          for (int s = 0; s < jj; ++s) {
            const float* src = ((s == 0) ? arr(LA_S1 + 3 * slot + 0) : arr(LA_DEL + s - 1)) + e0;
            const float cf = sd[jj + 1].coef[s];
#pragma unroll
            for (int i = 0; i < 16; ++i) ep[i] = fmaf(cf, __ldcg(src + (size_t)i * LR_ZROW), ep[i]);
          }
        }
      }
      if (tr) ATRACE(3, jj);
      // ---- alpha_j = alpha_n - dt Mh^T eps_j ; delta_j = s_j .* alpha_j
#pragma unroll
      for (int i = 0; i < 16; ++i) an[i] = rowv ? __ldcg(alpha_n + (size_t)i * LR_ZROW) : 0.0f;
      mbar_wait(&xdone[cg], (uint32_t)(jj & 1));
      if (tr) ATRACE(6, jj);
      tc_fence_after();
      tmem_ld16(c_acc + ((uint32_t)(L.q * 32) << 16) + (uint32_t)(cg * 32 + L.rbase), v);
      tc_fence_before();
      // ---- s_j from the ring (read after the MMA wait: not live across it)
      {
        const int b = jj % kTapeBufs;
        mbar_wait(&tfull[b], (uint32_t)((jj / kTapeBufs) & 1));
        const float* tb = ring_row + (size_t)b * (kTapeBufBytes / 4);
#pragma unroll
        for (int i = 0; i < 16; ++i) ss[i] = tb[i * LR_ZROW];
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[b]);
      }
      float* dst_del = (last ? arr(LA_S1 + 3 * next + 0) : arr(LA_DEL + jj)) + e0;
      float* dst_alpha = arr(LA_ALPHA + next) + e0;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float aj = fmaf(-dt, v[i], an[i]);
        dprev[i] = ss[i] * aj;
        dst_del[(size_t)i * LR_ZROW] = dprev[i];
        if (last) dst_alpha[(size_t)i * LR_ZROW] = rowv ? aj : 0.0f;
      }
    }
    if (tr) ATRACE(0, 3);
    // ---- Delta_bt = sum_j btilde_j delta_j (stage 7 in registers), three source arrays per round trip
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = s_bt[6] * dprev[i];
    if (rowv) {
      for (int s0 = 0; s0 < 6; s0 += 3) {
        float t[3][16];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const float* src = ((s0 + k == 0) ? arr(LA_S1 + 3 * slot + 0) : arr(LA_DEL + s0 + k - 1)) + e0;
#pragma unroll
          for (int i = 0; i < 16; ++i) t[k][i] = __ldcg(src + (size_t)i * LR_ZROW);
        }
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = fmaf(s_bt[s0 + k], t[k][i], v[i]);
      }
    }
    float* dbt = arr(LA_DBT) + e0;
#pragma unroll
    for (int i = 0; i < 16; ++i) dbt[(size_t)i * LR_ZROW] = v[i];
    L.tile_put16(tC(cg), v, p.passes);
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) mbar_arrive(&out_full);
    if (tr) ATRACE(0, 4);
    tc_fence_before();
  }
  __syncthreads();
  if (threadIdx.x == 0) ATRACE(0, 5);
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------------
// (4) pairacc kernel: batch contractions  acc[2a + v] += sum_b P[:, b] (s_v Q_v[:, b])^T  (v = 0, 1) on the tensor cores.
// Operands are [rows, B] arrays with the rows of a sample contiguous = MN-major for the MMA (same operand images as
// umma::wgrad_kernel).  Jobs (blockIdx): 0 = the hidden-space terms (P = c_j / H_j, Q = delta_j / eps_j scaled by
// b_j and btilde_j; 4 accumulators), 1 = x (Delta_b, Delta_bt)^T per 128-feature tile, 2 = lambda_n (HB_b, HB_bt)^T.
// ---------------------------------------------------------------------------------------------------------
struct PaTerm { int p_arr, q_arr; float s0, s1; int acc; };
struct PairAccP {
  SolveDev* S;
  const float* ws;
  size_t zlen;
  const float* x;
  int D, B;
  int nP, chunkP, nD, chunkD, ntile;
  float* partP; float* partX; float* partL;
  int nterm, passes;
  PaTerm term[13];
};
constexpr int kPaStageBytes = 6 * 16384;   // [P_hi | P_lo | Q0_hi | Q0_lo | Q1_hi | Q1_lo], 128 rows x 32 samples each
constexpr int kPaStages = 2;
constexpr int pairacc_smem() { return kPaStages * kPaStageBytes + 1024; }

__global__ void __launch_bounds__(kThreads, 1) pairacc_kernel(PairAccP q) {
  SolveDev* S = q.S;
  if (S->done) return;
  constexpr int NS = kPaStages;
  constexpr int PT = kEpiWarps * 32;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t full_bar[NS], empty_bar[NS], done_bar;
  __shared__ uint32_t tmem_slot;

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  int job, tile = 0, split, b_begin, b_end, nterm;
  if ((int)blockIdx.x < q.nP) {
    job = 0; split = blockIdx.x; nterm = q.nterm;
    b_begin = split * q.chunkP; b_end = min(q.B, b_begin + q.chunkP);
  } else {
    const int b2 = (int)blockIdx.x - q.nP;
    job = 1 + b2 / (q.ntile * q.nD);
    const int rem = b2 % (q.ntile * q.nD);
    tile = rem / q.nD; split = rem % q.nD; nterm = 1;
    b_begin = split * q.chunkD; b_end = min(q.B, b_begin + q.chunkD);
  }
  const int nchunks = (b_end > b_begin) ? (b_end - b_begin + 31) / 32 : 0;
  const int niter = nterm * nchunks;
  const int slot = S->slot, next = (S->slot + 1) % S->cap;
  auto arr = [&](int code) -> const float* {
    if (code >= 0) return q.ws + (size_t)code * q.zlen;
    if (code > -10) return q.ws + (size_t)(LA_S1 + 3 * slot + (-1 - code)) * q.zlen;
    return q.ws + (size_t)(LA_S1 + 3 * next + (-10 - code)) * q.zlen;
  };

  if (threadIdx.x == 0) {
    for (int s = 0; s < NS; ++s) {
      mbar_init(&full_bar[s], (uint32_t)kEpiWarps);
      mbar_init(&empty_bar[s], 1u);
    }
    mbar_init(&done_bar, 1u);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  if (warp == 1) {
    constexpr uint32_t idesc = make_idesc_mn(128, 128);
    uint32_t touched = 0u;
    for (int it = 0; it < niter; ++it) {
      const int s = it % NS, ph = (it / NS) & 1;
      const int ap = (job == 0) ? q.term[it / nchunks].acc : 0;
      mbar_wait(&full_bar[s], (uint32_t)ph);
      tc_fence_after();
      const uint32_t base = smem_u32(smem + (size_t)s * kPaStageBytes);
      const uint32_t p_hi = desc_lo_mn(base), p_lo = desc_lo_mn(base + 16384);
      const uint32_t q0_hi = desc_lo_mn(base + 32768), q0_lo = desc_lo_mn(base + 49152);
      const uint32_t q1_hi = desc_lo_mn(base + 65536), q1_lo = desc_lo_mn(base + 81920);
      const uint32_t d0 = tmem_base + (uint32_t)(ap * 256), d1 = d0 + 128u;
      if (elect_one_sync()) {
#pragma unroll
        for (int kg = 0; kg < 4; ++kg) {
          const uint32_t ko = (uint32_t)kg * (4096u >> 4);
          const uint32_t first = (((touched >> ap) & 1u) == 0u && kg == 0) ? 0u : 1u;
          if (q.passes == 3) {
            mma_tf32_mn<0>(d0, p_lo + ko, q0_hi + ko, idesc, first);
            mma_tf32_mn<1>(d0, p_hi + ko, q0_lo + ko, idesc, 1u);
            mma_tf32_mn<2>(d0, p_hi + ko, q0_hi + ko, idesc, 1u);
            mma_tf32_mn<0>(d1, p_lo + ko, q1_hi + ko, idesc, first);
            mma_tf32_mn<1>(d1, p_hi + ko, q1_lo + ko, idesc, 1u);
            mma_tf32_mn<2>(d1, p_hi + ko, q1_hi + ko, idesc, 1u);
          } else {
            mma_tf32_mn(d0, p_hi + ko, q0_hi + ko, idesc, first);
            mma_tf32_mn(d1, p_hi + ko, q1_hi + ko, idesc, first);
          }
        }
        mma_commit(&empty_bar[s]);
        if (it == niter - 1) mma_commit(&done_bar);
      }
      __syncwarp();
      touched |= (1u << ap);
    }
    if (niter == 0 && elect_one_sync()) mbar_arrive(&done_bar);
    __syncwarp();
  } else if (warp >= 2) {
    const int tid = threadIdx.x - 64;
    // per-iteration operands
    struct Ops { const float* P; long pld; int prows; const float* Q0; const float* Q1; float s0, s1; };
    auto ops_of = [&](int it) -> Ops {
      Ops o;
      if (job == 0) {
        const PaTerm& t = q.term[it / nchunks];
        o.P = arr(t.p_arr); o.pld = LR_ZROW; o.prows = LR_ZROW;
        o.Q0 = arr(t.q_arr); o.Q1 = nullptr; o.s0 = t.s0; o.s1 = t.s1;
      } else if (job == 1) {
        o.P = q.x + (size_t)tile * 128; o.pld = q.D; o.prows = q.D - tile * 128;
        o.Q0 = arr(LA_EPS + 5); o.Q1 = arr(LA_DBT); o.s0 = 1.0f; o.s1 = 1.0f;
      } else {
        o.P = lr_slot_u(S, slot) + (size_t)tile * 128; o.pld = q.D; o.prows = q.D - tile * 128;
        o.Q0 = arr(LA_HBB); o.Q1 = arr(LA_HBT); o.s0 = 1.0f; o.s1 = 1.0f;
      }
      return o;
    };
    const bool pvec = (job == 0) || ((q.D % 4 == 0) && ((((uintptr_t)q.x) & 15) == 0) &&
                                     ((((uintptr_t)lr_slot_u(S, slot)) & 15) == 0));
    // 3072 float4 groups per chunk: [0, 1024) P, [1024, 2048) Q0, [2048, 3072) Q1; group = (sample bl, float4 index c4)
    float4 v[2][6];
    auto load_iter = [&](int it, float4 (&dst)[6]) {
      const Ops o = ops_of(it);
      const int ch = it % nchunks;
#pragma unroll
      for (int g = 0; g < 6; ++g) {
        const int li = tid + (g & 1) * PT;          // g = 0,1: P ; 2,3: Q0 ; 4,5: Q1
        const int bl = li >> 5, c4 = li & 31;
        const int b = b_begin + ch * 32 + bl;
        float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
        if (b < b_end) {
          if (g < 2) {
            const int row = c4 * 4;
            const float* pp = o.P + (size_t)b * o.pld + row;
            if (pvec && row + 3 < o.prows) r = __ldcg(reinterpret_cast<const float4*>(pp));
            else {
              if (row + 0 < o.prows) r.x = __ldcg(pp + 0);
              if (row + 1 < o.prows) r.y = __ldcg(pp + 1);
              if (row + 2 < o.prows) r.z = __ldcg(pp + 2);
              if (row + 3 < o.prows) r.w = __ldcg(pp + 3);
            }
          } else if (g < 4) {
            r = __ldcg(reinterpret_cast<const float4*>(o.Q0 + (size_t)b * LR_ZROW + c4 * 4));
          } else if (o.Q1) {
            r = __ldcg(reinterpret_cast<const float4*>(o.Q1 + (size_t)b * LR_ZROW + c4 * 4));
          }
        }
        dst[g] = r;
      }
    };
    if (niter > 0) load_iter(0, v[0]);
    if (niter > 1) load_iter(1, v[1]);
    for (int it0 = 0; it0 < niter; it0 += 2) {
#pragma unroll
      for (int dd = 0; dd < 2; ++dd) {
        const int it = it0 + dd;
        if (it < niter) {
          const int s = it % NS, ph = (it / NS) & 1;
          uint8_t* stage = smem + (size_t)s * kPaStageBytes;
          const Ops o = ops_of(it);
          mbar_wait(&empty_bar[s], (uint32_t)(ph ^ 1));
#pragma unroll
          for (int g = 0; g < 6; ++g) {
            const int li = tid + (g & 1) * PT;
            const int bl = li >> 5, c4 = li & 31;
            const int grp = c4 >> 3, c32 = (c4 & 7) >> 1, half = c4 & 1, k4 = bl >> 2, r = bl & 3;
            const uint32_t off = (uint32_t)((k4 * 4 + grp) * 512 + r * 128 + ((c32 ^ r) << 5) + half * 16);
            float4 xv = (g >= 4 && !o.Q1) ? v[dd][g - 2] : v[dd][g];
            const float sc = (g < 2) ? 1.0f : ((g < 4) ? o.s0 : o.s1);
            xv.x *= sc; xv.y *= sc; xv.z *= sc; xv.w *= sc;
            float4 hi, lo;
            if (q.passes == 3) {
              hi = make_float4(tf32_rna(xv.x), tf32_rna(xv.y), tf32_rna(xv.z), tf32_rna(xv.w));
              lo = make_float4(tf32_rna(xv.x - hi.x), tf32_rna(xv.y - hi.y), tf32_rna(xv.z - hi.z), tf32_rna(xv.w - hi.w));
            } else { hi = xv; lo = make_float4(0.f, 0.f, 0.f, 0.f); }
            uint8_t* img = stage + (g >> 1) * 32768;
            *reinterpret_cast<float4*>(img + off) = hi;
            *reinterpret_cast<float4*>(img + 16384 + off) = lo;
          }
          if (it + 2 < niter) load_iter(it + 2, v[dd]);
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(&full_bar[s]);
        }
      }
    }
    // epilogue: lane = row of P, columns = rows of Q; partial block [acc][128][128]
    mbar_wait(&done_bar, 0);
    tc_fence_after();
    const int quarter = (warp & 3) * 32;
    const int wgroup = (warp - 2) >> 2;
    const int mrow = quarter + lane;
    const int nacc = (job == 0) ? 4 : 2;
    float* out;
    if (job == 0) out = q.partP + (size_t)split * 4 * 16384;
    else out = (job == 1 ? q.partX : q.partL) + ((size_t)split * q.ntile + tile) * 2 * 16384;
    for (int a = 0; a < nacc; ++a) {
      for (int cb = wgroup; cb < 8; cb += kEpiWarps / 4) {
        float r[16];
        tmem_ld16(tmem_base + ((uint32_t)quarter << 16) + (uint32_t)(a * 128 + cb * 16), r);
        float4* o4 = reinterpret_cast<float4*>(out + (size_t)a * 16384 + (size_t)mrow * 128 + cb * 16);
        if (niter == 0) {
#pragma unroll
          for (int j = 0; j < 16; ++j) r[j] = 0.0f;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) o4[j] = make_float4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------------
// (5) fixed-order reduction of the partial blocks, then the mu block of the attempt
// ---------------------------------------------------------------------------------------------------------
struct AReduceP {
  SolveDev* S;
  const float* partP; const float* partX; const float* partL;
  float* RP; float* RX; float* RL;   // RP[4][128][128]; RX / RL [2][ntile * 128][128]
  int nP, nD, ntile;
};
__global__ void __launch_bounds__(256) adj_reduce_kernel(AReduceP p) {
  if (p.S->done) return;
  const size_t nP4 = 4 * 4096, nX4 = (size_t)p.ntile * 2 * 4096;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nP4 + 2 * nX4; i += (size_t)gridDim.x * blockDim.x) {
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < nP4) {
      const float4* src = reinterpret_cast<const float4*>(p.partP) + i;
#pragma unroll 8
      for (int k = 0; k < p.nP; ++k) {
        const float4 v = __ldcg(src + (size_t)k * nP4);
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      }
      reinterpret_cast<float4*>(p.RP)[i] = s;
    } else {
      const bool isx = (i - nP4) < nX4;
      const size_t j = isx ? (i - nP4) : (i - nP4 - nX4);            // index inside [tile][v][128][128] / 4
      const float4* src = reinterpret_cast<const float4*>(isx ? p.partX : p.partL) + j;
      for (int k = 0; k < p.nD; ++k) {
        const float4 v = __ldcg(src + (size_t)k * nX4);
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      }
      // [tile][v][m][n] -> [v][tile * 128 + m][n]
      const size_t tile = j / (2 * 4096), rem = j % (2 * 4096), vv = rem / 4096, mn = rem % 4096;
      float4* dst = reinterpret_cast<float4*>(isx ? p.RX : p.RL);
      dst[(vv * p.ntile + tile) * 4096 + mn] = s;
    }
  }
}

struct AMuP {
  SolveDev* S;
  const float* RP; const float* RX; const float* RL;
  const float* W2a;   // [D x Kaug] column-major
  const float* W1T;   // [H][D]
  int D, H, td, Kaug, ntile;
  long w1_off, w2_off;   // offsets of the two [out x (in + td + 1)] blocks in the parameter vector
  long nparams;
};
// mu' = -J_p^T lambda:  mu_{n+1} = mu_n - dt dW_b,  utilde = -dt dW_bt,  residual partial sums (perform_step.jl:18-27,34-38)
__global__ void __launch_bounds__(512) adj_mu_kernel(AMuP p) {
  SolveDev* S = p.S;
  if (S->done) return;
  const int slot = S->slot, next = (S->slot + 1) % S->cap;
  const float* mu_n = lr_slot_u(S, slot) + S->lam_len;
  float* mu_new = lr_slot_u(S, next) + S->lam_len;
  const float dt = S->err.scale, abstol = S->abstol, reltol = S->reltol;
  const int H = p.H, D = p.D, Kaug = p.Kaug;
  const long n1 = (long)H * (D + p.td + 1), n2 = (long)D * Kaug;
  const size_t RXs = (size_t)p.ntile * 128 * 128;   // stride between the b and btilde blocks of RX / RL
  const bool multi = S->reduce_mu && S->nranks > 1;
  const int par = (int)(S->mseq & 1ull);
  float* st0 = multi ? lr_mbox_stage(S->mbox[S->rank], par, 0) : nullptr;
  float* st1 = multi ? lr_mbox_stage(S->mbox[S->rank], par, 1) : nullptr;
  double acc = 0.0;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n1 + n2; i += (long)gridDim.x * blockDim.x) {
    float g0, g1;   // dW_b, dW_bt
    long pidx;
    if (i < n1) {
      const int d = (int)(i / H), r = (int)(i % H);
      pidx = p.w1_off + i;
      if (d < D) {
        float a0 = p.RX[(size_t)d * 128 + r], a1 = p.RX[RXs + (size_t)d * 128 + r];
        const float* w = p.W2a + d;
        const float* P0 = p.RP + r;                 // RP[0][k][r]
        const float* P1 = p.RP + 16384 + r;         // RP[1][k][r]
#pragma unroll 8
        for (int k = 0; k < Kaug; ++k) {
          const float wv = __ldg(w + (size_t)k * D);
          a0 = fmaf(P0[k * 128], wv, a0);
          a1 = fmaf(P1[k * 128], wv, a1);
        }
        g0 = a0; g1 = a1;
      } else {
        const int krow = (p.td && d == D) ? Kaug : Kaug + 1;   // time column: sum tau_j delta_j ; bias: sum delta_j
        g0 = p.RP[(size_t)krow * 128 + r];
        g1 = p.RP[16384 + (size_t)krow * 128 + r];
      }
    } else {
      const long i2 = i - n1;
      const int k = (int)(i2 / D), d = (int)(i2 % D);
      pidx = p.w2_off + i2;
      float a0 = 0.0f, a1 = 0.0f;
      const float* P0 = p.RP + 2 * 16384 + (size_t)k * 128;   // RP[2][k][r]
      const float* P1 = p.RP + 3 * 16384 + (size_t)k * 128;   // RP[3][k][r]
      const float* w = p.W1T + d;
#pragma unroll 8
      for (int r = 0; r < H; ++r) {
        const float wv = __ldg(w + (size_t)r * D);
        a0 = fmaf(P0[r], wv, a0);
        a1 = fmaf(P1[r], wv, a1);
      }
      g0 = fmaf(-dt, a0, p.RL[(size_t)d * 128 + k]);
      g1 = fmaf(-dt, a1, p.RL[RXs + (size_t)d * 128 + k]);
    }
    if (multi) {   // this rank's batch-partial sums: published, summed over ranks by adj_mu_finish_kernel
      st0[pidx] = g0;
      st1[pidx] = g1;
      continue;
    }
    const float mn = mu_n[pidx];
    const float mv = fmaf(-dt, g0, mn);
    mu_new[pidx] = mv;
    const float ut = -dt * g1;
    const float r = ut / (abstol + fmaxf(fabsf(mn), fabsf(mv)) * reltol);
    acc += (double)(r * r);
  }
  if (multi) {
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned int prev = atomicAdd(S->mucounter, 1u);
      if (prev == gridDim.x - 1) {   // last block: everything of this rank is visible, raise the flags on every peer
        *S->mucounter = 0;
        __threadfence_system();
        for (int r = 0; r < S->nranks; ++r) {
          volatile unsigned long long* f = &S->mbox[r]->mflag[par][S->rank];
          *f = S->mseq + 1;
        }
      }
    }
    return;
  }
  // block sum (fixed order)
  __shared__ double sh[16];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += sh[w];
    S->partials[LR_ERR_BLOCKS + blockIdx.x] = s;
  }
}

// Data-parallel group (SURVEY 8e): mu is a batch sum and enters the error norm non-linearly, so every rank adds all
// ranks' (dW_b, dW_bt) in rank order (identical bits everywhere) and advances a replicated GLOBAL mu (S->muglob, one
// vector per ring slot) for the norm, next to its own batch-partial mu in the state (what the caller all-reduces).
// The exchange sequence number is advanced by controller_kernel.
__global__ void __launch_bounds__(256) adj_mu_finish_kernel(SolveDev* S) {
  if (S->done) return;
  const int par = (int)(S->mseq & 1ull);
  LrMailbox* mine = S->mbox[S->rank];
  if (threadIdx.x == 0) {
    long long spins = 0;
    for (int r = 0; r < S->nranks; ++r) {
      volatile unsigned long long* f = &mine->mflag[par][r];
      while (*f != S->mseq + 1) {
        __nanosleep(40);
        if (++spins > (1ll << 26)) { lr_peer_timeout(S); break; }   // a peer never arrived (~10 s): give up instead of hanging
      }
    }
    __threadfence_system();
  }
  __syncthreads();
  const int slot = S->slot, next = (S->slot + 1) % S->cap;
  const size_t P = S->mu_len;
  const float* mu_n = lr_slot_u(S, slot) + S->lam_len;
  float* mu_new = lr_slot_u(S, next) + S->lam_len;
  const float* mg_n = S->muglob + (size_t)slot * P;
  float* mg_new = S->muglob + (size_t)next * P;
  const float* own0 = lr_mbox_stage(mine, par, 0);
  const float dt = S->err.scale, abstol = S->abstol, reltol = S->reltol;
  double acc = 0.0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < P; i += (size_t)gridDim.x * blockDim.x) {
    float g0 = 0.0f, g1 = 0.0f;
    for (int r = 0; r < S->nranks; ++r) {
      g0 += ((const volatile float*)lr_mbox_stage(S->mbox[r], par, 0))[i];
      g1 += ((const volatile float*)lr_mbox_stage(S->mbox[r], par, 1))[i];
    }
    mu_new[i] = fmaf(-dt, ((const volatile float*)own0)[i], mu_n[i]);
    const float mn = mg_n[i];
    const float mv = fmaf(-dt, g0, mn);
    mg_new[i] = mv;
    const float ut = -dt * g1;
    const float rr = ut / (abstol + fmaxf(fabsf(mn), fabsf(mv)) * reltol);
    acc += (double)(rr * rr);
  }
  __shared__ double sh[8];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += sh[w];
    S->partials[LR_ERR_BLOCKS + blockIdx.x] = s;
  }
}

}  // namespace ladj

// ---------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------
#define LRA_COUNT(ctx) do { if ((ctx)->capturing) (ctx)->captured++; else (ctx)->launches++; } while (0)

bool LatentAdjoint::eligible(const lrnde_model* m) {
  FusedShape s;
  if (!lrf_shape(m, &s)) return false;
  return s.KS <= 14 && s.Kaug + 2 <= 128;
}

LatentAdjoint::LatentAdjoint(lrnde_ctx* c, const lrnde_model* mm, const float* p, int64_t b, int npasses)
    : ctx(c), m(mm), ps(p), B(b), passes(npasses) {
  lrf_shape(m, &sh);
  ntiles = (int)((B + fused::kNT - 1) / fused::kNT);
  zlen = (size_t)LR_ZROW * (size_t)ntiles * fused::kNT;   // work arrays padded to whole 64-sample tiles (adj_pre_kernel)
  nunits = (int)((B + 15) / 16);
  unit_bytes = (size_t)sh.nfull * 8192 + (size_t)sh.ntail * 2048;
  const int maxc = std::max(1, 148 / sh.n_mt);
  const int rounds = (nunits + maxc - 1) / maxc;
  nclusters = (nunits + rounds - 1) / rounds;
  ntile_d = (sh.D + 127) / 128;
  // pairacc: hidden-space terms (13 x B sample-terms) and the two D-dimensional terms (2 x ntile x B) share one wave
  const int nchunk_tot = (int)((B + 31) / 32);
  const double wP = 13.0, wD = 2.0 * ntile_d;
  int wantP = std::max(1, (int)(148.0 * wP / (wP + wD)));
  int cP = std::max(1, (nchunk_tot + wantP - 1) / wantP);
  chunkP = cP * 32;
  nP = (int)((B + chunkP - 1) / chunkP);
  int wantD = std::max(1, (148 - nP) / (2 * ntile_d));
  int cD = std::max(1, (nchunk_tot + wantD - 1) / wantD);
  chunkD = cD * 32;
  nD = (int)((B + chunkD - 1) / chunkD);
  Mz = (float*)ctx->alloc(sizeof(float) * 128 * 128);
  ws = (float*)ctx->alloc(sizeof(float) * LA_NARR * zlen);
  alpha_in = (float*)ctx->alloc(sizeof(float) * zlen);
  hbuf = (float*)ctx->alloc((size_t)ntiles * 4 * unit_bytes);
  partP = (float*)ctx->alloc(sizeof(float) * (size_t)nP * 4 * 16384);
  partX = (float*)ctx->alloc(sizeof(float) * (size_t)nD * ntile_d * 2 * 16384);
  partL = (float*)ctx->alloc(sizeof(float) * (size_t)nD * ntile_d * 2 * 16384);
  RP = (float*)ctx->alloc(sizeof(float) * 4 * 16384);
  RX = (float*)ctx->alloc(sizeof(float) * (size_t)ntile_d * 2 * 16384);
  RL = (float*)ctx->alloc(sizeof(float) * (size_t)ntile_d * 2 * 16384);
  int dev = 0, nsm = 0;
  LR_CUDA(cudaGetDevice(&dev));
  LR_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
  pre_ctas = std::max(1, std::min(ntiles, nsm));
  static bool attr_set = false;
  if (!attr_set) {
    // KS <= 14: at most 3 full chunks + 3 tail K-steps per operand tile
    constexpr int kTiles4 = 4 * (3 * 8192 + 3 * 2048);
    constexpr int kChainSmem = kTiles4 + ladj::kTapeBufs * ladj::kTapeBufBytes + 1024, kPreSmem = kTiles4 + 1024;
    LR_CUDA(cudaFuncSetAttribute(ladj::adj_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kChainSmem));
#define LRA_PRE_ATTR(A) do { \
      LR_CUDA(cudaFuncSetAttribute(ladj::adj_pre_kernel<A, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPreSmem)); \
      LR_CUDA(cudaFuncSetAttribute(ladj::adj_pre_kernel<A, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPreSmem)); } while (0)
    LRA_PRE_ATTR(ACT_IDENTITY); LRA_PRE_ATTR(ACT_TANH); LRA_PRE_ATTR(ACT_GELU); LRA_PRE_ATTR(ACT_SIGMOID); LRA_PRE_ATTR(ACT_RELU);
#undef LRA_PRE_ATTR
    LR_CUDA(cudaFuncSetAttribute(ladj::pairacc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ladj::pairacc_smem()));
    attr_set = true;
  }
  if (getenv("LRNDE_FUSED_VERBOSE"))
    fprintf(stderr, "[lrnde adjoint] B=%lld tiles=%d units=%d kgemm clusters=%d pairacc: nP=%d x %d samples, nD=%d x %d samples x %d tiles\n",
            (long long)B, ntiles, nunits, nclusters, nP, chunkP, nD, chunkD, ntile_d);
}

LatentAdjoint::~LatentAdjoint() {
  ctx->release(Mz); ctx->release(ws); ctx->release(alpha_in); ctx->release(hbuf);
  ctx->release(partP); ctx->release(partX); ctx->release(partL);
  ctx->release(RP); ctx->release(RX); ctx->release(RL);
}

void LatentAdjoint::prepare(const float* mz_plain) {
  if (mz_plain) { Mz_ext = mz_plain; return; }   // kept by the forward call (lrnde_tape)
  lrf_mz_plain(ctx, m, ps, Mz);
  LRA_COUNT(ctx);
}

// (0) interpolant, (1) pre kernel and, for an attempt, (2) the chain kernel; single: stage 1 of the current state only
static void lra_launch_chain(LatentAdjoint& E, SolveDev* S, int single) {
  const FusedShape& sh = E.sh;
  const LayerInfo& L1 = E.m->layers[0];
  const float* Mz = E.Mz_ext ? E.Mz_ext : E.Mz;
  const size_t tiles4 = 4 * ((size_t)sh.nfull * 8192 + (size_t)sh.ntail * 2048);
  cudaStream_t st = E.ctx->stream;
  ladj::AInterpP ip;
  ip.S = S; ip.single = single; ip.ws = E.ws; ip.zlen = E.zlen; ip.B = (int)E.B; ip.Kaug = sh.Kaug;
  ip.nunit = E.ntiles * fused::kNT * (LR_ZROW / 4);
  ladj::adj_interp_kernel<<<(ip.nunit + 255) / 256, 256, 0, st>>>(ip);
  LRA_COUNT(E.ctx);
  ladj::APreP pp;
  memset(&pp, 0, sizeof(pp));
  pp.S = S; pp.Mz = Mz;
  pp.w1t = sh.td ? E.ps + L1.w_off + (size_t)sh.D * sh.H : nullptr;
  pp.b1 = E.ps + L1.b_off;
  pp.Zx = E.Zx; pp.alpha_in = E.alpha_in; pp.ws = E.ws; pp.zlen = E.zlen;
  pp.H = sh.H; pp.td = sh.td; pp.Kaug = sh.Kaug; pp.KS = sh.KS; pp.nfull = sh.nfull; pp.ntail = sh.ntail;
  pp.passes = E.passes; pp.ntiles = E.ntiles;
  const size_t smem_p = tiles4 + 1024;
#define LRA_PRE(A) do { if (single) ladj::adj_pre_kernel<A, true><<<E.pre_ctas, fused::kThreads, smem_p, st>>>(pp); \
                       else ladj::adj_pre_kernel<A, false><<<E.pre_ctas, fused::kThreads, smem_p, st>>>(pp); } while (0)
  switch (sh.act) {
    case ACT_TANH: LRA_PRE(ACT_TANH); break;
    case ACT_GELU: LRA_PRE(ACT_GELU); break;
    case ACT_SIGMOID: LRA_PRE(ACT_SIGMOID); break;
    case ACT_RELU: LRA_PRE(ACT_RELU); break;
    default: LRA_PRE(ACT_IDENTITY); break;
  }
#undef LRA_PRE
  LRA_COUNT(E.ctx);
  if (!single) {
    ladj::AChainP cp;
    memset(&cp, 0, sizeof(cp));
    cp.S = S; cp.Mz = Mz; cp.ws = E.ws; cp.zlen = E.zlen;
    cp.hbuf = E.hbuf; cp.unit_bytes = (uint32_t)E.unit_bytes;
    cp.H = sh.H; cp.Kaug = sh.Kaug; cp.KS = sh.KS; cp.nfull = sh.nfull; cp.ntail = sh.ntail; cp.passes = E.passes;
    const size_t smem_c = tiles4 + ladj::kTapeBufs * ladj::kTapeBufBytes + 1024;
    ladj::adj_chain_kernel<<<E.ntiles, fused::kThreads, smem_c, st>>>(cp);
    LRA_COUNT(E.ctx);
  }
  LR_CUDA(cudaGetLastError());
}

static void lra_launch_pairacc(LatentAdjoint& E, SolveDev* S) {
  ladj::PairAccP q;
  memset(&q, 0, sizeof(q));
  q.S = S; q.ws = E.ws; q.zlen = E.zlen; q.x = E.x; q.D = E.sh.D; q.B = (int)E.B;
  q.nP = E.nP; q.chunkP = E.chunkP; q.nD = E.nD; q.chunkD = E.chunkD; q.ntile = E.ntile_d;
  q.partP = E.partP; q.partX = E.partX; q.partL = E.partL; q.passes = E.passes;
  // sum_j w_j delta_j c_j^T (accumulators 0, 1) and sum_j w_j eps_j H_j^T (2, 3); w = b, btilde; eps_1 = 0
  int n = 0;
  for (int j = 1; j <= 7; ++j) {
    const float bj = (j <= 6) ? lr_tsit5_a(5, j - 1) : 0.0f;
    const float btj = lr_tsit5_btilde(j - 1);
    const int del = (j == 1) ? -1 : ((j == 7) ? -10 : LA_DEL + j - 2);
    const int hh = (j == 1) ? -2 : ((j == 7) ? -11 : LA_HH + j - 2);
    const int cc = (j == 1) ? -3 : ((j == 7) ? -12 : LA_CC + j - 2);
    q.term[n++] = {cc, del, bj, btj, 0};
    if (j >= 2) q.term[n++] = {hh, LA_EPS + j - 2, bj, btj, 1};
  }
  q.nterm = n;
  const int grid = E.nP + 2 * E.ntile_d * E.nD;
  ladj::pairacc_kernel<<<grid, fused::kThreads, ladj::pairacc_smem(), E.ctx->stream>>>(q);
  LRA_COUNT(E.ctx);
  LR_CUDA(cudaGetLastError());
}

static void lra_launch_mu(LatentAdjoint& E, SolveDev* S) {
  cudaStream_t st = E.ctx->stream;
  ladj::AReduceP r;
  r.S = S; r.partP = E.partP; r.partX = E.partX; r.partL = E.partL; r.RP = E.RP; r.RX = E.RX; r.RL = E.RL;
  r.nP = E.nP; r.nD = E.nD; r.ntile = E.ntile_d;
  const size_t n4 = 4 * 4096 + 2 * (size_t)E.ntile_d * 2 * 4096;
  ladj::adj_reduce_kernel<<<(int)((n4 + 255) / 256), 256, 0, st>>>(r);
  LRA_COUNT(E.ctx);
  const LayerInfo& L1 = E.m->layers[0];
  const LayerInfo& L2 = E.m->layers[1];
  ladj::AMuP mp;
  memset(&mp, 0, sizeof(mp));
  mp.S = S; mp.RP = E.RP; mp.RX = E.RX; mp.RL = E.RL;
  mp.W2a = E.ps + L2.w_off; mp.W1T = E.W1T;
  mp.D = E.sh.D; mp.H = E.sh.H; mp.td = E.sh.td; mp.Kaug = E.sh.Kaug; mp.ntile = E.ntile_d;
  mp.w1_off = (long)L1.w_off; mp.w2_off = (long)L2.w_off; mp.nparams = (long)E.m->nparams;
  ladj::adj_mu_kernel<<<LR_ERR_BLOCKS, 512, 0, st>>>(mp);
  LRA_COUNT(E.ctx);
  if (E.ctx->nranks > 1) {
    ladj::adj_mu_finish_kernel<<<LR_ERR_BLOCKS, 256, 0, st>>>(S);
    LRA_COUNT(E.ctx);
  }
  LR_CUDA(cudaGetLastError());
}

void LatentAdjoint::begin(SolveDev* S) { lra_launch_chain(*this, S, 1); }

void LatentAdjoint::attempt(SolveDev* S) {
  lra_launch_chain(*this, S, 0);
  lrf_launch_kgemm_adj(ctx, S, sh, ps + m->layers[0].w_off, hbuf, unit_bytes, B, passes, nunits, nclusters);
  lra_launch_pairacc(*this, S);
  lra_launch_mu(*this, S);
}

void LatentAdjoint::attempt_part(SolveDev* S, int which) {
  if (which == 0) lra_launch_chain(*this, S, 0);
  else if (which == 1) lrf_launch_kgemm_adj(ctx, S, sh, ps + m->layers[0].w_off, hbuf, unit_bytes, B, passes, nunits, nclusters);
  else if (which == 2) lra_launch_pairacc(*this, S);
  else lra_launch_mu(*this, S);
}
