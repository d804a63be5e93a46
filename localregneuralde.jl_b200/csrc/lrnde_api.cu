// libLRNDE.so -- host orchestration + C ABI (include/lrnde.h).
//
// The layer logic restated here is the reference's src/layers/neural_ode.jl:56-116 (mode
// dispatch, saveat resolution, t1, nfe bookkeeping); the solver loop, initial-dt heuristic and
// continuous adjoint are the un-vendored OrdinaryDiffEq / SciMLSensitivity algorithms of
// SURVEY App. A.  All arithmetic happens in kernels (lrnde_kernels.cuh, lrnde_umma.cuh); the
// host only sequences launches and never waits inside a solve.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <functional>
#include <memory>

#include "lrnde_host.h"
#include "lrnde_kernels.cuh"
#include "lrnde_umma.cuh"
#include "lrnde_smem_mlp.cuh"
#include "lrnde_conv.cuh"
#include "lrnde_conv_tc.h"
#include "lrnde_fused.h"
#include "lrnde_adjoint.h"
#include "lrnde_regrev.cuh"
#include "lrnde_saveplan.h"

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
void lr_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
extern "C" const char* lrnde_last_error(void) { return g_err; }
extern "C" int lrnde_version(void) { return 100; }

#define LR_API_BEGIN try {
#define LR_API_END                                     \
  }                                                    \
  catch (const LrError& e) { return e.code; }          \
  catch (const std::bad_alloc&) {                      \
    lr_set_error("host out of memory");                \
    return LRNDE_ENOMEM;                               \
  }                                                    \
  return LRNDE_OK;

static inline long lr_now_us() {
  return (long)std::chrono::duration_cast<std::chrono::microseconds>(
             std::chrono::steady_clock::now().time_since_epoch()).count();
}

static void lr_fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  throw LrError(code);
}

// ------------------------------------------------------------------------------------------
// ctx: device memory pool (cudaMalloc synchronises; blocks are recycled across calls)
// ------------------------------------------------------------------------------------------
void* lrnde_ctx::alloc(size_t bytes) {
  if (bytes == 0) bytes = 256;
  bytes = (bytes + 255) & ~(size_t)255;
  int best = -1;
  for (size_t i = 0; i < pool.size(); ++i) {
    if (!pool[i].used && pool[i].bytes >= bytes && pool[i].bytes <= 2 * bytes + (1 << 20)) {
      if (best < 0 || pool[i].bytes < pool[best].bytes) best = (int)i;
    }
  }
  if (best >= 0) {
    pool[best].used = true;
    return pool[best].p;
  }
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    release_all_unused();
    e = cudaMalloc(&p, bytes);
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    lr_fail(LRNDE_ENOMEM, "cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
  }
  pool.push_back({p, bytes, true});
  return p;
}
void lrnde_ctx::release(void* p) {
  if (!p) return;
  for (auto& b : pool)
    if (b.p == p) { b.used = false; return; }
}
void lrnde_ctx::release_all_unused() {
  std::vector<PoolBlock> keep;
  for (auto& b : pool) {
    if (b.used) keep.push_back(b);
    else cudaFree(b.p);
  }
  pool.swap(keep);
}

#define LR_COUNT(ctx) do { if ((ctx)->capturing) (ctx)->captured++; else (ctx)->launches++; } while (0)
#define LR_CHECK_LAUNCH() LR_CUDA(cudaGetLastError())

static inline int lr_ew_blocks(size_t n) {
  size_t b = (n + 255) / 256;
  if (b < 1) b = 1;
  if (b > 148 * 8) b = 148 * 8;
  return (int)b;
}

struct DevBuf {  // pooled device scratch with RAII
  lrnde_ctx* ctx;
  float* p;
  DevBuf(lrnde_ctx* c, size_t nfloat) : ctx(c), p((float*)c->alloc(sizeof(float) * nfloat)) {}
  ~DevBuf() { ctx->release(p); }
};

// The caller's arrays of one C entry point: host memory when the call has host_buffers, device memory otherwise.
// Kernels see only the device pointers this hands out; n counts elements.  Two kinds each way:
//   in / out            staged: the caller's device array is used in place; a host array goes through a pooled
//                       buffer (copied in now, or back by finish())
//   copy_in / copy_out  owned copy: always a pooled buffer (or `dst` / `src`, a device buffer the entry point
//                       owns), copied from / back to the caller either way.  For arrays the call overwrites,
//                       arrays a tape keeps past the call, and kernels that want the pool's 256-byte alignment
//                       or must not alias another argument
// A NULL array gets no buffer and no copy.  Copies run on ctx->stream; finish() queues the copies back in the order
// the outputs were declared and does not synchronise.
struct CallerBufs {
  lrnde_ctx* ctx;
  const bool host;
  CallerBufs(lrnde_ctx* c, int host_buffers) : ctx(c), host(host_buffers != 0) {}
  ~CallerBufs() { for (void* q : pooled_) ctx->release(q); }
  CallerBufs(const CallerBufs&) = delete;
  CallerBufs& operator=(const CallerBufs&) = delete;

  template <class T> const T* in(const T* p, size_t n) { return (p && host) ? copy_in(p, n) : p; }
  template <class T> T* copy_in(const T* p, size_t n) {
    if (!p) return nullptr;
    T* d = pool<T>(n);
    copy_in(d, p, n);
    return d;
  }
  template <class T> void copy_in(T* dst, const T* p, size_t n) {
    if (p)
      LR_CUDA(cudaMemcpyAsync(dst, p, sizeof(T) * n, host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice,
                              ctx->stream));
  }
  template <class T> T* out(T* p, size_t n) { return (p && host) ? copy_out(p, n) : p; }
  template <class T> T* copy_out(T* p, size_t n) {
    if (!p) return nullptr;
    T* d = pool<T>(n);
    copy_out(p, (const T*)d, n);
    return d;
  }
  template <class T> void copy_out(T* p, const T* src, size_t n) {
    if (p) back_.push_back({p, src, sizeof(T) * n});
  }
  // staged input that the call also writes back (BatchNorm running statistics)
  template <class T> T* inout(T* p, size_t n) {
    if (!p || !host) return p;
    T* d = copy_in(p, n);
    copy_out(p, (const T*)d, n);
    return d;
  }
  void finish() {
    for (const Back& b : back_)
      LR_CUDA(cudaMemcpyAsync(b.dst, b.src, b.bytes, host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice,
                              ctx->stream));
    back_.clear();
  }

 private:
  struct Back { void* dst; const void* src; size_t bytes; };
  std::vector<void*> pooled_;
  std::vector<Back> back_;
  template <class T> T* pool(size_t n) {
    T* d = (T*)ctx->alloc(sizeof(T) * n);
    pooled_.push_back(d);
    return d;
  }
};

extern "C" int lrnde_ctx_create(lrnde_ctx** out, int device, void* stream) {
  LR_API_BEGIN
  if (!out) lr_fail(LRNDE_EINVAL, "lrnde_ctx_create: out is NULL");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    lr_fail(LRNDE_ECUDA, "libLRNDE needs a CUDA device (sm_100a); none is visible: %s",
            cudaGetErrorString(e));
  if (device < 0 || device >= ndev) lr_fail(LRNDE_EINVAL, "device %d out of range", device);
  LR_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  LR_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    lr_fail(LRNDE_ECUDA, "libLRNDE is built for sm_100a only; device %d is sm_%d%d", device,
            prop.major, prop.minor);
  auto* c = new lrnde_ctx();
  c->device = device;
  if (stream) c->stream = (cudaStream_t)stream;
  else {
    // a BLOCKING stream: it synchronises implicitly with the legacy default stream (stream 0), so a caller that
    // prepares its buffers on stream 0 (PyTorch's default stream has handle 0) and passes NULL cannot race with the
    // library: work queued on stream 0 before a call is complete before the library's kernels start, and stream-0
    // work queued after the call waits for them.  (Graph capture needs a non-default stream, hence not stream 0 itself.)
    LR_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamDefault));
    c->own_stream = true;
  }
  c->pinned_bytes = 1 << 20;
  LR_CUDA(cudaMallocHost(&c->pinned, c->pinned_bytes));
  *out = c;
  LR_API_END
}

extern "C" int lrnde_ctx_destroy(lrnde_ctx* c) {
  LR_API_BEGIN
  if (!c) return LRNDE_OK;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  for (auto& b : c->pool) cudaFree(b.p);
  if (c->mailbox) cudaFree(c->mailbox);
  if (c->bn_seq) cudaFree(c->bn_seq);
  for (auto& sg : c->staged) {
    if (sg.x) cudaFree(sg.x);
    if (sg.y) cudaFree(sg.y);
    if (sg.ev) cudaEventDestroy(sg.ev);
  }
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  for (auto& cg : c->graph_cache) { cudaGraphExecDestroy(cg.exec); cudaGraphDestroy(cg.graph); }
  if (c->pinned) cudaFreeHost(c->pinned);
  if (c->own_stream) cudaStreamDestroy(c->stream);
  delete c;
  LR_API_END
}

extern "C" int lrnde_ctx_sync(lrnde_ctx* c) {
  LR_API_BEGIN
  if (!c) lr_fail(LRNDE_EINVAL, "ctx is NULL");
  LR_CUDA(cudaSetDevice(c->device));
  LR_CUDA(cudaStreamSynchronize(c->stream));
  LR_API_END
}

extern "C" int lrnde_ctx_set_tape_budget(lrnde_ctx* c, uint64_t bytes) {
  LR_API_BEGIN
  if (!c) lr_fail(LRNDE_EINVAL, "ctx is NULL");
  c->tape_budget = bytes;
  LR_API_END
}

extern "C" int lrnde_ctx_mailbox(lrnde_ctx* c, void** dev_ptr, uint64_t* bytes) {
  LR_API_BEGIN
  if (!c || !dev_ptr) lr_fail(LRNDE_EINVAL, "ctx/dev_ptr is NULL");
  LR_CUDA(cudaSetDevice(c->device));
  if (!c->mailbox) {
    // a dedicated cudaMalloc so the block can be exported with cudaIpcGetMemHandle
    LR_CUDA(cudaMalloc((void**)&c->mailbox, LR_MAILBOX_BYTES));
    LR_CUDA(cudaMemset(c->mailbox, 0, LR_MAILBOX_BYTES));
  }
  *dev_ptr = c->mailbox;
  if (bytes) *bytes = LR_MAILBOX_BYTES;
  LR_API_END
}

extern "C" int lrnde_ctx_set_dist(lrnde_ctx* c, int rank, int nranks, void* const* mailboxes,
                                  int64_t total_batch) {
  LR_API_BEGIN
  if (!c) lr_fail(LRNDE_EINVAL, "ctx is NULL");
  if (nranks < 1 || nranks > LR_MAX_RANKS || rank < 0 || rank >= nranks)
    lr_fail(LRNDE_EINVAL, "bad rank/nranks %d/%d (max %d)", rank, nranks, LR_MAX_RANKS);
  if (nranks > 1 && !mailboxes) lr_fail(LRNDE_EINVAL, "mailboxes is NULL");
  c->rank = rank;
  c->nranks = nranks;
  c->total_batch = total_batch;
  for (int r = 0; r < nranks && nranks > 1; ++r) c->peer_mbox[r] = (LrMailbox*)mailboxes[r];
  // the exchange sequence numbers (seq, mseq, bn_seq) are NOT reset: the mailbox flags of earlier exchanges stay in
  // place, and every rank of the group calls this the same number of times, so the counters stay in step
  LR_CUDA(cudaSetDevice(c->device));
  if (!c->bn_seq) {
    LR_CUDA(cudaMalloc((void**)&c->bn_seq, sizeof(unsigned long long) * (LR_BN_MAXC + 1)));
    LR_CUDA(cudaMemset(c->bn_seq, 0, sizeof(unsigned long long) * (LR_BN_MAXC + 1)));
  }
  LR_API_END
}

BnDist lrnde_ctx::bn_dist() {
  BnDist d;
  memset(&d, 0, sizeof(d));
  d.rank = rank;
  d.nranks = bn_seq ? nranks : 1;
  for (int r = 0; r < LR_MAX_RANKS; ++r) d.mbox[r] = peer_mbox[r];
  d.seq = bn_seq;
  d.timed_out = bn_seq ? (int*)(bn_seq + LR_BN_MAXC) : nullptr;
  return d;
}

void lrnde_ctx::bn_check() {
  if (nranks <= 1 || !bn_seq) return;
  int flag = 0;
  LR_CUDA(cudaMemcpyAsync(&flag, bn_seq + LR_BN_MAXC, sizeof(int), cudaMemcpyDeviceToHost, stream));
  LR_CUDA(cudaStreamSynchronize(stream));
  if (flag) lr_fail(LRNDE_ESTATE, "BatchNorm statistics exchange: a rank of the data-parallel group did not arrive within ~10 s");
}

// ------------------------------------------------------------------------------------------
// model
// ------------------------------------------------------------------------------------------
static int lr_map_act(int a) {
  switch (a) {
    case LRNDE_ACT_IDENTITY: case LRNDE_ACT_NONE: return ACT_IDENTITY;
    case LRNDE_ACT_TANH: return ACT_TANH;
    case LRNDE_ACT_GELU: return ACT_GELU;
    case LRNDE_ACT_SIGMOID: return ACT_SIGMOID;
    case LRNDE_ACT_RELU: return ACT_RELU;
  }
  lr_fail(LRNDE_EINVAL, "unknown activation %d", a);
  return 0;
}

extern "C" int lrnde_model_create(lrnde_ctx* ctx, const lrnde_layer_desc* layers, int nlayers,
                                  int time_dependent, int input_act, lrnde_model** out) {
  LR_API_BEGIN
  if (!ctx || !layers || !out || nlayers < 1) lr_fail(LRNDE_EINVAL, "lrnde_model_create: bad args");
  auto m = std::make_unique<lrnde_model>();
  m->ctx = ctx;
  m->td = time_dependent ? 1 : 0;
  m->input_act = lr_map_act(input_act);
  int64_t off = 0;
  for (int l = 0; l < nlayers; ++l) {
    LayerInfo L;
    L.in = layers[l].in_dims;
    L.out = layers[l].out_dims;
    if (L.in < 1 || L.out < 1) lr_fail(LRNDE_EINVAL, "layer %d: bad dims", l);
    L.act = lr_map_act(layers[l].act);
    L.w_off = off;
    off += (int64_t)L.out * (L.in + m->td);
    L.b_off = off;
    off += L.out;
    if (l > 0 && m->layers.back().out != L.in)
      lr_fail(LRNDE_EINVAL, "layer %d: in_dims %d != previous out_dims %d", l, L.in,
              m->layers.back().out);
    m->layers.push_back(L);
  }
  if (m->layers.front().in != m->layers.back().out)
    lr_fail(LRNDE_EINVAL, "dynamics must map R^D -> R^D (got %d -> %d)", m->layers.front().in,
            m->layers.back().out);
  m->nparams = off;
  m->D = m->layers.front().in;
  *out = m.release();
  LR_API_END
}
extern "C" int lrnde_conv_model_create(lrnde_ctx* ctx, const lrnde_conv_layer_desc* layers, int nlayers, int width,
                                       int height, int time_dependent, lrnde_model** out) {
  LR_API_BEGIN
  if (!ctx || !layers || !out || nlayers < 1) lr_fail(LRNDE_EINVAL, "lrnde_conv_model_create: bad args");
  if (width < 4 || width > 32 || (width & 3) || height < 1)
    lr_fail(LRNDE_EINVAL, "lrnde_conv_model_create: width must be a multiple of 4 in 4..32 (got %d x %d)", width, height);
  auto m = std::make_unique<lrnde_model>();
  m->ctx = ctx;
  m->td = time_dependent ? 1 : 0;
  m->input_act = ACT_IDENTITY;
  m->Wd = width; m->Ht = height;
  int64_t off = 0;
  for (int l = 0; l < nlayers; ++l) {
    ConvLayerInfo L;
    L.cin = layers[l].in_ch; L.cout = layers[l].out_ch; L.bn = layers[l].batchnorm ? 1 : 0;
    L.act = lr_map_act(layers[l].act);
    if (L.cin < 1 || L.cout < 1) lr_fail(LRNDE_EINVAL, "conv layer %d: bad channel counts", l);
    if (l > 0 && m->conv.back().cout != L.cin)
      lr_fail(LRNDE_EINVAL, "conv layer %d: in_ch %d != previous out_ch %d", l, L.cin, m->conv.back().cout);
    L.w_off = off; off += (int64_t)9 * (L.cin + m->td) * L.cout;
    L.g_off = off; if (L.bn) off += 2 * (int64_t)L.cout;
    m->conv.push_back(L);
  }
  if (m->conv.back().bn || m->conv.back().act != ACT_IDENTITY)
    lr_fail(LRNDE_EINVAL, "the last layer of the conv dynamics must be a plain Conv (no BatchNorm / activation)");
  if (m->conv.front().cin != m->conv.back().cout)
    lr_fail(LRNDE_EINVAL, "dynamics must map the state onto itself (got %d -> %d channels)", m->conv.front().cin,
            m->conv.back().cout);
  m->nparams = off;
  m->D = width * height * m->conv.front().cin;
  *out = m.release();
  LR_API_END
}
extern "C" int lrnde_model_destroy(lrnde_model* m) {
  delete m;
  return LRNDE_OK;
}
extern "C" int64_t lrnde_model_nparams(const lrnde_model* m) { return m ? m->nparams : -1; }
extern "C" int64_t lrnde_model_state_dims(const lrnde_model* m) { return m ? m->D : -1; }

// ------------------------------------------------------------------------------------------
// Conv evaluator (lrnde_conv.cuh): the same forward / vjp contract as MlpEval below
// ------------------------------------------------------------------------------------------
struct ConvEval {
  lrnde_ctx* ctx;
  const lrnde_model* m;
  const float* ps;
  int64_t B;
  bool with_vjp;
  int L, maxC = 0, nblk_max = 0;
  size_t HW;
  std::vector<float*> z, ab, stat, pack, packT;
  float2* spart = nullptr;
  float* ybuf = nullptr; float* lbuf = nullptr; float* G[2] = {nullptr, nullptr};
  float* part = nullptr; double2* bpart = nullptr; float* coef = nullptr; float* dgb = nullptr;
  std::vector<int> wS, wImg, wCic, wChunks, wSwap;
  int bnS = 1, bnImg = 1;
  // st.model of the layer: running statistics of every BatchNorm (device), see lrnde_opts.model_state
  float* bn_state = nullptr;
  std::vector<int64_t> s_off;
  int64_t nstate = 0;
  int testmode = 0;
  bool bn_update = false;
  bool first_call_twice = false;  // OrdinaryDiffEq calls f(u0, t0) twice (initialize! and the initial-dt heuristic);
                                  // the library evaluates it once, the running statistics see two closure calls
  // tensor-core engine (lrnde_conv_tc.h): every layer has channel counts that are multiples of 8 and at most 64
  bool tc = false;
  ConvTcGeom geo;
  float* Fhi = nullptr; float* Flo = nullptr;           // (F) operand of the convolution about to run
  std::vector<uint8_t*> wimg, wimgT;                    // weight images: forward / data-gradient convolution
  std::vector<float*> tsum;                             // time-channel tables
  bool wg_tc = false;                                   // weight gradients on the tensor cores as well (Wd == 32)
  float* PD = nullptr;                                  // plain fp32 cotangent of the layer at hand (operand of its weight gradient)
  float* rowsum = nullptr;                              // per-row sums of that cotangent (time channel's weight gradient)

  static bool tc_eligible(const lrnde_model* m) {
    const char* e = getenv("LRNDE_CONV_TC");
    if (e && e[0] == '0') return false;
    for (auto& Li : m->conv)
      if ((Li.cin & 7) || (Li.cout & 7) || Li.cin > 64 || Li.cout > 64) return false;
    return m->Wd + 3 <= kCtGuard;
  }
  // haloed positions of the batch are indexed with 32 bits inside the kernels
  static bool tc_fits(const lrnde_model* m, int64_t b) { return (double)b * (m->Wd + 2) * (m->Ht + 2) < 2.0e9; }

  static int tile_rows(int PT, int Wd, int Ht) { return std::min(PT / (Wd >> 2), Ht); }
  static bool narrow(int cout) { return cout <= 16; }   // <8,8,4> instantiation (whole-image tiles)
  int conv_nblk(int cout) const {
    const int TR = tile_rows(narrow(cout) ? 256 : 64, m->Wd, m->Ht);
    return (int)B * ((m->Ht + TR - 1) / TR);
  }

  ConvEval(lrnde_ctx* c, const lrnde_model* mm, const float* p, int64_t b, bool vjp)
      : ctx(c), m(mm), ps(p), B(b), with_vjp(vjp) {
    for (auto& Li : m->conv)
      if (Li.bn && Li.cout > LR_BN_MAXC && ctx->nranks > 1)
        lr_fail(LRNDE_EINVAL, "BatchNorm with %d channels on a multi-rank ctx (the statistics exchange holds %d)", Li.cout, LR_BN_MAXC);
    L = (int)m->conv.size();
    HW = (size_t)m->Wd * m->Ht;
    tc = tc_eligible(m) && tc_fits(m, b);
    if (tc) geo.set(m->Wd, m->Ht, (int)B);
    wg_tc = tc && vjp && convtc_wgrad_ok(geo) && !getenv("LRNDE_CONV_WG_SIMT");
    z.assign(L, nullptr); ab.assign(L, nullptr); stat.assign(L, nullptr); pack.assign(L, nullptr); packT.assign(L, nullptr);
    wimg.assign(L, nullptr); wimgT.assign(L, nullptr); tsum.assign(L, nullptr);
    for (int l = 0; l < L; ++l) {
      const ConvLayerInfo& Li = m->conv[l];
      maxC = std::max(maxC, std::max(Li.cin, Li.cout));
      nblk_max = std::max(nblk_max, conv_nblk(Li.cout) * Li.cout);
      if (tc) {
        nblk_max = std::max(nblk_max, geo.ngroups * 8 * std::max(Li.cout, Li.cin));
        wimg[l] = (uint8_t*)ctx->alloc(convtc_wimg_bytes(Li.cin, convtc_nout(Li.cout)));
        if (m->td) tsum[l] = (float*)ctx->alloc(4 * 64 * (size_t)convtc_nout(Li.cout));
        if (vjp) wimgT[l] = (uint8_t*)ctx->alloc(convtc_wimg_bytes(Li.cout, convtc_nout(Li.cin)));
      }
      const size_t nw = (size_t)9 * (Li.cin + m->td) * Li.cout;
      pack[l] = (float*)ctx->alloc(4 * nw);
      if (l < L - 1) z[l] = (float*)ctx->alloc(4 * HW * Li.cout * B);
      if (Li.bn) { ab[l] = (float*)ctx->alloc(8 * Li.cout); stat[l] = (float*)ctx->alloc(8 * Li.cout); }
      s_off.push_back(nstate);
      if (Li.bn) nstate += 2 * (int64_t)Li.cout;
      if (vjp) packT[l] = (float*)ctx->alloc(4 * (size_t)9 * Li.cin * Li.cout);
    }
    spart = (float2*)ctx->alloc(sizeof(float2) * (size_t)nblk_max);
    if (tc) {
      // the guard positions and the tail of the last tile group are read by the bulk copies and never written
      const size_t nf = geo.f_floats(maxC);
      Fhi = (float*)ctx->alloc(4 * nf); Flo = (float*)ctx->alloc(4 * nf);
      LR_CUDA(cudaMemsetAsync(Fhi, 0, 4 * nf, ctx->stream));
      LR_CUDA(cudaMemsetAsync(Flo, 0, 4 * nf, ctx->stream));
    }
    if (vjp) {
      int n_sm = 148;
      ybuf = (float*)ctx->alloc(4 * (size_t)m->D * B);
      lbuf = (float*)ctx->alloc(4 * (size_t)m->D * B);
      G[0] = (float*)ctx->alloc(4 * HW * maxC * B);
      G[1] = (float*)ctx->alloc(4 * HW * maxC * B);
      size_t maxpart = 0;
      for (int l = 0; l < L; ++l) {
        const ConvLayerInfo& Li = m->conv[l];
        const int cintot = Li.cin + m->td;
        // few output channels (65 => 8): delta takes the patch role and the input the 64-wide tile role
        const bool swapped = Li.cout <= 16 && cintot > Li.cout;
        const int pt = swapped ? Li.cout : cintot, qt = swapped ? cintot : Li.cout;
        const int chunks = (pt + 15) / 16, cic = (pt + chunks - 1) / chunks;
        const int nqb = (qt + 63) / 64;
        int S = std::max(1, std::min((int)B, (4 * n_sm) / (chunks * nqb)));
        const int img = (int)((B + S - 1) / S);
        S = (int)((B + img - 1) / img);
        wS.push_back(S); wImg.push_back(img); wCic.push_back(cic); wChunks.push_back(chunks); wSwap.push_back(swapped ? 1 : 0);
        maxpart = std::max(maxpart, (size_t)S * 9 * cintot * Li.cout);
        if (wg_tc) maxpart = std::max(maxpart, (size_t)convtc_wgrad_splits(geo) * 9 * cintot * Li.cout);
      }
      if (wg_tc) {
        PD = (float*)ctx->alloc(4 * HW * maxC * B);
        rowsum = (float*)ctx->alloc(4 * (size_t)3 * m->Ht * maxC * B);
      }
      part = (float*)ctx->alloc(4 * maxpart);
      bnS = std::max(1, std::min((int)B, 16));
      bnImg = (int)((B + bnS - 1) / bnS);
      bnS = (int)((B + bnImg - 1) / bnImg);
      bpart = (double2*)ctx->alloc(sizeof(double2) * (size_t)maxC * bnS);
      coef = (float*)ctx->alloc(8 * maxC);
      dgb = (float*)ctx->alloc(8 * maxC);
    }
  }
  ~ConvEval() {
    for (auto p : z) ctx->release(p);
    for (auto p : ab) ctx->release(p);
    for (auto p : stat) ctx->release(p);
    for (auto p : pack) ctx->release(p);
    for (auto p : packT) ctx->release(p);
    for (auto p : wimg) ctx->release(p);
    for (auto p : wimgT) ctx->release(p);
    for (auto p : tsum) ctx->release(p);
    ctx->release(Fhi); ctx->release(Flo);
    ctx->release(PD); ctx->release(rowsum);
    ctx->release(spart); ctx->release(ybuf); ctx->release(lbuf); ctx->release(G[0]); ctx->release(G[1]);
    ctx->release(part); ctx->release(bpart); ctx->release(coef); ctx->release(dgb);
  }

  // o->model_state (NULL: batch statistics, nothing tracked), staged through the call's `io`.  With `update` and
  // outside testmode the f evaluations move the running statistics (until bn_update is cleared) and io.finish()
  // returns st'.model.  Returns the device pointer in use.
  float* attach_state(const lrnde_opts* o, CallerBufs& io, bool update) {
    bn_state = nullptr; testmode = 0; bn_update = false;
    if (!o) return nullptr;
    if (o->model_testmode && !o->model_state && nstate > 0)
      lr_fail(LRNDE_EINVAL, "model_testmode needs model_state (the running statistics BatchNorm normalises with)");
    if (!o->model_state || nstate == 0) return nullptr;
    testmode = o->model_testmode ? 1 : 0;
    bn_update = update && !testmode;
    bn_state = bn_update ? io.inout(o->model_state, nstate) : const_cast<float*>(io.in(o->model_state, nstate));
    return bn_state;
  }

  void prepare() {
    for (int l = 0; l < L; ++l) {
      const ConvLayerInfo& Li = m->conv[l];
      const int cintot = Li.cin + m->td;
      conv_pack_kernel<<<lr_ew_blocks((size_t)9 * cintot * Li.cout), 256, 0, ctx->stream>>>(ps + Li.w_off, cintot, Li.cout, 0, 0, pack[l]);
      LR_COUNT(ctx);
      if (with_vjp) {
        conv_pack_kernel<<<lr_ew_blocks((size_t)9 * Li.cin * Li.cout), 256, 0, ctx->stream>>>(ps + Li.w_off, cintot, Li.cout, 1, Li.cin, packT[l]);
        LR_COUNT(ctx);
      }
      if (tc) {
        convtc_wpack(ctx, ps + Li.w_off, cintot, Li.cout, 0, 0, m->td, wimg[l], tsum[l]);
        if (with_vjp) convtc_wpack(ctx, ps + Li.w_off, cintot, Li.cout, 1, Li.cin, m->td, wimgT[l], nullptr);
      }
    }
    LR_CHECK_LAUNCH();
  }

  int stat_nblk(int cout) const { return tc ? convtc_stat_rows(geo, cout) : conv_nblk(cout); }
  // tensor-core convolution of (F): packed operand -> [W,H,Cout,B]
  void launch_tc(const uint8_t* img, int K, const float* ts, const LinComb* tdesc, float* Y, const LinComb* ydesc, float scale,
                 int cout, float2* sp, const int* done) {
    ConvTcP q;
    memset(&q, 0, sizeof(q));
    q.Fhi = Fhi; q.Flo = Flo; q.Wimg = img; q.K = K; q.tsum = ts; q.tdesc = tdesc; q.Y = Y; q.ydesc = ydesc;
    q.out_scale = scale; q.Cout = cout; q.stat_part = sp; q.done = done;
    convtc_conv(ctx, geo, q);
  }

  void launch(ConvP& q) {
    q.Wd = m->Wd; q.Ht = m->Ht; q.B = (int)B;
    const bool nar = narrow(q.Cout);
    dim3 g(conv_nblk(q.Cout), (q.Cout + (nar ? 8 : 64) - 1) / (nar ? 8 : 64));
    if (nar) conv3x3_kernel<8, 8, 4><<<g, 256, 0, ctx->stream>>>(q);
    else conv3x3_kernel<64, 16, 8><<<g, 256, 0, ctx->stream>>>(q);
    LR_COUNT(ctx);
  }

  // layers 0..upto-1 of the dynamics on lincomb(in); `side` / `side_desc`: keep the combined input
  void run_layers(const LinComb* in, const int* done, int upto, const LinComb* out, bool side_to_in_dst, float* side,
                  bool update_state) {
    const int ncalls = (update_state && first_call_twice) ? 2 : 1;
    if (update_state) first_call_twice = false;
    for (int l = 0; l < upto; ++l) {
      const ConvLayerInfo& Li = m->conv[l];
      if (tc) {
        static const bool fuse = !(getenv("LRNDE_CONV_FUSE") && getenv("LRNDE_CONV_FUSE")[0] == '0');
        // (the producers address the source with 32-bit pixel offsets)
        if (l > 0 && fuse && (Li.cin & 15) == 0 && (double)HW * Li.cin * (double)B < 4.0e9) {
          // the convolution forms its operand itself from the stored raw output of the previous layer (BatchNorm scale /
          // shift + activation + hi / lo split by producer warps): no pack launch, no (F) round trip through HBM
          ConvTcP q;
          memset(&q, 0, sizeof(q));
          q.srcZ = z[l - 1]; q.src_ab = m->conv[l - 1].bn ? ab[l - 1] : nullptr; q.src_act = m->conv[l - 1].act;
          q.Wimg = wimg[l]; q.K = Li.cin; q.tsum = m->td ? tsum[l] : nullptr; q.tdesc = m->td ? in : nullptr;
          q.Y = l == L - 1 ? nullptr : z[l]; q.ydesc = l == L - 1 ? (out ? out : in) : nullptr;
          q.out_scale = 1.0f; q.Cout = Li.cout; q.stat_part = (Li.bn && !testmode) ? spart : nullptr; q.done = done;
          convtc_conv(ctx, geo, q);
        } else {
        ConvTcPackP pk;
        memset(&pk, 0, sizeof(pk));
        if (l == 0) { pk.xdesc = in; pk.side_to_desc_dst = side_to_in_dst ? 1 : 0; pk.side = side; pk.in_act = ACT_IDENTITY; }
        else { pk.X = z[l - 1]; pk.in_ab = m->conv[l - 1].bn ? ab[l - 1] : nullptr; pk.in_act = m->conv[l - 1].act; }
        pk.Fhi = Fhi; pk.Flo = Flo; pk.C = Li.cin; pk.done = done;
        convtc_pack(ctx, geo, pk);
        launch_tc(wimg[l], Li.cin, m->td ? tsum[l] : nullptr, m->td ? in : nullptr, l == L - 1 ? nullptr : z[l],
                  l == L - 1 ? (out ? out : in) : nullptr, 1.0f, Li.cout, (Li.bn && !testmode) ? spart : nullptr, done);
        }
      } else {
      ConvP q;
      memset(&q, 0, sizeof(q));
      if (l == 0) {
        q.xdesc = in; q.side_desc = side_to_in_dst ? in : nullptr; q.side = side; q.in_act = ACT_IDENTITY;
      } else {
        q.X = z[l - 1]; q.in_ab = m->conv[l - 1].bn ? ab[l - 1] : nullptr; q.in_act = m->conv[l - 1].act;
      }
      q.td = m->td; q.tdesc = in; q.Wp = pack[l]; q.Cin = Li.cin; q.Cout = Li.cout; q.out_scale = 1.0f; q.done = done;
      if (l == L - 1) q.ydesc = out ? out : in; else q.Y = z[l];
      if (Li.bn && !testmode) q.stat_part = spart;
      launch(q);
      }
      if (Li.bn) {
        bn_finalize_kernel<<<Li.cout, 128, 0, ctx->stream>>>(spart, stat_nblk(Li.cout), Li.cout, (double)HW * (double)B,
                                                           ps + Li.g_off, 1e-5f, ab[l], stat[l],
                                                           bn_state ? bn_state + s_off[l] : nullptr, testmode,
                                                           (update_state && bn_update) ? ncalls : 0, done, ctx->bn_dist());
        LR_COUNT(ctx);
      }
    }
  }

  void forward(const LinComb* in, const int* done, const LinComb* out, bool side_to_in_dst) {
    run_layers(in, done, L, out, side_to_in_dst, nullptr, true);
    LR_CHECK_LAUNCH();
  }


  // the reverse pass with every contraction on the tensor cores: the pack kernel writes each activation and each
  // cotangent once as the (F) operand of the next convolution and as the plain hi / lo operand of the weight gradient
  void vjp_tc(const LinComb* y, const LinComb* lamd, float* out_a, const LinComb* out_desc, float a_scale,
              float* dps_ptr, const LinComb* dps_desc, size_t dps_off, float p_scale, float p_beta, const int* done) {
    cudaStream_t st = ctx->stream;
    // recompute z_0..z_{L-2} (the weight gradients read them, and y(t) = ybuf, through TMA and transform on the fly)
    if (L > 1) run_layers(y, done, L - 1, nullptr, false, ybuf, false);
    else {
      ConvTcPackP pk;
      memset(&pk, 0, sizeof(pk));
      pk.xdesc = y; pk.side = ybuf; pk.in_act = ACT_IDENTITY; pk.C = m->conv[0].cin; pk.done = done;
      convtc_pack(ctx, geo, pk);
    }
    {   // cotangent of the output
      ConvTcPackP pk;
      memset(&pk, 0, sizeof(pk));
      pk.xdesc = lamd; pk.in_act = ACT_IDENTITY; pk.Fhi = Fhi; pk.Flo = Flo; pk.Pv = PD;
      pk.rowsum = m->td ? rowsum : nullptr;
      pk.C = m->conv[L - 1].cout; pk.done = done;
      convtc_pack(ctx, geo, pk);
    }
    const int S = convtc_wgrad_splits(geo);
    int cur = 0;
    for (int l = L - 1; l >= 0; --l) {
      const ConvLayerInfo& Li = m->conv[l];
      const int cintot = Li.cin + m->td;
      const size_t nw = (size_t)9 * cintot * Li.cout;
      ConvTcWgP w;
      memset(&w, 0, sizeof(w));
      if (l == 0) { w.X = ybuf; w.x_act = ACT_IDENTITY; }
      else { w.X = z[l - 1]; w.x_ab = m->conv[l - 1].bn ? ab[l - 1] : nullptr; w.x_act = m->conv[l - 1].act; }
      w.Cx = Li.cin; w.D = PD; w.Cd = Li.cout; w.CinTot = cintot;
      w.part = part; w.block = nw; w.tdesc = m->td ? y : nullptr; w.Drowsum = rowsum; w.done = done;
      convtc_wgrad(ctx, geo, w);
      wgrad_reduce_kernel<<<lr_ew_blocks(nw), 256, 0, st>>>(part, S, nw, dps_ptr ? dps_ptr + Li.w_off : nullptr, dps_desc,
                                                           dps_off + (size_t)Li.w_off, p_scale, p_beta, done);
      LR_COUNT(ctx);
      if (l == 0) {
        launch_tc(wimgT[l], Li.cout, nullptr, nullptr, out_a, out_a ? nullptr : out_desc, a_scale, Li.cin, nullptr, done);
      } else {
        const ConvLayerInfo& Lp = m->conv[l - 1];
        {
          ConvTcP q;
          memset(&q, 0, sizeof(q));
          q.Fhi = Fhi; q.Flo = Flo; q.Wimg = wimgT[l]; q.K = Li.cout; q.Y = G[cur]; q.out_scale = 1.0f; q.Cout = Li.cin; q.done = done;
          if (Lp.bn) { q.stat_part = spart; q.bwd_z = z[l - 1]; q.bwd_ab = ab[l - 1]; q.bwd_stat = stat[l - 1]; q.bwd_act = Lp.act; }
          convtc_conv(ctx, geo, q);
        }
        ConvTcPackP pk;
        memset(&pk, 0, sizeof(pk));
        pk.Fhi = Fhi; pk.Flo = Flo; pk.Pv = PD; pk.C = Lp.cout; pk.done = done; pk.in_act = ACT_IDENTITY;
        pk.rowsum = m->td ? rowsum : nullptr;
        if (Lp.bn) {
          bn_bwd_finalize_tc_kernel<<<Lp.cout, 128, 0, st>>>(spart, convtc_stat_rows(geo, Lp.cout), Lp.cout, (double)HW * (double)B, coef, dgb, testmode,
                                                            done, ctx->bn_dist());
          LR_COUNT(ctx);
          wgrad_reduce_kernel<<<1, 256, 0, st>>>(dgb, 1, (size_t)2 * Lp.cout, dps_ptr ? dps_ptr + Lp.g_off : nullptr, dps_desc,
                                               dps_off + (size_t)Lp.g_off, p_scale, p_beta, done);
          LR_COUNT(ctx);
          pk.X = z[l - 1]; pk.bwd_g = G[cur]; pk.in_ab = ab[l - 1]; pk.bwd_stat = stat[l - 1]; pk.bwd_coef = coef; pk.bwd_act = Lp.act;
        } else if (Lp.act != ACT_IDENTITY) {
          pk.X = z[l - 1]; pk.bwd_g = G[cur]; pk.bwd_act = Lp.act;
        } else {
          pk.X = G[cur];
        }
        convtc_pack(ctx, geo, pk);
        cur ^= 1;
      }
    }
    LR_CHECK_LAUNCH();
  }

  void vjp(const LinComb* y, const LinComb* lamd, float* out_a, const LinComb* out_desc, float a_scale,
           float* dps_ptr, const LinComb* dps_desc, size_t dps_off, float p_scale, float p_beta, const int* done) {
    if (wg_tc) { vjp_tc(y, lamd, out_a, out_desc, a_scale, dps_ptr, dps_desc, dps_off, p_scale, p_beta, done); return; }
    cudaStream_t st = ctx->stream;
    const size_t DB = (size_t)m->D * B;
    if (L > 1) run_layers(y, done, L - 1, nullptr, false, ybuf, false);     // recompute; y(t) kept for dW_1
    else { lincomb_kernel<<<lr_ew_blocks(DB), 256, 0, st>>>(y, ybuf, DB, done); LR_COUNT(ctx); }
    lincomb_kernel<<<lr_ew_blocks(DB), 256, 0, st>>>(lamd, lbuf, DB, done);
    LR_COUNT(ctx);
    const float* delta = lbuf;
    int cur = 0;
    for (int l = L - 1; l >= 0; --l) {
      const ConvLayerInfo& Li = m->conv[l];
      const int cintot = Li.cin + m->td;
      const size_t nw = (size_t)9 * cintot * Li.cout;
      ConvWgP w;
      memset(&w, 0, sizeof(w));
      ConvWgOp ox, od;
      memset(&ox, 0, sizeof(ox)); memset(&od, 0, sizeof(od));
      if (l == 0) { ox.ptr = ybuf; ox.act = ACT_IDENTITY; }
      else { ox.ptr = z[l - 1]; ox.ab = m->conv[l - 1].bn ? ab[l - 1] : nullptr; ox.act = m->conv[l - 1].act; }
      ox.C = Li.cin; ox.td = m->td;
      od.ptr = delta; od.act = ACT_IDENTITY; od.C = Li.cout; od.td = 0;
      w.swapped = wSwap[l];
      w.P = w.swapped ? od : ox; w.Q = w.swapped ? ox : od;
      w.tdesc = y; w.Wd = m->Wd; w.Ht = m->Ht; w.B = (int)B; w.CinTot = cintot; w.Cout = Li.cout;
      w.pcc = wCic[l]; w.img_per_split = wImg[l]; w.part = part; w.block = nw; w.done = done;
      const int qt = w.Q.C + w.Q.td;
      conv3x3_wgrad_kernel<<<dim3(wChunks[l], wS[l], (qt + 63) / 64), 256, 0, st>>>(w);
      LR_COUNT(ctx);
      wgrad_reduce_kernel<<<lr_ew_blocks(nw), 256, 0, st>>>(part, wS[l], nw, dps_ptr ? dps_ptr + Li.w_off : nullptr, dps_desc,
                                                           dps_off + (size_t)Li.w_off, p_scale, p_beta, done);
      LR_COUNT(ctx);
      // data gradient: transposed convolution over the first cin channels (the time channel has no cotangent)
      ConvP q;
      memset(&q, 0, sizeof(q));
      q.X = delta; q.in_act = ACT_IDENTITY; q.td = 0; q.Wp = packT[l]; q.Cin = Li.cout; q.Cout = Li.cin; q.done = done;
      if (tc) {   // (F) image of the cotangent, then the data-gradient convolution on the tensor cores
        ConvTcPackP pk;
        memset(&pk, 0, sizeof(pk));
        pk.X = delta; pk.in_act = ACT_IDENTITY; pk.Fhi = Fhi; pk.Flo = Flo; pk.C = Li.cout; pk.done = done;
        convtc_pack(ctx, geo, pk);
      }
      if (l == 0) {
        q.out_scale = a_scale;
        if (out_a) q.Y = out_a; else q.ydesc = out_desc;
        if (tc) launch_tc(wimgT[l], Li.cout, nullptr, nullptr, q.Y, q.ydesc, a_scale, Li.cin, nullptr, done);
        else launch(q);
      } else {
        q.out_scale = 1.0f; q.Y = G[cur];
        if (tc) launch_tc(wimgT[l], Li.cout, nullptr, nullptr, G[cur], nullptr, 1.0f, Li.cin, nullptr, done);
        else launch(q);
        const ConvLayerInfo& Lp = m->conv[l - 1];
        const size_t n = HW * Lp.cout * B;
        if (Lp.bn) {
          bn_bwd_stats_kernel<<<dim3(Lp.cout, bnS), 256, 0, st>>>(G[cur], z[l - 1], ab[l - 1], stat[l - 1], Lp.act, Lp.cout, HW,
                                                                (int)B, bnImg, bpart, done);
          LR_COUNT(ctx);
          bn_bwd_finalize_kernel<<<(Lp.cout + 63) / 64, 64, 0, st>>>(bpart, bnS, Lp.cout, (double)HW * (double)B, coef, dgb, testmode, done, ctx->bn_dist());
          LR_COUNT(ctx);
          wgrad_reduce_kernel<<<1, 256, 0, st>>>(dgb, 1, (size_t)2 * Lp.cout, dps_ptr ? dps_ptr + Lp.g_off : nullptr, dps_desc,
                                               dps_off + (size_t)Lp.g_off, p_scale, p_beta, done);
          LR_COUNT(ctx);
          bn_bwd_apply_kernel<<<lr_ew_blocks(n), 256, 0, st>>>(G[cur], z[l - 1], ab[l - 1], stat[l - 1], coef, Lp.act, Lp.cout, HW, n, done);
          LR_COUNT(ctx);
        } else if (Lp.act != ACT_IDENTITY) {
          bn_bwd_apply_kernel<<<lr_ew_blocks(n), 256, 0, st>>>(G[cur], z[l - 1], nullptr, nullptr, nullptr, Lp.act, Lp.cout, HW, n, done);
          LR_COUNT(ctx);
        }
        delta = G[cur];
        cur ^= 1;
      }
    }
    LR_CHECK_LAUNCH();
  }
};

// ------------------------------------------------------------------------------------------
// Engine route of one call: which engines evaluate f, its pullback and the regulariser's reverse pass.  lr_ode_route
// decides it once per call and is the only reader of LRNDE_NO_FUSED, LRNDE_NO_SMEM, LRNDE_NO_LATENT_ADJ,
// LRNDE_FULL_TAPE and LRNDE_NO_HIDDEN_REG; a kept tape stores the route of its forward call and the pullback follows it.
// The shared-memory engine is sized for the reverse pass (small_smem_bytes(bwd = true)) even without a pullback, so a
// forward and its pullback agree on small and umma.  lean => latent_adj => fused => umma; umma excludes small.
// ------------------------------------------------------------------------------------------
struct OdeRoute {
  bool conv = false;        // conv dynamics: ConvEval, which keeps its own switches
  bool small = false;       // the shared-memory engine (lrnde_smem_mlp.cuh): the whole network in one launch
  bool umma = false;        // per-layer tcgen05 kernels, else FP32 SIMT
  bool fused = false;       // forward attempts on FusedEngine; an MlpEval built for pullbacks (vjp) does not use it
  bool latent_adj = false;  // the pullback runs on LatentAdjoint: the forward keeps its hidden tape
  bool lean = false;        // the forward does not store k_2..k_6 (saves and the pullback read the hidden tape)
  bool reg_hidden = false;  // the regulariser's reverse pass runs in hidden space (lrnde_regrev.cuh)
  bool fused_model = false; // FusedEngine accepts the model at this precision (whether or not the call runs it)
  int passes = 3;           // tf32 hi/lo products of the tensor-core engines: 1 = single-pass TF32
};

// Shared-memory engine: the padded network (twice, for the reverse pass) and the tile buffers must fit one SM.  Fills
// *net and returns the samples per tile, 0 when the network does not fit.
static int lr_small_tile(lrnde_ctx* ctx, const lrnde_model* m, int64_t B, SdeNet* net) {
  if ((int)m->layers.size() > SDE_MAXL) return 0;
  SdeNet& snet = *net;
  memset(&snet, 0, sizeof(snet));
  snet.nl = (int)m->layers.size(); snet.td = m->td; snet.D = m->D; snet.nparams = (int)m->nparams;
  int woff = 0, hoff = 0, md = m->D;
  for (int l = 0; l < snet.nl; ++l) {
    const LayerInfo& L = m->layers[l];
    snet.in[l] = L.in; snet.out[l] = L.out; snet.outp[l] = (L.out + 3) & ~3; snet.act[l] = L.act;
    snet.ps_w[l] = L.w_off; snet.ps_b[l] = L.b_off;
    snet.w_off[l] = woff; woff += (L.in + m->td + 1) * snet.outp[l];
    snet.hid_off[l] = hoff; hoff += snet.outp[l];
    md = std::max(md, std::max(L.in, snet.outp[l]));
  }
  snet.wfloats = woff; snet.hid_rows = hoff; snet.maxdim = md;
  int n_sm = 0;
  size_t smem_optin = 0;
  sde_device_limits(ctx->device, &n_sm, &smem_optin);
  int S = 32;
  while (S > 8 && ((B + S - 1) / S) < n_sm / 2) S >>= 1;
  for (;; S >>= 1) {
    if (small_smem_bytes(snet, m->D, S + 1, true) + 2048 <= smem_optin) return S;   // 2 KB of static shared memory
    if (S <= 4) return 0;
  }
}

// Hidden-space reverse pass of the regulariser step (lrnde_regrev.cuh): 2-layer TD-MLP with tanh,
// regularize_type = :error_estimate
static bool lr_reg_hidden_eligible(const lrnde_model* m, int reg_type) {
  FusedShape sh;
  if (reg_type != LRNDE_REGTYPE_ERROR || !lrf_shape(m, &sh)) return false;
  if (m->layers.size() != 2 || m->layers[0].act != ACT_TANH || m->layers[1].act != ACT_IDENTITY) return false;
  if (m->input_act != ACT_IDENTITY) return false;
  const LayerInfo &L1 = m->layers[0], &L2 = m->layers[1];
  // the layer blocks must be [weight | bias] back to back (ComponentArray order), D a multiple of 4 (16-byte rows)
  if (L1.b_off != L1.w_off + (int64_t)L1.out * (L1.in + m->td) || L2.b_off != L2.w_off + (int64_t)L2.out * (L2.in + m->td)) return false;
  return sh.D % 4 == 0 && sh.H % 4 == 0 && sh.Kaug + m->td + 1 <= 104;
}

// o == NULL: precision 0 (auto), no tape
static OdeRoute lr_ode_route(lrnde_ctx* ctx, const lrnde_model* m, const lrnde_opts* o, int64_t B) {
  OdeRoute r;
  if (!m->conv.empty()) { r.conv = true; return r; }
  const int prec = o ? o->precision : LRNDE_PREC_AUTO;
  const bool keep_tape = o && o->keep_tape;
  r.passes = (prec == LRNDE_PREC_TF32) ? 1 : 3;
  // LRNDE_PREC_SMEM asks for the shared-memory engine; LRNDE_PREC_AUTO picks it for batches the per-layer tcgen05
  // kernels cannot fill (their cost is per-CTA latency, ~25 us per layer launch)
  if (prec == LRNDE_PREC_SMEM || prec == LRNDE_PREC_AUTO) {
    const bool want = (prec == LRNDE_PREC_SMEM);
    if (want && (int)m->layers.size() > SDE_MAXL) lr_fail(LRNDE_EINVAL, "precision smem: at most %d layers", SDE_MAXL);
    SdeNet net;
    const bool fits = lr_small_tile(ctx, m, B, &net) > 0;
    if (want && !fits) lr_fail(LRNDE_EINVAL, "precision smem: the network does not fit shared memory");
    r.small = fits && (want || (B <= 4096 && !getenv("LRNDE_NO_SMEM")));
  }
  r.umma = prec != LRNDE_PREC_FP32_SIMT && !r.small;
  r.fused_model = prec != LRNDE_PREC_FP32_SIMT && FusedEngine::eligible(m);
  r.fused = r.fused_model && r.umma && !getenv("LRNDE_NO_FUSED");
  r.latent_adj = r.fused && keep_tape && LatentAdjoint::eligible(m) && !getenv("LRNDE_NO_LATENT_ADJ");
  r.lean = r.latent_adj && !getenv("LRNDE_FULL_TAPE");
  r.reg_hidden = r.fused && keep_tape && lr_reg_hidden_eligible(m, o->reg_type) && !getenv("LRNDE_NO_HIDDEN_REG");
  return r;
}

// ------------------------------------------------------------------------------------------
// MLP evaluator: f(u, ps, t) and its VJP as sequences of kernels reading device descriptors
// ------------------------------------------------------------------------------------------
struct MlpEval {
  lrnde_ctx* ctx;
  const lrnde_model* m;
  const float* ps;
  int64_t B;
  bool with_vjp;
  std::vector<float*> act;  // act[l]: [out_l x B]
  std::vector<float*> pre;  // pre[l]: [out_l x B] (vjp only)
  std::vector<float*> WT;   // [in_l x out_l] (vjp only)
  std::vector<float*> packW, packWT;  // tcgen05 path: tf32 hi/lo shared-memory images of the weights
  bool use_umma = false;
  bool use_cluster = true;
  int max_layers = 1 << 30;  // profiling probe: evaluate only the first layers
  int nacc_max = 8;
  bool use_lean = true;
  bool use_wide = true;
  // small-state engine (lrnde_smem_mlp.cuh): the whole network out of shared memory, one launch per evaluation
  bool use_small = false;
  SdeNet snet;
  int sS = 32, s_tiles = 1, s_grid = 1;
  float* s_gpart = nullptr;
  int passes = 3;
  float* ybuf = nullptr;
  float* delta[2] = {nullptr, nullptr};
  float* part = nullptr;
  std::unique_ptr<ConvEval> conv;  // conv dynamics: every call below is forwarded
  std::unique_ptr<FusedEngine> fe; // latent-space engine (lrnde_fused.h): forward attempts of 2-layer TD-MLPs
  float* packW1x = nullptr;        // images of W1[:, :D] alone: Z(x) = W1[:, :D] x
  float* mz_plain_out = nullptr;   // where prepare() leaves the plain copy of Mz = W1 W2a (kept in the tape for the pullback)
  std::vector<int> wS, wChunk;    // SIMT weight-gradient split
  std::vector<int> uS, uChunk;    // tcgen05 weight-gradient split (0 = layer not eligible)

  // vjp: the evaluator of a pullback, which never runs the fused forward (route.fused is ignored)
  MlpEval(lrnde_ctx* c, const lrnde_model* mm, const float* p, int64_t b, const OdeRoute& route, bool vjp)
      : ctx(c), m(mm), ps(p), B(b), with_vjp(vjp) {
    if (route.conv) {
      conv = std::make_unique<ConvEval>(c, mm, p, b, vjp);
      return;
    }
    const int L = (int)m->layers.size();
    use_umma = route.umma;
    if (route.small) setup_small();
    use_cluster = (getenv("LRNDE_NO_CLUSTER") == nullptr);
    if (const char* e = getenv("LRNDE_NACC")) nacc_max = std::max(1, std::min(8, atoi(e)));
    use_lean = (getenv("LRNDE_NO_LEAN") == nullptr);
    use_wide = (getenv("LRNDE_NO_WIDE") == nullptr);
    passes = route.passes;
    if (route.fused && !vjp) {
      fe = std::make_unique<FusedEngine>(ctx, m, ps, B, passes);
      packW1x = (float*)ctx->alloc(sizeof(float) * 2 * umma::kAChunkFloats * umma::kReplicas *
                                   (size_t)tiles_m(m->layers[0].out) * chunks_k(m->layers[0].in));
    }
    act.assign(L, nullptr);
    packW.assign(L, nullptr);
    packWT.assign(L, nullptr);
    for (int l = 0; l < L; ++l) {
      if (l < L - 1 || vjp) act[l] = (float*)ctx->alloc(sizeof(float) * m->layers[l].out * B);
      if (use_umma) {
        const LayerInfo& Li = m->layers[l];
        packW[l] = (float*)ctx->alloc(sizeof(float) * 2 * umma::kAChunkFloats * umma::kReplicas *
                                      (size_t)tiles_m(Li.out) * chunks_k(Li.in + m->td + 1));
        if (vjp)
          packWT[l] = (float*)ctx->alloc(sizeof(float) * 2 * umma::kAChunkFloats * umma::kReplicas *
                                         (size_t)tiles_m(Li.in) * chunks_k(Li.out));
      }
    }
    if (vjp) {
      pre.assign(L, nullptr);
      WT.assign(L, nullptr);
      size_t maxd = 0, maxpart = 0;
      for (int l = 0; l < L; ++l) {
        const LayerInfo& Li = m->layers[l];
        pre[l] = (float*)ctx->alloc(sizeof(float) * Li.out * B);
        WT[l] = (float*)ctx->alloc(sizeof(float) * (size_t)Li.in * Li.out);
        maxd = std::max(maxd, (size_t)std::max(Li.in, Li.out) * (size_t)B);
        int naug = Li.in + m->td + 1;
        int tiles = ((Li.out + DN_BM - 1) / DN_BM) * ((naug + DN_BN - 1) / DN_BN);
        int S = std::max(1, std::min(64, (2 * 148 + tiles - 1) / tiles));
        int chunk = (int)((B + S - 1) / S);
        chunk = std::max(16, ((chunk + 15) / 16) * 16);
        S = (int)((B + chunk - 1) / chunk);
        wS.push_back(S);
        wChunk.push_back(chunk);
        maxpart = std::max(maxpart, (size_t)S * Li.out * naug);
        // tensor-core version: the smaller operand must fit one 128-column accumulator
        int us = 0, uc = 0;
        if (use_umma && std::min(Li.out, naug) <= 128) {
          int n_mt = (std::max(Li.out, naug) + 127) / 128;
          us = std::max(1, std::min(64, (getenv("LRNDE_WG_2WAVES") ? 256 : 148) / n_mt));  // one CTA per SM (196 KB of shared memory): a single wave
          uc = (int)((B + us - 1) / us);
          uc = std::max(32, ((uc + 31) / 32) * 32);
          us = (int)((B + uc - 1) / uc);
          maxpart = std::max(maxpart, (size_t)us * Li.out * naug);
        }
        uS.push_back(us);
        uChunk.push_back(uc);
      }
      ybuf = (float*)ctx->alloc(sizeof(float) * (size_t)m->D * B);
      delta[0] = (float*)ctx->alloc(sizeof(float) * maxd);
      delta[1] = (float*)ctx->alloc(sizeof(float) * maxd);
      part = (float*)ctx->alloc(sizeof(float) * maxpart);
    }
  }
  static int tiles_m(int M) { return (M + 127) / 128; }
  static int chunks_k(int K) { return (K + umma::kChunkK - 1) / umma::kChunkK; }
  ~MlpEval() {
    for (auto p : packW) ctx->release(p);
    for (auto p : packWT) ctx->release(p);
    for (auto p : act) ctx->release(p);
    for (auto p : pre) ctx->release(p);
    for (auto p : WT) ctx->release(p);
    ctx->release(ybuf);
    ctx->release(delta[0]);
    ctx->release(delta[1]);
    ctx->release(part);
    ctx->release(s_gpart);
    ctx->release(packW1x);
  }

  // the shared-memory engine's network image, tile size and grid (the route chose it, so lr_small_tile fits)
  void setup_small() {
    int n_sm = 0;
    size_t smem_optin = 0;
    sde_device_limits(ctx->device, &n_sm, &smem_optin);
    const int S = lr_small_tile(ctx, m, B, &snet);
    use_small = true;
    sS = S;
    const int ntiles = (int)((B + S - 1) / S);
    s_tiles = (ntiles + 4 * n_sm - 1) / (4 * n_sm);
    s_grid = (ntiles + s_tiles - 1) / s_tiles;
    if (with_vjp) s_gpart = (float*)ctx->alloc(sizeof(float) * (size_t)s_grid * snet.wfloats);
    static bool attr_set = false;
    if (!attr_set) {
      LR_CUDA(cudaFuncSetAttribute(small_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_optin - 2048));
      LR_CUDA(cudaFuncSetAttribute(small_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_optin - 2048));
      attr_set = true;
    }
  }
  SmallP small_params(const LinComb* in, const int* done) const {
    SmallP q;
    memset(&q, 0, sizeof(q));
    q.n = snet; q.in_act = m->input_act; q.ps = ps; q.in = in; q.done = done;
    q.B = (int)B; q.D = m->D; q.S = sS; q.SP = sS + 1; q.tiles_per_cta = s_tiles;
    return q;
  }

  // once per call: transposed weights for the data-gradient GEMMs, and (tcgen05 path) the
  // tf32 hi/lo shared-memory images of every weight matrix
  void prepare() {
    if (conv) { conv->prepare(); return; }
    if (use_small) return;
    if (fe) {
      fe->prepare(mz_plain_out);
      const LayerInfo& L1 = m->layers[0];
      umma::pack_weights_kernel<<<dim3(tiles_m(L1.out) * chunks_k(L1.in), umma::kReplicas), 256, 0, ctx->stream>>>(
          ps + L1.w_off, L1.out, L1.out, L1.in, chunks_k(L1.in), packW1x, passes);
      LR_COUNT(ctx);
    }
    for (size_t l = 0; l < m->layers.size(); ++l) {
      const LayerInfo& Li = m->layers[l];
      if (with_vjp) {
        dim3 g((Li.out + 31) / 32, (Li.in + 31) / 32), b(32, 8);
        transpose_kernel<<<g, b, 0, ctx->stream>>>(ps + Li.w_off, Li.out, Li.in, WT[l]);
        LR_COUNT(ctx);
      }
      if (use_umma) {
        const int kaug = Li.in + m->td + 1;
        umma::pack_weights_kernel<<<dim3(tiles_m(Li.out) * chunks_k(kaug), umma::kReplicas), 256, 0, ctx->stream>>>(
            ps + Li.w_off, Li.out, Li.out, kaug, chunks_k(kaug), packW[l], passes);
        LR_COUNT(ctx);
        if (with_vjp) {
          umma::pack_weights_kernel<<<dim3(tiles_m(Li.in) * chunks_k(Li.out), umma::kReplicas), 256, 0, ctx->stream>>>(
              WT[l], Li.in, Li.in, Li.out, chunks_k(Li.out), packWT[l], passes);
          LR_COUNT(ctx);
        }
      }
    }
    LR_CHECK_LAUNCH();
  }

  // pack == nullptr: FP32 SIMT kernel; else the tcgen05 kernel on the packed weight images
  void dense(const DenseP& p, const float* pack = nullptr) {
    if (!pack) {
      dim3 g((p.M + DN_BM - 1) / DN_BM, (p.N + DN_BN - 1) / DN_BN);
      dense_nn_kernel<<<g, 256, 0, ctx->stream>>>(p);
      LR_COUNT(ctx);
      return;
    }
    constexpr int NT = 64;
    constexpr int CL = 4;
    using C = umma::Cfg<NT>;
    static bool attr_set = false;
    if (!attr_set) {
      LR_CUDA(cudaFuncSetAttribute(umma::dense_kernel<NT, false, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::ring_smem()));
      LR_CUDA(cudaFuncSetAttribute(umma::dense_kernel<NT, true, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::res_smem(C::kMaxResKC)));
      LR_CUDA(cudaFuncSetAttribute(umma::dense_kernel<NT, false, CL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::ring_smem()));
      LR_CUDA(cudaFuncSetAttribute(umma::dense_kernel<NT, true, CL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::res_smem(C::kMaxResKC)));
      LR_CUDA(cudaFuncSetAttribute(umma::dense_kernel<NT, false, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::ring_smem()));
      LR_CUDA(cudaFuncSetAttribute(umma::dense_kernel<NT, true, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::res_smem(C::kMaxResKC)));
      LR_CUDA(cudaFuncSetAttribute(umma::dense_kernel<NT, false, CL, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::ring_smem()));
      LR_CUDA(cudaFuncSetAttribute(umma::dense_kernel<NT, true, CL, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::res_smem(C::kMaxResKC)));
      using CW = umma::Cfg<128>;
      LR_CUDA(cudaFuncSetAttribute(umma::dense_kernel<128, true, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, CW::res_smem(CW::kMaxResKC)));
      LR_CUDA(cudaFuncSetAttribute(umma::dense_kernel<128, true, CL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, CW::res_smem(CW::kMaxResKC)));
      LR_CUDA(cudaFuncSetAttribute(umma::dense_kernel<128, true, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, CW::res_smem(CW::kMaxResKC)));
      LR_CUDA(cudaFuncSetAttribute(umma::dense_kernel<128, true, CL, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, CW::res_smem(CW::kMaxResKC)));
      attr_set = true;
    }
    umma::UmmaP q;
    q.d = p;
    q.Apack = pack;
    q.n_mt = tiles_m(p.M);
    q.KC = chunks_k(p.K + p.td + p.bias);
    q.passes = passes;
    q.replicas = umma::kReplicas;
    q.nacc_max = nacc_max;
    q.res_group = q.n_mt;
    unsigned ntile = (unsigned)((p.N + NT - 1) / NT);
    const bool resident = q.n_mt > 1 && q.n_mt * NT <= 512 && q.KC <= C::kMaxResKC;
    // wide RESIDENT schedule: 128 samples per CTA (N = 128 per MMA runs at the tensor floor, N = 64 is
    // shared-memory bound), the weight tiles split into groups of 4 (512 TMEM columns) over grid.y
    const unsigned ntile_w = (unsigned)((p.N + 127) / 128);
    const unsigned ngroup_w = (unsigned)((q.n_mt + 3) / 4);
    const bool wide = use_wide && q.n_mt > 1 && q.KC <= umma::Cfg<128>::kMaxResKC && ntile_w * ngroup_w >= 96;
    if (wide) { ntile = ntile_w; q.res_group = 4; }
    const bool cluster = ntile >= (unsigned)CL && use_cluster;
    if (cluster) ntile = ((ntile + CL - 1) / CL) * CL;  // padded CTAs produce zeros and store nothing
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = wide ? dim3(ntile, ngroup_w) : (resident ? dim3(ntile) : dim3(ntile, q.n_mt));
    cfg.blockDim = dim3(umma::kThreads);
    cfg.dynamicSmemBytes = wide ? umma::Cfg<128>::res_smem(q.KC) : (resident ? C::res_smem(q.KC) : C::ring_smem());
    cfg.stream = ctx->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cluster ? CL : 1;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    // lean instantiation (no scalar fallback / activation switch in the hot loops) when the shape allows:
    // K % 4 == 0, rows 16-byte aligned (library buffers are 256-byte aligned and D*B % 4 == 0 follows from
    // ldx % 4 == 0), no input activation, tanh / identity epilogues
    const bool lean = use_lean && (p.K % 4 == 0) && (p.ldx % 4 == 0) && p.in_act == ACT_IDENTITY &&
                      (p.act == ACT_IDENTITY || p.act == ACT_TANH) &&
                      (p.dact < 0 || p.dact == ACT_IDENTITY || p.dact == ACT_TANH) &&
                      (!p.X || (((uintptr_t)p.X) & 15) == 0) && (!p.side || (((uintptr_t)p.side) & 15) == 0);
#define LR_LAUNCH_DENSE(RES, CLV, GENV) LR_CUDA(cudaLaunchKernelEx(&cfg, umma::dense_kernel<NT, RES, CLV, GENV>, q))
#define LR_LAUNCH_WIDE(CLV, GENV) LR_CUDA(cudaLaunchKernelEx(&cfg, umma::dense_kernel<128, true, CLV, GENV>, q))
    if (wide) {
      if (cluster) { if (lean) LR_LAUNCH_WIDE(CL, false); else LR_LAUNCH_WIDE(CL, true); }
      else { if (lean) LR_LAUNCH_WIDE(1, false); else LR_LAUNCH_WIDE(1, true); }
    } else if (resident) {
      if (cluster) { if (lean) LR_LAUNCH_DENSE(true, CL, false); else LR_LAUNCH_DENSE(true, CL, true); }
      else { if (lean) LR_LAUNCH_DENSE(true, 1, false); else LR_LAUNCH_DENSE(true, 1, true); }
    } else {
      if (cluster) { if (lean) LR_LAUNCH_DENSE(false, CL, false); else LR_LAUNCH_DENSE(false, CL, true); }
      else { if (lean) LR_LAUNCH_DENSE(false, 1, false); else LR_LAUNCH_DENSE(false, 1, true); }
    }
#undef LR_LAUNCH_DENSE
#undef LR_LAUNCH_WIDE
    LR_COUNT(ctx);
  }

  // z[B][LR_ZROW] <- W1[:, :D] u   (the latent image of a state array, lrnde_fused.h)
  void latent_of(const float* u, float* z) {
    const LayerInfo& L1 = m->layers[0];
    DenseP p;
    memset(&p, 0, sizeof(p));
    p.A = ps + L1.w_off; p.lda = L1.out; p.M = L1.out; p.K = L1.in; p.td = 0; p.bias = 0;
    p.X = u; p.ldx = L1.in; p.N = (int)B;
    p.Y = z; p.ldy = LR_ZROW; p.act = ACT_IDENTITY; p.dact = -1; p.out_scale = 1.0f;
    dense(p, packW1x);
    LR_CHECK_LAUNCH();
  }

  DenseP layer_fwd(int l, const LinComb* in, const float* xplain) const {
    const LayerInfo& Li = m->layers[l];
    DenseP p;
    memset(&p, 0, sizeof(p));
    p.A = ps + Li.w_off; p.lda = Li.out; p.M = Li.out; p.K = Li.in; p.td = m->td; p.bias = 1;
    if (l == 0) {
      if (xplain) p.X = xplain; else p.xdesc = in;
      p.in_act = m->input_act;
    } else p.X = act[l - 1];
    p.ldx = Li.in; p.N = (int)B;
    p.ldy = Li.out; p.ldpre = Li.out;
    p.act = Li.act; p.dact = -1; p.out_scale = 1.0f; p.tdesc = in;
    return p;
  }

  // (out ? out : in)->dst <- f(lincomb(in), ps, in->t); when side_to_in_dst the combined input
  // itself is also written to in->dst (u_{n+1} of the step, fused into stage 7's prologue)
  void forward(const LinComb* in, const int* done, const LinComb* out = nullptr,
               bool side_to_in_dst = false) {
    if (conv) { conv->forward(in, done, out, side_to_in_dst); return; }
    if (use_small) {
      SmallP q = small_params(in, done);
      q.out = out; q.side_to_in_dst = side_to_in_dst ? 1 : 0;
      small_kernel<false><<<s_grid, SDE_THREADS, small_smem_bytes(snet, m->D, sS + 1, false), ctx->stream>>>(q);
      LR_COUNT(ctx);
      LR_CHECK_LAUNCH();
      return;
    }
    const int L = (int)m->layers.size();
    for (int l = 0; l < std::min(L, max_layers); ++l) {
      DenseP p = layer_fwd(l, in, nullptr);
      if (l == L - 1) { p.ydesc = out ? out : in; p.y_off = 0; } else p.Y = act[l];
      if (l == 0 && side_to_in_dst) p.side_desc = in;
      p.done = done;
      dense(p, use_umma ? packW[l] : nullptr);
    }
    LR_CHECK_LAUNCH();
  }

  // data-gradient GEMM of layer l: g_{l-1} = W_l[:, :in]^T delta_l (times act'_{l-1}, or the final
  // scaled output when l == 0)
  DenseP data_gemm(int l, int cur, float* out_a, const LinComb* out_desc, float a_scale, const int* done) const {
    const LayerInfo& Li = m->layers[l];
    DenseP p;
    memset(&p, 0, sizeof(p));
    p.A = WT[l]; p.lda = Li.in; p.M = Li.in; p.K = Li.out; p.td = 0; p.bias = 0;
    p.X = delta[cur]; p.ldx = Li.out; p.N = (int)B;
    p.ldy = Li.in; p.act = ACT_IDENTITY; p.dact = -1; p.out_scale = 1.0f; p.done = done;
    if (l > 0) {
      p.Y = delta[cur ^ 1];
      if (m->layers[l - 1].act != ACT_IDENTITY) {
        p.dact = m->layers[l - 1].act; p.dpre = pre[l - 1]; p.lddpre = Li.in;
      }
    } else {
      if (out_a) p.Y = out_a; else { p.ydesc = out_desc; p.y_off = 0; }
      if (m->input_act != ACT_IDENTITY) { p.dact = m->input_act; p.dpre = ybuf; p.lddpre = Li.in; }
      p.out_scale = a_scale;
    }
    return p;
  }

  // (a, dps) = (J_u^T lam, J_p^T lam) of f at (lincomb(y), y->t), lam = lincomb(lamd) over D*B.
  //   a   -> a_scale * a   written to out_a, or to out_desc->dst
  //   dps -> dst = p_beta * dst + p_scale * dps with dst = dps_ptr or dps_desc->dst + dps_off
  void vjp(const LinComb* y, const LinComb* lamd, float* out_a, const LinComb* out_desc,
           float a_scale, float* dps_ptr, const LinComb* dps_desc, size_t dps_off, float p_scale,
           float p_beta, const int* done) {
    if (conv) { conv->vjp(y, lamd, out_a, out_desc, a_scale, dps_ptr, dps_desc, dps_off, p_scale, p_beta, done); return; }
    if (use_small) {
      SmallP q = small_params(y, done);
      q.lam = lamd; q.out_a = out_a; q.out_desc = out_desc; q.a_scale = a_scale; q.gpart = s_gpart;
      small_kernel<true><<<s_grid, SDE_THREADS, small_smem_bytes(snet, m->D, sS + 1, true), ctx->stream>>>(q);
      LR_COUNT(ctx);
      small_dps_reduce_kernel<<<(snet.wfloats + 255) / 256, 256, 0, ctx->stream>>>(snet, s_gpart, s_grid, dps_ptr, dps_desc, dps_off, p_scale,
                                                          p_beta, done);
      LR_COUNT(ctx);
      LR_CHECK_LAUNCH();
      return;
    }
    const int L = (int)m->layers.size();
    const size_t DB = (size_t)m->D * B;
    cudaStream_t st = ctx->stream;
    const bool last_identity = (m->layers[L - 1].act == ACT_IDENTITY);
    const bool fwd_runs = !(L == 1 && last_identity);
    if (!fwd_runs) {  // nothing will form y(t) in a prologue: materialise it
      lincomb_kernel<<<lr_ew_blocks(DB), 256, 0, st>>>(y, ybuf, DB, done);
      LR_COUNT(ctx);
    }
    for (int l = 0; l < L; ++l) {
      if (l == L - 1 && last_identity) break;  // output itself is not needed
      DenseP p = layer_fwd(l, y, nullptr);
      if (l == 0) p.side = ybuf;               // y(t) formed in the prologue, kept for dW_1 and act'
      p.Y = act[l];
      p.pre = pre[l];
      p.done = done;
      dense(p, use_umma ? packW[l] : nullptr);
    }
    if (!last_identity) {
      dact_mul_kernel<<<lr_ew_blocks(DB), 256, 0, st>>>(lamd, pre[L - 1], m->layers[L - 1].act, delta[0], DB,
                                                         done);
      LR_COUNT(ctx);
    }
    int cur = 0;
    for (int l = L - 1; l >= 0; --l) {
      const LayerInfo& Li = m->layers[l];
      const int naug = Li.in + m->td + 1;
      // identity output layer: delta_L is the lincomb lambda_g itself; the data-gradient GEMM
      // of that layer forms it in its prologue and keeps a copy (delta[0]) for dW_L
      const bool lam_in_prologue = (l == L - 1) && last_identity;
      if (lam_in_prologue) {
        DenseP p = data_gemm(l, cur, out_a, out_desc, a_scale, done);
        p.X = nullptr; p.xdesc = lamd; p.side = delta[0];
        dense(p, use_umma ? packWT[l] : nullptr);
      }
      const size_t nw = (size_t)Li.out * naug;
      const float* xin = (l == 0) ? ybuf : act[l - 1];
      const int xact = (l == 0) ? m->input_act : 0;
      int nsplit;
      if (uS[l] > 0) {
        // dW_aug = delta [x;t;1]^T on the tensor cores (MN-major operands, 3xTF32)
        static bool attr_set = false;
        if (!attr_set) {
          LR_CUDA(cudaFuncSetAttribute(umma::wgrad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       umma::wgrad_smem()));
          LR_CUDA(cudaFuncSetAttribute(umma::wgrad_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       umma::wgrad_smem()));
          attr_set = true;
        }
        umma::WgradUP w;
        memset(&w, 0, sizeof(w));
        umma::WgOperand od = {delta[cur], Li.out, Li.out, 0, 0, 0};
        umma::WgOperand ox = {xin, Li.in, Li.in, m->td, 1, xact};
        const bool normal = Li.out >= naug;
        w.P = normal ? od : ox;
        w.Q = normal ? ox : od;
        w.transposed = normal ? 0 : 1;
        w.ldo = Li.out;
        w.B = (int)B; w.chunk = uChunk[l]; w.part = part; w.block = nw; w.passes = passes;
        w.tdesc = y; w.done = done;
        dim3 g((std::max(Li.out, naug) + 127) / 128, uS[l]);
        const bool wlean = use_lean && w.P.rows % 4 == 0 && w.Q.rows % 4 == 0 && w.P.ld % 4 == 0 && w.Q.ld % 4 == 0 &&
                           w.P.in_act == ACT_IDENTITY && w.Q.in_act == ACT_IDENTITY &&
                           (((uintptr_t)w.P.ptr) & 15) == 0 && (((uintptr_t)w.Q.ptr) & 15) == 0;
        if (wlean) umma::wgrad_kernel<false><<<g, umma::kThreads, umma::wgrad_smem(), st>>>(w);
        else umma::wgrad_kernel<true><<<g, umma::kThreads, umma::wgrad_smem(), st>>>(w);
        nsplit = uS[l];
      } else {
        WgradP w;
        memset(&w, 0, sizeof(w));
        w.Dl = delta[cur]; w.ldd = Li.out; w.M = Li.out;
        w.X = xin; w.ldx = Li.in; w.Nin = Li.in; w.td = m->td; w.bias = 1;
        w.in_act = xact;
        w.B = (int)B; w.chunk = wChunk[l]; w.part = part; w.tdesc = y; w.done = done;
        dim3 g((Li.out + DN_BM - 1) / DN_BM, (naug + DN_BN - 1) / DN_BN, wS[l]);
        wgrad_nt_kernel<<<g, 256, 0, st>>>(w);
        nsplit = wS[l];
      }
      LR_COUNT(ctx);
      wgrad_reduce_kernel<<<lr_ew_blocks(nw), 256, 0, st>>>(
          part, nsplit, nw, dps_ptr ? dps_ptr + Li.w_off : nullptr, dps_desc,
          dps_off + (size_t)Li.w_off, p_scale, p_beta, done);
      LR_COUNT(ctx);
      if (!lam_in_prologue) {
        DenseP p = data_gemm(l, cur, out_a, out_desc, a_scale, done);
        dense(p, use_umma ? packWT[l] : nullptr);
      }
      cur ^= 1;
    }
    LR_CHECK_LAUNCH();
  }
};

// ------------------------------------------------------------------------------------------
// Solver: one adaptive Tsit5 integration whose state lives on the device
// ------------------------------------------------------------------------------------------
struct Solver {
  lrnde_ctx* ctx;
  SolveDev h;            // host image used to initialise / read back
  SolveDev* dev = nullptr;
  float* tape = nullptr;
  float* ts = nullptr;
  float* logbuf = nullptr;
  unsigned char* logacc = nullptr;
  double* partials = nullptr;
  unsigned int* counters = nullptr;
  float* muglob = nullptr;
  float* ztape = nullptr;
  float* htape = nullptr;
  cudaGraph_t while_graph = nullptr, body_graph = nullptr;
  cudaGraphExec_t while_exec = nullptr, body_exec = nullptr;
  long body_nodes = 0;
  bool graph_cached = false;   // while_graph / while_exec belong to ctx->graph_cache
  std::function<void()> body;

  Solver(lrnde_ctx* c, size_t len, size_t lam_len, int cap, int ring, int logcap) : ctx(c) {
    memset(&h, 0, sizeof(h));
    h.len = len;
    h.lam_len = lam_len;
    h.cap = cap;
    h.ring = ring;
    h.logcap = logcap;
    dev = (SolveDev*)ctx->alloc(sizeof(SolveDev));
    tape = (float*)ctx->alloc(sizeof(float) * 7 * len * (size_t)cap);
    if (!ring) ts = (float*)ctx->alloc(sizeof(float) * ((size_t)cap + 1));
    logbuf = (float*)ctx->alloc(sizeof(float) * 3 * (size_t)std::max(logcap, 1));
    logacc = (unsigned char*)ctx->alloc((size_t)std::max(logcap, 1));
    partials = (double*)ctx->alloc(sizeof(double) * 4 * LR_ERR_BLOCKS);
    counters = (unsigned int*)ctx->alloc(sizeof(unsigned int) * 8);
    h.tape = tape;
    h.ts = ts;
    h.log_t = logbuf;
    h.log_dt = logbuf + std::max(logcap, 1);
    h.log_eest = logbuf + 2 * (size_t)std::max(logcap, 1);
    h.log_acc = logacc;
    h.partials = partials;
    h.counters = counters;
    h.rank = ctx->rank;
    h.nranks = ctx->nranks;
    h.total_len = len;
    for (int r = 0; r < LR_MAX_RANKS; ++r) h.mbox[r] = ctx->peer_mbox[r];
  }
  ~Solver() {
    if (while_exec && !graph_cached) cudaGraphExecDestroy(while_exec);
    if (body_exec) cudaGraphExecDestroy(body_exec);
    if (while_graph && !graph_cached) cudaGraphDestroy(while_graph);
    if (body_graph) cudaGraphDestroy(body_graph);
    ctx->release(dev);
    ctx->release(tape);
    ctx->release(ts);
    ctx->release(logbuf);
    ctx->release(logacc);
    ctx->release(partials);
    ctx->release(counters);
    ctx->release(muglob);
    ctx->release(ztape);
    ctx->release(htape);
  }

  // latent tape of the fused engine: one [B][LR_ZROW] image per tape array (+ the hidden tape when the adjoint follows)
  void enable_latent(size_t zlen, bool hidden = false) {
    ztape = (float*)ctx->alloc(sizeof(float) * 7 * zlen * (size_t)h.cap);
    h.ztape = ztape;
    h.zlen = zlen;
    if (hidden) {
      htape = (float*)ctx->alloc(sizeof(float) * 7 * zlen * (size_t)h.cap);
      h.htape = htape;
    }
  }

  // adjoint in a data-parallel group: buffers of the mu-vector exchange
  void enable_mu_exchange(size_t P) {
    if (P > (size_t)LR_MU_MAX) {
      lr_set_error("data-parallel adjoint supports up to %d parameters, model has %zu", LR_MU_MAX, P);
      throw LrError(LRNDE_EINVAL);
    }
    muglob = (float*)ctx->alloc(sizeof(float) * 3 * P);
    h.muglob = muglob;
    h.mu_len = P;
    h.mucounter = counters + 4;
    h.reduce_mu = 1;
  }
  void upload() {
    h.seq = ctx->seq;
    h.mseq = ctx->mseq;
    LR_CUDA(cudaMemsetAsync(counters, 0, sizeof(unsigned int) * 8, ctx->stream));
    LR_CUDA(cudaMemcpyAsync(dev, &h, sizeof(SolveDev), cudaMemcpyHostToDevice, ctx->stream));
  }
  void download() {
    SolveDev* pin = (SolveDev*)ctx->pinned;
    LR_CUDA(cudaMemcpyAsync(pin, dev, sizeof(SolveDev), cudaMemcpyDeviceToHost, ctx->stream));
    LR_CUDA(cudaStreamSynchronize(ctx->stream));
    h = *pin;
    ctx->seq = h.seq;
    ctx->mseq = h.mseq;
  }

  void init_ctrl(float t0, float tend, float first_stop, int maxiters, int pow_mode,
                 float abstol, float reltol) {
    float dtmin = std::max(lr_spacing(t0), lr_spacing(tend));
    lr_ctrl_init(h.c, t0, tend, 0.0f, dtmin, maxiters, pow_mode);
    h.c.tstop = first_stop;
    h.abstol = abstol;
    h.reltol = reltol;
    h.slot = 0;
    h.done = 0;
    h.failed = 0;
    h.tape_full = 0;
  }

  // signature of the body: a throw-away capture, then every kernel node's function, launch shape and parameter bytes
  void body_signature(std::vector<lrnde_ctx::GraphNodeSig>& sig) {
    cudaStream_t st = ctx->stream;
    cudaGraph_t probe = nullptr;
    ctx->capturing = true;
    const long before = ctx->captured;
    cudaError_t e = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
    if (e != cudaSuccess) { ctx->capturing = false; LR_CUDA(e); }
    try { body(); } catch (...) {
      cudaGraph_t dummy; cudaStreamEndCapture(st, &dummy); ctx->capturing = false; ctx->captured = before; throw;
    }
    e = cudaStreamEndCapture(st, &probe);
    ctx->capturing = false;
    ctx->captured = before;
    LR_CUDA(e);
    size_t n = 0;
    LR_CUDA(cudaGraphGetNodes(probe, nullptr, &n));
    std::vector<cudaGraphNode_t> nodes(n);
    if (n) LR_CUDA(cudaGraphGetNodes(probe, nodes.data(), &n));
    sig.clear();
    bool ok = true;
    for (size_t i = 0; i < n && ok; ++i) {
      cudaGraphNodeType ty;
      LR_CUDA(cudaGraphNodeGetType(nodes[i], &ty));
      if (ty != cudaGraphNodeTypeKernel) { ok = false; break; }
      cudaKernelNodeParams kp;
      LR_CUDA(cudaGraphKernelNodeGetParams(nodes[i], &kp));
      lrnde_ctx::GraphNodeSig s;
      s.func = kp.func;
      s.g[0] = kp.gridDim.x; s.g[1] = kp.gridDim.y; s.g[2] = kp.gridDim.z;
      s.b[0] = kp.blockDim.x; s.b[1] = kp.blockDim.y; s.b[2] = kp.blockDim.z;
      s.smem = kp.sharedMemBytes;
      if (!kp.kernelParams) { ok = false; break; }
      for (size_t pi = 0;; ++pi) {
        size_t off = 0, sz = 0;
        if (cudaFuncGetParamInfo(kp.func, pi, &off, &sz) != cudaSuccess) { cudaGetLastError(); break; }
        const char* src = (const char*)kp.kernelParams[pi];
        s.params.insert(s.params.end(), src, src + sz);
      }
      sig.push_back(std::move(s));
    }
    cudaGraphDestroy(probe);
    if (!ok) sig.clear();   // something other than kernel nodes: no caching
  }

  // one step attempt = body(); captured once, then looped on the device
  void build_graphs(int loop_mode) {
    cudaStream_t st = ctx->stream;
    if (loop_mode == 0) {
      std::vector<lrnde_ctx::GraphNodeSig> sig;
      const bool use_cache = getenv("LRNDE_NO_GRAPH_CACHE") == nullptr;
      if (use_cache) {
        body_signature(sig);
        for (auto& cg : ctx->graph_cache) {
          if (cg.dev != (void*)dev || cg.sig.size() != sig.size()) continue;
          bool same = true;
          for (size_t i = 0; i < sig.size() && same; ++i) {
            const auto &a = cg.sig[i], &b = sig[i];
            same = a.func == b.func && memcmp(a.g, b.g, sizeof(a.g)) == 0 && memcmp(a.b, b.b, sizeof(a.b)) == 0 &&
                   a.smem == b.smem && a.params == b.params;
          }
          if (!same) continue;
          while_graph = cg.graph; while_exec = cg.exec; graph_cached = true;
          h.cond_handle = cg.handle; h.use_cond = 1; body_nodes = cg.body_nodes;
          cg.last_use = ++ctx->graph_clock;
          return;
        }
      }
      LR_CUDA(cudaGraphCreate(&while_graph, 0));
      cudaGraphConditionalHandle handle;
      LR_CUDA(cudaGraphConditionalHandleCreate(&handle, while_graph, 0, 0));
      h.cond_handle = (unsigned long long)handle;
      h.use_cond = 1;
      cudaGraphNode_t prime;
      cudaKernelNodeParams kp;
      memset(&kp, 0, sizeof(kp));
      SolveDev* d = dev;
      void* args[] = {&d};
      kp.func = (void*)cond_prime_kernel_entry();
      kp.gridDim = dim3(1);
      kp.blockDim = dim3(32);
      kp.kernelParams = args;
      LR_CUDA(cudaGraphAddKernelNode(&prime, while_graph, nullptr, 0, &kp));
      cudaGraphNodeParams cp = {cudaGraphNodeTypeConditional};
      cp.type = cudaGraphNodeTypeConditional;
      cp.conditional.handle = handle;
      cp.conditional.type = cudaGraphCondTypeWhile;
      cp.conditional.size = 1;
      cudaGraphNode_t cond;
      LR_CUDA(cudaGraphAddNode(&cond, while_graph, &prime, 1, &cp));
      cudaGraph_t bodyg = cp.conditional.phGraph_out[0];
      ctx->capturing = true;
      long before = ctx->captured;
      cudaError_t e = cudaStreamBeginCaptureToGraph(st, bodyg, nullptr, nullptr, 0,
                                                    cudaStreamCaptureModeThreadLocal);
      if (e != cudaSuccess) { ctx->capturing = false; LR_CUDA(e); }
      try { body(); } catch (...) {
        cudaGraph_t dummy; cudaStreamEndCapture(st, &dummy); ctx->capturing = false; throw;
      }
      cudaGraph_t outg = nullptr;
      e = cudaStreamEndCapture(st, &outg);
      ctx->capturing = false;
      LR_CUDA(e);
      body_nodes = ctx->captured - before;
      LR_CUDA(cudaGraphInstantiate(&while_exec, while_graph, 0));
      if (use_cache && !sig.empty()) {
        if (ctx->graph_cache.size() >= 8) {   // evict the least recently used entry (no live solver launches it again:
                                              // solvers only launch their graph inside the call that built it)
          size_t lru = 0;
          for (size_t i = 1; i < ctx->graph_cache.size(); ++i)
            if (ctx->graph_cache[i].last_use < ctx->graph_cache[lru].last_use) lru = i;
          cudaGraphExecDestroy(ctx->graph_cache[lru].exec);
          cudaGraphDestroy(ctx->graph_cache[lru].graph);
          ctx->graph_cache.erase(ctx->graph_cache.begin() + lru);
        }
        lrnde_ctx::CachedGraph cg;
        cg.graph = while_graph; cg.exec = while_exec; cg.handle = h.cond_handle; cg.body_nodes = body_nodes;
        cg.dev = (void*)dev; cg.sig = std::move(sig); cg.last_use = ++ctx->graph_clock;
        ctx->graph_cache.push_back(std::move(cg));
        graph_cached = true;
      }
    } else if (loop_mode == 2) {
      // no graph at all (profilers that cannot see into graphs): body() is launched directly
      h.use_cond = 0;
      long before = ctx->launches;
      (void)before;
      body_nodes = 0;
    } else {
      h.use_cond = 0;
      ctx->capturing = true;
      long before = ctx->captured;
      cudaError_t e = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
      if (e != cudaSuccess) { ctx->capturing = false; LR_CUDA(e); }
      try { body(); } catch (...) {
        cudaGraph_t dummy; cudaStreamEndCapture(st, &dummy); ctx->capturing = false; throw;
      }
      e = cudaStreamEndCapture(st, &body_graph);
      ctx->capturing = false;
      LR_CUDA(e);
      body_nodes = ctx->captured - before;
      LR_CUDA(cudaGraphInstantiate(&body_exec, body_graph, 0));
    }
  }
  static void* cond_prime_kernel_entry();

  // run attempts until the device says done.  WHILE mode: no host involvement at all.
  // Chunked mode (diagnostic): replay the body in groups of 8 and poll the flag.
  void run_segment() {
    cudaStream_t st = ctx->stream;
    if (while_exec) {
      LR_CUDA(cudaGraphLaunch(while_exec, st));
      ctx->launches += 1;
    } else {
      int* pin = (int*)((char*)ctx->pinned + sizeof(SolveDev) + 64);
      for (;;) {
        for (int i = 0; i < 8; ++i) {
          if (body_exec) LR_CUDA(cudaGraphLaunch(body_exec, st));
          else body();
        }
        LR_CUDA(cudaMemcpyAsync(pin, &dev->done, sizeof(int), cudaMemcpyDeviceToHost, st));
        LR_CUDA(cudaStreamSynchronize(st));
        if (*pin) break;
      }
    }
  }
};

__global__ void cond_prime_kernel(SolveDev* S) {
  if (threadIdx.x == 0) lr_set_cond(S);
}
void* Solver::cond_prime_kernel_entry() { return (void*)cond_prime_kernel; }

// ------------------------------------------------------------------------------------------
// tape: everything the pullback needs
// ------------------------------------------------------------------------------------------
struct lrnde_tape {
  lrnde_ctx* ctx;
  const lrnde_model* model;
  lrnde_opts opts;
  int64_t B;
  float* ps = nullptr;  // device copy of the parameters the forward used
  float* bn_state = nullptr;  // conv dynamics: device copy of st.model the forward normalised with (testmode)
  float* Mz = nullptr;        // latent-space engines: W1 W2a of the parameters the forward used ([128][128])
  OdeRoute route;             // the engines of the forward call; its pullback runs on the same ones
  std::unique_ptr<Solver> fwd;
  std::unique_ptr<Solver> reg;  // regulariser integrator (2-slot ring), reg modes only
  std::vector<float> fts;       // host copy of accepted times
  SavePlan saves;               // the saved solution of the forward call, t1
  int reg_mode = 0;
  // step logs (host copies)
  std::vector<float> log_t[2], log_dt[2], log_eest[2];
  std::vector<unsigned char> log_acc[2];
  ~lrnde_tape() { ctx->release(ps); ctx->release(bn_state); ctx->release(Mz); }
};

static void lr_copy_log(Solver& S, lrnde_tape* T, int which) {
  int n = std::min(S.h.nlog, S.h.logcap);
  T->log_t[which].resize(n);
  T->log_dt[which].resize(n);
  T->log_eest[which].resize(n);
  T->log_acc[which].resize(n);
  if (n == 0) return;
  cudaStream_t st = S.ctx->stream;
  LR_CUDA(cudaMemcpyAsync(T->log_t[which].data(), S.h.log_t, 4 * (size_t)n, cudaMemcpyDeviceToHost, st));
  LR_CUDA(cudaMemcpyAsync(T->log_dt[which].data(), S.h.log_dt, 4 * (size_t)n, cudaMemcpyDeviceToHost, st));
  LR_CUDA(cudaMemcpyAsync(T->log_eest[which].data(), S.h.log_eest, 4 * (size_t)n, cudaMemcpyDeviceToHost, st));
  LR_CUDA(cudaMemcpyAsync(T->log_acc[which].data(), S.h.log_acc, (size_t)n, cudaMemcpyDeviceToHost, st));
  LR_CUDA(cudaStreamSynchronize(st));
}

// data-parallel adjoint: exchange the mu vectors the next norm reads (no-op otherwise)
static void lr_mu_exchange(Solver& S, int mode, int nvec, const int* done) {
  if (!(S.h.reduce_mu && S.h.nranks > 1)) return;
  lrnde_ctx* ctx = S.ctx;
  cudaStream_t st = ctx->stream;
  mu_publish_kernel<<<64, 256, 0, st>>>(S.dev, mode, done);
  LR_COUNT(ctx);
  mu_gather_kernel<<<64, 256, 0, st>>>(S.dev, nvec, done);
  LR_COUNT(ctx);
  mu_norm_kernel<<<LR_ERR_BLOCKS, 256, 0, st>>>(S.dev, mode, done);
  LR_COUNT(ctx);
}

// fsalfirst + initial dt of a freshly initialised solver (OrdinaryDiffEq __init: initialize!
// then auto_dt_reset!), then the header of the first attempt when `begin`.
template <class EvalFn>
static void lr_solver_start(Solver& S, EvalFn&& eval, int begin) {
  lrnde_ctx* ctx = S.ctx;
  cudaStream_t st = ctx->stream;
  k1_desc_kernel<<<1, 32, 0, st>>>(S.dev);
  LR_COUNT(ctx);
  eval(&S.dev->st[6], &S.dev->yint[6], &S.dev->failed, nullptr, false);
  initdt_norm1_kernel<<<LR_ERR_BLOCKS, 256, 0, st>>>(S.dev);
  LR_COUNT(ctx);
  lr_mu_exchange(S, 0, 1, &S.dev->failed);
  initdt_a_kernel<<<1, 32, 0, st>>>(S.dev);
  LR_COUNT(ctx);
  eval(&S.dev->st[0], &S.dev->yint[1], &S.dev->failed, nullptr, false);
  initdt_norm2_kernel<<<LR_ERR_BLOCKS, 256, 0, st>>>(S.dev);
  LR_COUNT(ctx);
  lr_mu_exchange(S, 1, 1, &S.dev->failed);
  initdt_b_kernel<<<1, 32, 0, st>>>(S.dev, begin);
  LR_COUNT(ctx);
  LR_CHECK_LAUNCH();
}

// the kernels of one step attempt (perform_step! + loopfooter! + next loopheader!)
template <class EvalFn>
static void lr_step_body(Solver& S, EvalFn&& eval, bool fuse_unew = false) {
  lrnde_ctx* ctx = S.ctx;
  cudaStream_t st = ctx->stream;
  for (int j = 0; j < 5; ++j) eval(&S.dev->st[j], &S.dev->yint[j + 1], &S.dev->done, nullptr, false);
  if (fuse_unew) {
    // u_{n+1} = uprev + dt * sum a_7i k_i is formed in the prologue of stage 7's first GEMM and
    // stored from there (perform_step.jl:18-19 in one kernel)
    eval(&S.dev->st[5], &S.dev->yint[6], &S.dev->done, &S.dev->st[6], true);
  } else {
    lincomb_kernel<<<lr_ew_blocks(S.h.len), 256, 0, st>>>(&S.dev->st[5], nullptr, S.h.len, &S.dev->done);
    LR_COUNT(ctx);
    eval(&S.dev->st[6], &S.dev->yint[6], &S.dev->done, nullptr, false);
  }
  err_norm_kernel<<<LR_ERR_BLOCKS, 256, 0, st>>>(S.dev);
  LR_COUNT(ctx);
  lr_mu_exchange(S, 2, 3, &S.dev->done);
  controller_kernel<<<1, 32, 0, st>>>(S.dev);
  LR_COUNT(ctx);
  LR_CHECK_LAUNCH();
}

static void lr_grow_tape(Solver& S) {
  lrnde_ctx* ctx = S.ctx;
  cudaStream_t st = ctx->stream;
  int newcap = S.h.cap * 2;
  size_t slot_bytes = sizeof(float) * 7 * S.h.len;
  float* nt = (float*)ctx->alloc(slot_bytes * (size_t)newcap);
  float* nts = (float*)ctx->alloc(sizeof(float) * ((size_t)newcap + 1));
  LR_CUDA(cudaMemcpyAsync(nt, S.tape, slot_bytes * (size_t)(S.h.slot + 1), cudaMemcpyDeviceToDevice, st));
  LR_CUDA(cudaMemcpyAsync(nts, S.ts, sizeof(float) * (size_t)(S.h.slot + 1), cudaMemcpyDeviceToDevice, st));
  LR_CUDA(cudaStreamSynchronize(st));
  ctx->release(S.tape);
  ctx->release(S.ts);
  S.tape = nt;
  S.ts = nts;
  S.h.tape = nt;
  S.h.ts = nts;
  if (S.ztape) {
    float* nz = (float*)ctx->alloc(sizeof(float) * 7 * S.h.zlen * (size_t)newcap);
    LR_CUDA(cudaMemcpyAsync(nz, S.ztape, sizeof(float) * 7 * S.h.zlen * (size_t)(S.h.slot + 1), cudaMemcpyDeviceToDevice, st));
    LR_CUDA(cudaStreamSynchronize(st));
    ctx->release(S.ztape);
    S.ztape = nz;
    S.h.ztape = nz;
    LR_CUDA(cudaMemcpyAsync(&S.dev->ztape, &S.h.ztape, sizeof(float*), cudaMemcpyHostToDevice, st));
    if (S.htape) {
      float* nh = (float*)ctx->alloc(sizeof(float) * 7 * S.h.zlen * (size_t)newcap);
      LR_CUDA(cudaMemcpyAsync(nh, S.htape, sizeof(float) * 7 * S.h.zlen * (size_t)(S.h.slot + 1), cudaMemcpyDeviceToDevice, st));
      LR_CUDA(cudaStreamSynchronize(st));
      ctx->release(S.htape);
      S.htape = nh;
      S.h.htape = nh;
      LR_CUDA(cudaMemcpyAsync(&S.dev->htape, &S.h.htape, sizeof(float*), cudaMemcpyHostToDevice, st));
    }
  }
  S.h.cap = newcap;
  // patch the three fields in the device image
  LR_CUDA(cudaMemcpyAsync(&S.dev->tape, &S.h.tape, sizeof(float*), cudaMemcpyHostToDevice, st));
  LR_CUDA(cudaMemcpyAsync(&S.dev->ts, &S.h.ts, sizeof(float*), cudaMemcpyHostToDevice, st));
  LR_CUDA(cudaMemcpyAsync(&S.dev->cap, &S.h.cap, sizeof(int), cudaMemcpyHostToDevice, st));
}

static size_t lr_tape_budget(lrnde_ctx* ctx) {
  if (ctx->tape_budget) return (size_t)ctx->tape_budget;
  // cudaMemGetInfo takes a driver lock (measured 0.08 ... 60 ms per call on a shared host), so the
  // automatic budget is computed once per ctx; a failing allocation still falls back to
  // release_all_unused() + retry in lrnde_ctx::alloc
  if (ctx->auto_budget) return ctx->auto_budget;
  size_t fr = 0, tot = 0;
  LR_CUDA(cudaMemGetInfo(&fr, &tot));
  size_t pooled = 0;
  for (auto& b : ctx->pool)
    if (!b.used) pooled += b.bytes;
  ctx->auto_budget = (size_t)(0.6 * (double)(fr + pooled));
  return ctx->auto_budget;
}

// host-side evaluation of "sol(t)" on the dense forward tape: descriptor of the interpolant
// (or of the stored state on an exact hit), oracle ODESolution.__call__(exact_hit_stored=True)
static LinComb lr_host_interp(const Solver& F, const std::vector<float>& fts, float tval) {
  LinComb d;
  memset(&d, 0, sizeof(d));
  const int nsteps = (int)fts.size() - 1;
  for (int n = 0; n <= nsteps; ++n) {
    if (fts[n] == tval) {
      d.base = F.tape + (size_t)n * 7 * F.h.len;
      d.t = tval;
      return d;
    }
  }
  if (nsteps < 1) {
    d.base = F.tape;
    d.t = tval;
    return d;
  }
  int n = lr_locate(fts.data(), nsteps, 1, tval);
  float dt = lr_sub(fts[n + 1], fts[n]);
  float th = lr_div(lr_sub(tval, fts[n]), dt);
  float b[7];
  lr_tsit5_interp(th, b);
  const float* slot = F.tape + (size_t)n * 7 * F.h.len;
  d.base = slot;
  for (int k = 0; k < 6; ++k) d.src[k] = slot + (size_t)(k + 1) * F.h.len;
  d.src[6] = slot + (size_t)8 * F.h.len;
  for (int k = 0; k < 7; ++k) d.coef[k] = b[k];
  d.scale = dt;
  d.n = 7;
  d.t = tval;
  return d;
}

// y(t) of the forward solution into dst (device): the stored state on an exact hit, else the dense interpolant --
// from the D-dimensional tape, or (lean tape, lean_fe: an engine of the forward's model) from the hidden tape:
// y(t) = x + W2a c(t) (FusedEngine::dense_output)
static void lr_sol_at(lrnde_ctx* ctx, lrnde_tape* T, FusedEngine* lean_fe, float tq, float* dst, LinComb* host_desc,
                      const LinComb* dev_desc) {
  Solver& F = *T->fwd;
  cudaStream_t st = ctx->stream;
  const size_t DB = F.h.len;
  *host_desc = lr_host_interp(F, T->fts, tq);
  host_desc->dst = dst;
  LR_CUDA(cudaMemcpyAsync((void*)dev_desc, host_desc, sizeof(LinComb), cudaMemcpyHostToDevice, st));
  if (lean_fe && host_desc->n > 0) {
    const size_t n = (size_t)(host_desc->base - F.tape) / ((size_t)7 * DB);
    const size_t zl = F.h.zlen;
    const float* harr[8];
    for (int i = 0; i < 7; ++i) harr[i] = F.htape + (n * 7 + i) * zl;
    harr[7] = F.htape + ((n + 1) * 7 + 1) * zl;
    lean_fe->dense_output(F.dev, harr, host_desc->coef, host_desc->scale, F.tape, dev_desc);
  } else {
    lincomb_kernel<<<lr_ew_blocks(DB), 256, 0, st>>>(dev_desc, dst, DB, nullptr);
    LR_COUNT(ctx);
  }
}

static void lr_validate_opts(const lrnde_opts* o) {
  if (!o) lr_fail(LRNDE_EINVAL, "opts is NULL");
  if (o->reg_mode < LRNDE_REG_NONE || o->reg_mode > LRNDE_REG_BIASED)
    lr_fail(LRNDE_EINVAL, "regularize must be one of (:none, :unbiased, :biased)");
  if (o->reg_type != LRNDE_REGTYPE_ERROR && o->reg_type != LRNDE_REGTYPE_STIFFNESS)
    lr_fail(LRNDE_EINVAL, "regularize must be one of (:error_estimate, :stiffness_estimate)");
  if (!(o->t2 > o->t0)) lr_fail(LRNDE_EINVAL, "tspan must satisfy t0 < t2");
  if (o->maxiters < 1) lr_fail(LRNDE_EINVAL, "maxiters must be >= 1");
  if (o->nsave > 0 && !o->saveat) lr_fail(LRNDE_EINVAL, "saveat is NULL but nsave > 0");
  if (o->precision < LRNDE_PREC_AUTO || o->precision > LRNDE_PREC_SMEM)
    lr_fail(LRNDE_EINVAL, "unknown precision %d", o->precision);
}

// The returned blocks of the saved solution into u_save (may be NULL) and their times into save_times (host, may be
// NULL).  u_save is a HOST pointer when the forward call had host_buffers: then each block goes through one D*B
// device buffer, with a synchronisation before the next block reuses it, instead of CallerBufs, which would hold
// nout*D*B of device scratch for the whole call.
static void lr_write_saves(lrnde_ctx* ctx, lrnde_tape* T, FusedEngine* lean_fe, float* u_save, float* save_times) {
  const SavePlan& plan = T->saves;
  for (size_t i = 0; i < plan.times.size(); ++i)
    if (plan.out[i] >= 0 && save_times) save_times[plan.out[i]] = plan.times[i];
  if (!u_save || plan.nout == 0) return;
  cudaStream_t st = ctx->stream;
  const size_t DB = T->fwd->h.len;
  const bool per_block = T->opts.host_buffers != 0;
  DevBuf dd(ctx, (size_t)plan.nout * (sizeof(LinComb) / 4 + 1)), stage(ctx, per_block ? DB : 1);
  for (size_t i = 0; i < plan.times.size(); ++i) {
    const int blk = plan.out[i];
    if (blk < 0) continue;
    LinComb hd;
    float* dst = per_block ? stage.p : u_save + (size_t)blk * DB;
    lr_sol_at(ctx, T, lean_fe, std::min(plan.times[i], T->fts.back()), dst, &hd, (const LinComb*)dd.p + blk);
    if (per_block) {
      LR_CUDA(cudaMemcpyAsync(u_save + (size_t)blk * DB, dst, sizeof(float) * DB, cudaMemcpyDeviceToHost, st));
      LR_CUDA(cudaStreamSynchronize(st));   // stage is reused by the next block
    }
  }
  LR_CHECK_LAUNCH();
  LR_CUDA(cudaStreamSynchronize(st));
}

// ------------------------------------------------------------------------------------------
// f(u, ps, t) once (parity hook)
// ------------------------------------------------------------------------------------------
extern "C" int lrnde_dynamics_eval(lrnde_ctx* ctx, const lrnde_model* m, const lrnde_opts* o,
                                   const float* ps, const float* u, float t, int64_t B,
                                   float* du) {
  LR_API_BEGIN
  if (!ctx || !m || !ps || !u || !du || B < 1) lr_fail(LRNDE_EINVAL, "lrnde_dynamics_eval: bad args");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t DB = (size_t)m->D * B;
  CallerBufs io(ctx, o ? o->host_buffers : 0);
  const float* psd = io.in(ps, m->nparams);
  const float* ud = io.in(u, DB);
  float* outd = io.out(du, DB);
  DevBuf ddesc(ctx, sizeof(LinComb) / 4 + 1);
  LinComb d;
  memset(&d, 0, sizeof(d));
  d.base = ud; d.t = t; d.dst = outd;
  LR_CUDA(cudaMemcpyAsync(ddesc.p, &d, sizeof(d), cudaMemcpyHostToDevice, st));
  MlpEval ev(ctx, m, psd, B, lr_ode_route(ctx, m, o, B), false);
  ev.prepare();
  if (ev.conv) ev.conv->attach_state(o, io, true);
  if (ev.fe) {   // the same two kernels a solve uses for f(u0, t0): Z(u) by the layer-1 GEMM, then chain + kgemm
    Solver tmp(ctx, DB, DB, 2, 1, 1);
    tmp.init_ctrl(t, t + 1.0f, t + 1.0f, 10, 0, 1e-6f, 1e-6f);
    tmp.enable_latent(ev.fe->zlen());
    tmp.upload();
    LR_CUDA(cudaMemcpyAsync(tmp.tape, ud, 4 * DB, cudaMemcpyDeviceToDevice, st));
    ev.latent_of(tmp.tape, tmp.ztape);
    k1_desc_kernel<<<1, 32, 0, st>>>(tmp.dev);
    LR_COUNT(ctx);
    ev.fe->eval(tmp.dev, &tmp.dev->st[6], nullptr, nullptr, 1);
    LR_CUDA(cudaMemcpyAsync(outd, lr_slot_k(&tmp.h, 0, 1), 4 * DB, cudaMemcpyDeviceToDevice, st));
    LR_CUDA(cudaStreamSynchronize(st));
  } else
  ev.forward((const LinComb*)ddesc.p, nullptr);
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  LR_API_END
}

extern "C" int lrnde_dynamics_vjp(lrnde_ctx* ctx, const lrnde_model* m, const lrnde_opts* o, const float* ps,
                                  const float* u, float t, const float* lam, int64_t B, float* a, float* dps) {
  LR_API_BEGIN
  if (!ctx || !m || !ps || !u || !lam || !a || !dps || B < 1) lr_fail(LRNDE_EINVAL, "lrnde_dynamics_vjp: bad args");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t DB = (size_t)m->D * B;
  CallerBufs io(ctx, o ? o->host_buffers : 0);
  const float* psd = io.in(ps, m->nparams);
  const float* ud = io.in(u, DB);
  const float* ld = io.in(lam, DB);
  float* ad = io.out(a, DB);
  float* gd = io.out(dps, m->nparams);
  DevBuf ddesc(ctx, 2 * (sizeof(LinComb) / 4 + 1));
  LinComb d[2];
  memset(d, 0, sizeof(d));
  d[0].base = ud; d[0].t = t;
  d[1].base = ld; d[1].t = t;
  LinComb* dd = (LinComb*)ddesc.p;
  LR_CUDA(cudaMemcpyAsync(dd, d, sizeof(d), cudaMemcpyHostToDevice, st));
  MlpEval ev(ctx, m, psd, B, lr_ode_route(ctx, m, o, B), true);
  ev.prepare();
  if (ev.conv) ev.conv->attach_state(o, io, false);
  ev.vjp(dd, dd + 1, ad, nullptr, 1.0f, gd, nullptr, 0, 1.0f, 0.0f, nullptr);
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  LR_API_END
}

// ------------------------------------------------------------------------------------------
// forward functor
// ------------------------------------------------------------------------------------------
extern "C" int lrnde_ode_forward(lrnde_ctx* ctx, const lrnde_model* m, const lrnde_opts* o,
                                 const float* ps, const float* x, int64_t B, float* u_save,
                                 int64_t u_save_cap, float* save_times, lrnde_stats* stats,
                                 lrnde_tape** tape_out) {
  LR_API_BEGIN
  if (!ctx || !m || !ps || !x || !stats || B < 1) lr_fail(LRNDE_EINVAL, "lrnde_ode_forward: bad args");
  lr_validate_opts(o);
  if (o->keep_tape && !tape_out) lr_fail(LRNDE_EINVAL, "keep_tape set but tape is NULL");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  memset(stats, 0, sizeof(*stats));
  const long t_call = lr_now_us();
  const long launches0 = ctx->launches;
  const int D = m->D;
  const size_t DB = (size_t)D * B;
  const int64_t P = m->nparams;
  CallerBufs io(ctx, o->host_buffers);

  auto T = std::make_unique<lrnde_tape>();
  T->ctx = ctx;
  T->model = m;
  T->opts = *o;
  T->opts.saveat = nullptr;
  T->B = B;
  T->reg_mode = o->reg_mode;
  T->ps = (float*)ctx->alloc(sizeof(float) * P);
  io.copy_in(T->ps, ps, P);   // kept by the tape
  const bool timing = getenv("LRNDE_TIMING") != nullptr;
  const long tq0 = lr_now_us();
  T->route = lr_ode_route(ctx, m, o, B);
  const OdeRoute& route = T->route;

  // ---- dense tape
  size_t slot_bytes = sizeof(float) * 7 * DB;
  if (route.fused_model)   // latent (+ hidden) tape of the fused engine
    slot_bytes += sizeof(float) * 7 * (size_t)LR_ZROW * (size_t)B * (o->keep_tape ? 2 : 1);
  size_t budget_slots = std::max<size_t>(3, lr_tape_budget(ctx) / slot_bytes);
  const long tq1 = lr_now_us();
  int cap = (int)std::min<size_t>({(size_t)o->maxiters + 2, (size_t)96, budget_slots});
  cap = std::max(cap, 3);
  T->fwd = std::make_unique<Solver>(ctx, DB, DB, cap, 0, o->maxiters + 1);
  Solver& F = *T->fwd;
  if (ctx->nranks > 1) F.h.total_len = (unsigned long long)D * (unsigned long long)ctx->total_batch;
  F.init_ctrl(o->t0, o->t2, o->t2, o->maxiters, o->pow_mode, o->abstol, o->reltol);
  io.copy_in(F.tape, x, DB);   // u_0, the first state of the tape
  LR_CUDA(cudaMemcpyAsync(F.ts, &o->t0, sizeof(float), cudaMemcpyHostToDevice, st));
  const long tq2 = lr_now_us();

  const bool need_vjp = false;
  MlpEval ev(ctx, m, T->ps, B, route, need_vjp);
  if (ev.fe && o->keep_tape) {
    T->Mz = (float*)ctx->alloc(sizeof(float) * 128 * 128);
    ev.mz_plain_out = T->Mz;
  }
  ev.prepare();
  if (ev.conv) {   // st.model: tracked by the main solve's f evaluations only (the closure's st_ at the time
                   // _solve_neuralode_generic returns, neural_ode.jl:44-53)
    const float* used = ev.conv->attach_state(o, io, true);
    if (used && ev.conv->testmode) {   // kept by the tape: the backward normalises with the same statistics
      T->bn_state = (float*)ctx->alloc(4 * ev.conv->nstate);
      LR_CUDA(cudaMemcpyAsync(T->bn_state, used, 4 * ev.conv->nstate, cudaMemcpyDeviceToDevice, st));
    }
  }
  const long tq3 = lr_now_us();
  // latent-space engine (lrnde_fused.h): stage chain in H dimensions + one GEMM per attempt for k_2..k_7
  FusedEngine* fe = ev.fe.get();
  // Z(k_j) and the hidden activations of every stage go to the latent / hidden tapes when a pullback will follow
  // (the latent-space adjoint interpolates them instead of the D-dimensional k's)
  const int write_z = o->keep_tape ? 1 : 0;
  // lean tape: when the pullback will run in hidden space nothing reads k_2..k_6 of the D-dimensional tape (saves and
  // the regulariser's start state come from the hidden tape: FusedEngine::dense_output), so they are not stored
  if (fe) fe->lean = route.lean ? 1 : 0;
  if (fe) {
    F.enable_latent(fe->zlen(), write_z != 0);
    ev.latent_of(F.tape, F.ztape);
    if (F.htape) LR_CUDA(cudaMemsetAsync(F.htape, 0, sizeof(float) * fe->zlen(), st));   // C_0 = 0: u_0 = x + W2a C_0
  }
  auto eval = [&](const LinComb* in, const LinComb*, const int* done, const LinComb* out, bool side) {
    if (fe) fe->eval(F.dev, in, out, done, 1);   // Z(k1) is always needed (next attempt), H(k1) when the tape is kept
    else ev.forward(in, done, out, side);
  };
  F.body = [&]() {
    if (fe) {
      fe->step(F.dev, write_z);
      controller_kernel<<<1, 32, 0, st>>>(F.dev);
      LR_COUNT(ctx);
      LR_CHECK_LAUNCH();
    } else lr_step_body(F, eval, /*fuse_unew=*/true);
  };
  F.build_graphs(o->loop_mode);
  F.upload();
  const long t_start = lr_now_us();
  if (timing)
    fprintf(stderr, "[lrnde] fwd setup us: stage_ps %ld budget %ld tape_alloc %ld prepare %ld graphs %ld (pool %zu blocks)\n",
            tq0 - t_call, tq1 - tq0, tq2 - tq1, tq3 - tq2, t_start - tq3, ctx->pool.size());
  if (ev.conv) ev.conv->first_call_twice = true;   // after the graphs were captured: applies to the k1 launch only
  lr_solver_start(F, eval, 1);
  for (;;) {
    F.run_segment();
    F.download();
    if (!F.h.tape_full) break;
    if ((size_t)F.h.cap * 2 > budget_slots) {
      F.h.c.retcode = LR_RET_TAPEFULL;
      break;
    }
    lr_grow_tape(F);
    segment_begin_kernel<<<1, 32, 0, st>>>(F.dev, 0.0f, 0);
    LR_COUNT(ctx);
  }
  const long t_solve = lr_now_us();
  if (ev.conv) ev.conv->bn_update = false;   // the regulariser's evaluations leave st.model alone
  io.finish();
  const int naccept = F.h.c.naccept, nreject = F.h.c.nreject;
  T->fts.resize(naccept + 1);
  LR_CUDA(cudaMemcpyAsync(T->fts.data(), F.ts, sizeof(float) * (naccept + 1), cudaMemcpyDeviceToHost, st));
  LR_CUDA(cudaStreamSynchronize(st));
  lr_copy_log(F, T.get(), 0);
  const float t_last = T->fts.back();

  // ---- which times the returned solution holds (neural_ode.jl:102-116), and their states
  T->saves = lr_save_plan(*o, T->fts);
  const float t1 = T->saves.t1;
  const int mode = o->reg_mode;
  const int nout = T->saves.nout;
  if (u_save && nout > u_save_cap)
    lr_fail(LRNDE_EINVAL, "u_save holds %lld blocks but the solution has %d", (long long)u_save_cap, nout);
  lr_write_saves(ctx, T.get(), route.lean ? fe : nullptr, u_save, save_times);

  const long t_saves = lr_now_us();
  // ---- local regulariser: integrator at t1 + one differentiable step (neural_ode.jl:75-78)
  int nf_reg = 0;
  float reg_val = 0.0f, dt_reg = 0.0f;
  if (mode != LRNDE_REG_NONE) {
    T->reg = std::make_unique<Solver>(ctx, DB, DB, 2, 1, 1);
    Solver& R = *T->reg;
    if (ctx->nranks > 1) R.h.total_len = F.h.total_len;
    R.init_ctrl(t1, o->t2, o->t2, o->maxiters, o->pow_mode, o->abstol, o->reltol);
    // hidden images [h_j ; t_j ; 1] of the regulariser's stages for the hidden-space reverse pass (lrnde_regrev.cuh)
    if (fe) R.enable_latent(fe->zlen(), route.reg_hidden);
    R.upload();
    LinComb u1;
    DevBuf dd(ctx, sizeof(LinComb) / 4 + 1);
    lr_sol_at(ctx, T.get(), route.lean ? fe : nullptr, std::min(t1, t_last), R.tape, &u1, (const LinComb*)dd.p);
    if (fe) fe->lean = 0;   // the regulariser integrator keeps k_2..k_6 (its reverse pass reads them)
    if (fe) {
      ev.latent_of(R.tape, R.ztape);
      auto evalR = [&](const LinComb* in, const LinComb*, const int* done, const LinComb* out, bool) {
        fe->eval(R.dev, in, out, done, 1);
      };
      lr_solver_start(R, evalR, 0);
      fe->step(R.dev, 0);   // the six stages, u, k7 and the residual partial sums (perform_step.jl:10-27)
    } else {
      lr_solver_start(R, eval, 0);
      for (int j = 0; j < 5; ++j) eval(&R.dev->st[j], nullptr, &R.dev->failed, nullptr, false);
      eval(&R.dev->st[5], nullptr, &R.dev->failed, &R.dev->st[6], true);   // u and k7 in one pass
      err_norm_kernel<<<LR_ERR_BLOCKS, 256, 0, st>>>(R.dev);
      LR_COUNT(ctx);
    }
    if (o->reg_type == LRNDE_REGTYPE_STIFFNESS) {
      reg_stiff_sums_kernel<<<LR_ERR_BLOCKS, 256, 0, st>>>(R.dev);
      LR_COUNT(ctx);
    }
    reg_value_kernel<<<1, 32, 0, st>>>(R.dev, o->reg_type);
    LR_COUNT(ctx);
    LR_CHECK_LAUNCH();
    R.download();
    reg_val = R.h.reg_val;
    dt_reg = R.h.c.dt;
    nf_reg = 9;  // 6 + integrator.sol.destats.nf (perform_step.jl:31)
  }

  if (ev.conv) ctx->bn_check();
  stats->naccept = naccept;
  stats->nreject = nreject;
  stats->retcode = F.h.c.retcode;
  stats->nfe = 3 + 6 * (naccept + nreject) + nf_reg;
  stats->reg_val = reg_val;
  stats->t1_used = t1;
  stats->dt_reg = dt_reg;
  stats->nsave_out = nout;
  stats->gpu_launches = (int)((ctx->launches - launches0) + F.body_nodes * (long)F.h.nlog);
  // host wall-clock of the phases (each ends on a stream sync), microseconds: diagnostics
  stats->reserved[0] = (int32_t)(t_solve - t_start);
  stats->reserved[1] = (int32_t)(t_saves - t_solve);
  stats->reserved[2] = (int32_t)(lr_now_us() - t_saves);
  stats->reserved[5] = (int32_t)(t_start - t_call);   // setup: staging, weight images, graph capture + instantiation
  if (o->keep_tape) *tape_out = T.release();
  else if (tape_out) *tape_out = nullptr;
  LR_API_END
}

// The saved states of a kept solution, written after the call (every-step saves of the :biased path: the number of
// accepted steps is only known after the solve, so lrnde_ode_forward can run with u_save = NULL and the caller sizes
// the buffer from stats->nsave_out).  u_save / save_times: as in lrnde_ode_forward (HOST pointers when the forward
// call had host_buffers).
extern "C" int lrnde_ode_saved_states(lrnde_ctx* ctx, const lrnde_model* m, lrnde_tape* T, float* u_save,
                                      int64_t u_save_cap, float* save_times) {
  LR_API_BEGIN
  if (!ctx || !m || !T || !u_save) lr_fail(LRNDE_EINVAL, "lrnde_ode_saved_states: bad args");
  if (T->ctx != ctx || T->model != m) lr_fail(LRNDE_ESTATE, "tape belongs to another ctx/model");
  LR_CUDA(cudaSetDevice(ctx->device));
  if (T->saves.nout > u_save_cap)
    lr_fail(LRNDE_EINVAL, "u_save holds %lld blocks but the solution has %d", (long long)u_save_cap, T->saves.nout);
  std::unique_ptr<FusedEngine> lean_fe;
  if (T->route.lean) lean_fe = std::make_unique<FusedEngine>(ctx, m, T->ps, T->B, T->route.passes);
  lr_write_saves(ctx, T, lean_fe.get(), u_save, save_times);
  LR_API_END
}

extern "C" int lrnde_tape_free(lrnde_tape* t) {
  LR_API_BEGIN
  if (t) {
    cudaSetDevice(t->ctx->device);
    cudaStreamSynchronize(t->ctx->stream);
    delete t;
  }
  LR_API_END
}

extern "C" int lrnde_step_log(const lrnde_tape* t, int which, float* tt, float* dt, float* eest,
                              uint8_t* accepted, int cap, int* n) {
  LR_API_BEGIN
  if (!t || which < 0 || which > 1 || !n) lr_fail(LRNDE_EINVAL, "lrnde_step_log: bad args");
  int cnt = (int)t->log_t[which].size();
  *n = cnt;
  int k = std::min(cnt, cap);
  for (int i = 0; i < k; ++i) {
    if (tt) tt[i] = t->log_t[which][i];
    if (dt) dt[i] = t->log_dt[which][i];
    if (eest) eest[i] = t->log_eest[which][i];
    if (accepted) accepted[i] = t->log_acc[which][i];
  }
  LR_API_END
}

// ------------------------------------------------------------------------------------------
// pullback: continuous adjoint over z = [lambda; mu] + reverse pass of the regulariser step
// ------------------------------------------------------------------------------------------
// last result of the LRNDE_PROFILE_ADJ=<iters> hook of lrnde_ode_backward: microseconds per launch of one attempt
// of the latent-space adjoint {chain, lambda GEMM, pairacc, reduce + mu, whole attempt} (CUDA events on the ctx stream)
static float g_adj_profile_us[5] = {0, 0, 0, 0, 0};
extern "C" int lrnde_profile_adjoint_last(float* us5) {
  if (!us5) return LRNDE_EINVAL;
  for (int k = 0; k < 5; ++k) us5[k] = g_adj_profile_us[k];
  return LRNDE_OK;
}

// the launches of the first attempt, repeated (same descriptors: the controller does not run; they only write the next
// ring slot, which the real attempt recomputes), timed with CUDA events on the library's stream
static void lr_profile_adjoint(lrnde_ctx* ctx, LatentAdjoint& la, SolveDev* A, int iters, bool timing) {
  cudaStream_t st = ctx->stream;
  cudaEvent_t e[6];
  for (auto& ev_ : e) LR_CUDA(cudaEventCreate(&ev_));
  for (int w = 0; w < 2; ++w) la.attempt(A);
  for (int k = 0; k < 4; ++k) {
    LR_CUDA(cudaEventRecord(e[k], st));
    for (int i = 0; i < iters; ++i) la.attempt_part(A, k);
  }
  LR_CUDA(cudaEventRecord(e[4], st));
  for (int i = 0; i < iters; ++i) la.attempt(A);
  LR_CUDA(cudaEventRecord(e[5], st));
  LR_CUDA(cudaEventSynchronize(e[5]));
  const char* nm[5] = {"chain", "lambda gemm", "pairacc", "reduce + mu", "attempt"};
  for (int k = 0; k < 5; ++k) {
    float ms = 0.0f;
    LR_CUDA(cudaEventElapsedTime(&ms, e[k], e[k + 1]));
    g_adj_profile_us[k] = 1000.0f * ms / (float)iters;
    if (timing) fprintf(stderr, "[lrnde] adjoint attempt: %-12s %8.1f us\n", nm[k], g_adj_profile_us[k]);
  }
  for (auto& ev_ : e) cudaEventDestroy(ev_);
}

// ------------------------------------------------------------------------------------------
// Reverse pass of the regulariser step in hidden space (lrnde_regrev.cuh): 2-layer TD-MLP with tanh,
// regularize_type = :error_estimate.  dps += d_reg * d reg_val / d ps.
// ------------------------------------------------------------------------------------------
static void lr_wgrad_launch(lrnde_ctx* ctx, const umma::WgOperand& P, const umma::WgOperand& Q, int transposed, int ldo, int64_t N,
                            float* part, size_t block, int nsplit, int chunk, int passes, const int* done) {
  static bool attr_set = false;
  if (!attr_set) {
    LR_CUDA(cudaFuncSetAttribute(umma::wgrad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, umma::wgrad_smem()));
    LR_CUDA(cudaFuncSetAttribute(umma::wgrad_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, umma::wgrad_smem()));
    attr_set = true;
  }
  umma::WgradUP w;
  memset(&w, 0, sizeof(w));
  w.P = P; w.Q = Q; w.transposed = transposed; w.ldo = ldo;
  w.B = (int)N; w.chunk = chunk; w.part = part; w.block = block; w.passes = passes; w.tdesc = nullptr; w.done = done;
  dim3 g((P.rows + 127) / 128, nsplit);
  const bool lean = P.rows % 4 == 0 && Q.rows % 4 == 0 && P.ld % 4 == 0 && Q.ld % 4 == 0 &&
                    (((uintptr_t)P.ptr) & 15) == 0 && (((uintptr_t)Q.ptr) & 15) == 0;
  if (lean) umma::wgrad_kernel<false><<<g, umma::kThreads, umma::wgrad_smem(), ctx->stream>>>(w);
  else umma::wgrad_kernel<true><<<g, umma::kThreads, umma::wgrad_smem(), ctx->stream>>>(w);
  LR_COUNT(ctx);
}
// batch split of a contraction over N samples with n_mt row tiles: one wave of CTAs, chunks of a multiple of 32
static void lr_wgrad_split(int64_t N, int n_mt, int* nsplit, int* chunk) {
  int us = std::max(1, std::min(64, 148 / n_mt));
  int uc = (int)((N + us - 1) / us);
  uc = std::max(32, ((uc + 31) / 32) * 32);
  *nsplit = (int)((N + uc - 1) / uc);
  *chunk = uc;
}

static void lr_reg_pullback_hidden(lrnde_ctx* ctx, const lrnde_model* m, lrnde_tape* T, MlpEval& ev, float d_reg, float* dps_dev) {
  cudaStream_t st = ctx->stream;
  Solver& R = *T->reg;
  const int64_t B = T->B;
  FusedShape sh;
  lrf_shape(m, &sh);
  const int D = sh.D, H = sh.H, Kaug = sh.Kaug, td = m->td;
  const int KP = 104;                         // rows of the padded hidden operands (multiple of 4 >= Kaug + td + 1)
  const size_t DB = (size_t)D * B, ZB = (size_t)LR_ZROW * B;
  const LayerInfo &L1 = m->layers[0], &L2 = m->layers[1];
  const int* done = nullptr;

  // (1) G, Q
  DevBuf gq(ctx, 2 * DB);
  RegSeedGQP sp;
  sp.R = R.dev; sp.d_reg = d_reg; sp.gq = gq.p; sp.DB = DB;
  reg_seed_gq_kernel<<<lr_ew_blocks(DB), 256, 0, st>>>(sp);
  LR_COUNT(ctx);
  // (2) A = W2^T G, Bq = W2^T Q: one GEMM over 2B columns
  DevBuf ab(ctx, 2 * ZB);
  {
    DenseP p;
    memset(&p, 0, sizeof(p));
    p.A = ev.WT[1]; p.lda = L2.in; p.M = L2.in; p.K = L2.out; p.td = 0; p.bias = 0;
    p.X = gq.p; p.ldx = L2.out; p.N = (int)(2 * B);
    p.Y = ab.p; p.ldy = LR_ZROW; p.act = ACT_IDENTITY; p.dact = -1; p.out_scale = 1.0f; p.done = done;
    ev.dense(p, ev.use_umma ? ev.packWT[1] : nullptr);
  }
  // (3) the stage cotangents in hidden space
  DevBuf work(ctx, (6 + 6 + 1 + 1 + 2) * ZB);
  RegRevP rp;
  memset(&rp, 0, sizeof(rp));
  rp.R = R.dev; rp.Mz = T->Mz; rp.ab = ab.p;
  for (int j = 1; j <= 6; ++j) rp.hh[j - 1] = R.htape + (size_t)j * R.h.zlen;     // K(0, j)
  rp.hh[6] = R.htape + (size_t)8 * R.h.zlen;                                       // k7 = K(1, 1)
  rp.del = work.p; rp.cc = work.p + 6 * ZB; rp.dsum = work.p + 12 * ZB; rp.uv = work.p + 13 * ZB; rp.hba = work.p + 14 * ZB;
  rp.B = (int)B; rp.H = H; rp.Kaug = Kaug; rp.td = td;
  for (int r = 0; r < 6; ++r) for (int i = 0; i < 6; ++i) rp.a[r][i] = lr_tsit5_a(r, i);
  for (int i = 0; i < 7; ++i) rp.bt[i] = lr_tsit5_btilde(i);
  {
    const size_t smem = sizeof(float) * ((size_t)H * 128 + 2 * 128 * 4);
    static bool attr_set = false;
    if (!attr_set) {
      LR_CUDA(cudaFuncSetAttribute(reg_rev_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 128 * 4 + 4096));
      attr_set = true;
    }
    const int npairs = (int)((B + 2 * kRegRevS - 1) / (2 * kRegRevS));
    reg_rev_chain_kernel<<<std::min(npairs, 2 * 148), 256, smem, st>>>(rp);
    LR_COUNT(ctx);
  }
  // (4) the four batch contractions on the tensor cores (fixed split, fixed-order reduce in (5))
  int s1, c1, s2, c2, s3, c3, s4, c4;
  lr_wgrad_split(2 * B, (D + 127) / 128, &s1, &c1);
  lr_wgrad_split(B, (D + 127) / 128, &s2, &c2);
  lr_wgrad_split(6 * B, 1, &s3, &c3);
  lr_wgrad_split(B, 1, &s4, &c4);
  const size_t b1 = (size_t)D * KP, b2 = (size_t)H * D, b3 = (size_t)H * KP;
  DevBuf part(ctx, s1 * b1 + s2 * b2 + (size_t)(s3 + s4) * b3 + 2 * (size_t)H * Kaug);
  float* t1 = part.p; float* t2 = t1 + s1 * b1; float* ssb = t2 + s2 * b2; float* uhb = ssb + s3 * b3; float* smb = uhb + s4 * b3;
  const float* uprev = R.tape;   // U(0) of the regulariser integrator
  {
    umma::WgOperand oG = {gq.p, D, D, 0, 0, 0};
    umma::WgOperand oHBA = {rp.hba, LR_ZROW, KP, 0, 0, 0};
    lr_wgrad_launch(ctx, oG, oHBA, 0, D, 2 * B, t1, b1, s1, c1, ev.passes, done);
    umma::WgOperand oU = {uprev, D, D, 0, 0, 0};
    umma::WgOperand oDS = {rp.dsum, LR_ZROW, H, 0, 0, 0};
    lr_wgrad_launch(ctx, oU, oDS, 1, H, B, t2, b2, s2, c2, ev.passes, done);
    umma::WgOperand oCC = {rp.cc, LR_ZROW, KP, 0, 0, 0};
    umma::WgOperand oDEL = {rp.del, LR_ZROW, H, 0, 0, 0};
    lr_wgrad_launch(ctx, oCC, oDEL, 1, H, 6 * B, ssb, b3, s3, c3, ev.passes, done);
    umma::WgOperand oH1 = {rp.hh[0], LR_ZROW, KP, 0, 0, 0};
    umma::WgOperand oUV = {rp.uv, LR_ZROW, H, 0, 0, 0};
    lr_wgrad_launch(ctx, oH1, oUV, 1, H, B, uhb, b3, s4, c4, ev.passes, done);
  }
  // (5) d_ps += ...
  RegAsmP ap;
  memset(&ap, 0, sizeof(ap));
  ap.R = R.dev; ap.ps = T->ps; ap.dps = dps_dev; ap.t1 = t1; ap.t2 = t2; ap.ss = ssb; ap.uh = uhb; ap.sm = smb;
  ap.S1 = s1; ap.S2 = s2; ap.S3 = s3; ap.S4 = s4; ap.D = D; ap.H = H; ap.Kaug = Kaug; ap.td = td; ap.KP = KP;
  ap.w1_off = (long)L1.w_off; ap.w2_off = (long)L2.w_off;
  reg_ss_kernel<<<(H * Kaug + 255) / 256, 256, 0, st>>>(ap);
  LR_COUNT(ctx);
  reg_assemble_kernel<<<lr_ew_blocks((size_t)D * Kaug + (size_t)H * D), 256, 0, st>>>(ap);
  LR_COUNT(ctx);
  LR_CHECK_LAUNCH();
  LR_CUDA(cudaStreamSynchronize(st));   // the scratch buffers go back to the pool
}

// The same reverse pass through the per-layer pullback of f, stage by stage (any model and regularize_type)
static void lr_reg_pullback_layers(lrnde_ctx* ctx, const lrnde_model* m, lrnde_tape* T, MlpEval& ev, float d_reg,
                                   float* dps_dev) {
  cudaStream_t st = ctx->stream;
  Solver& R = *T->reg;
  const size_t DB = (size_t)m->D * T->B;
  DevBuf work(ctx, 9 * DB);
  RegSeedP sp;
  sp.R = R.dev; sp.reg_type = T->opts.reg_type; sp.d_reg = d_reg;
  for (int k = 0; k < 6; ++k) sp.dk[k] = work.p + (size_t)k * DB;
  sp.du = work.p + 6 * DB;
  sp.dg6 = work.p + 7 * DB;
  float* abuf = work.p + 8 * DB;
  reg_seed_kernel<<<lr_ew_blocks(DB), 256, 0, st>>>(sp);
  LR_COUNT(ctx);
  std::vector<LinComb> lam(6);
  for (int k = 0; k < 6; ++k) { memset(&lam[k], 0, sizeof(LinComb)); lam[k].base = sp.dk[k]; }
  DevBuf dl(ctx, 6 * (sizeof(LinComb) / 4 + 1));
  LR_CUDA(cudaMemcpyAsync(dl.p, lam.data(), sizeof(LinComb) * 6, cudaMemcpyHostToDevice, st));
  const LinComb* lamd = (const LinComb*)dl.p;
  for (int row = 5; row >= 0; --row) {
    const LinComb* y = (row == 5) ? &R.dev->st[6] : &R.dev->st[row];
    ev.vjp(y, lamd + row, abuf, nullptr, 1.0f, dps_dev, nullptr, 0, 1.0f, 1.0f, nullptr);
    if (row == 0) break;  // k2's input depends on k1 only (constant)
    RegBwdP bp;
    bp.R = R.dev; bp.row = row; bp.a = abuf; bp.du = sp.du; bp.dg6 = sp.dg6;
    for (int k = 0; k < 6; ++k) { bp.dk[k] = sp.dk[k]; bp.coef[k] = lr_tsit5_a(row, k); }
    reg_bwd_stage_kernel<<<lr_ew_blocks(DB), 256, 0, st>>>(bp);
    LR_COUNT(ctx);
  }
  LR_CHECK_LAUNCH();
  LR_CUDA(cudaStreamSynchronize(st));
}


extern "C" int lrnde_ode_backward(lrnde_ctx* ctx, const lrnde_model* m, lrnde_tape* T,
                                  const float* d_u_save, float d_reg, float* d_ps, float* d_x,
                                  lrnde_stats* stats) {
  LR_API_BEGIN
  if (!ctx || !m || !T || !d_ps || (!d_x && !T->opts.no_dx)) lr_fail(LRNDE_EINVAL, "lrnde_ode_backward: bad args");
  if (T->ctx != ctx || T->model != m) lr_fail(LRNDE_ESTATE, "tape belongs to another ctx/model");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const lrnde_opts& o = T->opts;
  const int64_t B = T->B;
  const int D = m->D;
  const size_t DB = (size_t)D * B;
  const size_t P = (size_t)m->nparams;
  const size_t len = DB + P;
  const long launches0 = ctx->launches;
  const long tb_call = lr_now_us();
  Solver& F = *T->fwd;
  const int nsteps = (int)T->fts.size() - 1;
  const float t0 = T->fts.front(), t2 = T->fts.back();
  const OdeRoute& route = T->route;

  // cotangent blocks on the device
  CallerBufs io(ctx, o.host_buffers);
  const float* dU = io.in(d_u_save, DB * (size_t)T->saves.nout);
  auto cot_blocks = [&](float tval, std::vector<const float*>& out) {
    out.clear();
    if (!dU) return;
    for (int blk : T->saves.blocks_at(tval, t2)) out.push_back(dU + (size_t)blk * DB);
  };

  MlpEval ev(ctx, m, T->ps, B, route, true);
  ev.prepare();
  if (ev.conv && o.model_testmode) { ev.conv->bn_state = T->bn_state; ev.conv->testmode = 1; }

  const bool no_dx = o.no_dx != 0;   // the caller has no use for dL/dx (nothing upstream has parameters)
  float* dx_dev = io.out(no_dx ? nullptr : d_x, DB);
  float* dps_dev = io.out(d_ps, P);
  DevBuf dx_scratch(ctx, dx_dev ? 1 : DB);   // the adjoint solve forms dL/dx even when it is not returned
  if (!dx_dev) dx_dev = dx_scratch.p;

  const long tb_start = lr_now_us();
  int nbwd_stops = 0;
  int retcode_bwd = 0, nacc_b = 0, nrej_b = 0;
  long body_launches = 0;
  if (nsteps >= 1) {
    const bool timing = getenv("LRNDE_TIMING") != nullptr;
    long tmark = lr_now_us();
    auto mark = [&](const char* what) {
      if (!timing) return;
      cudaStreamSynchronize(st);
      const long now = lr_now_us();
      fprintf(stderr, "[lrnde] bwd %-14s %8ld us\n", what, now - tmark);
      tmark = now;
    };
    Solver A(ctx, len, DB, 2, 1, o.maxiters + 1);
    mark("solver alloc");
    A.h.is_adjoint = 1;
    A.h.fts = F.ts;
    A.h.ftape = F.tape;
    A.h.flen = DB;
    A.h.fnsteps = nsteps;
    A.h.ftdir = 1;
    // latent-space adjoint (lrnde_adjoint.h): the forward solve kept its hidden tape
    std::unique_ptr<LatentAdjoint> la;
    if (route.latent_adj) {
      la = std::make_unique<LatentAdjoint>(ctx, m, T->ps, B, ev.passes);
      la->W1T = ev.WT[0]; la->Zx = F.ztape; la->x = F.tape;
      la->prepare(T->Mz);
      A.h.fhtape = F.htape;
      A.h.fztape = F.ztape;
      A.h.fzlen = F.h.zlen;
      A.h.lat_mu_row = 1;
    }
    // alpha = W2^T lambda of the current state (start of a segment), then the stage-1 quantities
    auto latent_begin = [&]() {
      const LayerInfo& L2 = m->layers[1];
      DenseP p;
      memset(&p, 0, sizeof(p));
      p.A = ev.WT[1]; p.lda = L2.in; p.M = L2.in; p.K = L2.out; p.td = 0; p.bias = 0;
      p.xdesc = &A.dev->cur; p.ldx = L2.out; p.N = (int)B;
      p.Y = la->alpha_in; p.ldy = LR_ZROW; p.act = ACT_IDENTITY; p.dact = -1; p.out_scale = 1.0f;
      p.done = &A.dev->failed;
      ev.dense(p, ev.packWT[1]);
      la->begin(A.dev);
    };
    if (ctx->nranks > 1) {
      A.h.total_len = (unsigned long long)D * (unsigned long long)ctx->total_batch + P;
      A.enable_mu_exchange(P);
    }
    // tstops: the saved times strictly inside (t0, t2), descending, then t0
    std::vector<float> stops = T->saves.interior_stops(t0, t2);
    stops.push_back(t0);
    A.init_ctrl(t2, t0, stops[0], o.maxiters, o.pow_mode, o.abstol, o.reltol);
    // lean tape: the per-layer right-hand side (initial-dt probes only) reads y(t) materialised from the hidden tape
    std::unique_ptr<FusedEngine> fe_y;
    std::unique_ptr<DevBuf> ybuf, ydescs;
    if (route.lean) {
      fe_y = std::make_unique<FusedEngine>(ctx, m, T->ps, B, ev.passes);
      ybuf = std::make_unique<DevBuf>(ctx, DB);
      ydescs = std::make_unique<DevBuf>(ctx, 2 * (sizeof(LinComb) / 4 + 1));
      LinComb od;
      memset(&od, 0, sizeof(od));
      od.dst = ybuf->p;
      LR_CUDA(cudaMemcpyAsync(ydescs->p, &od, sizeof(LinComb), cudaMemcpyHostToDevice, st));
    }
    auto rhs = [&](const LinComb* in, const LinComb* y, const int* done, const LinComb*, bool) {
      if (route.lean) {
        LinComb* out_desc = (LinComb*)ydescs->p;       // {dst = ybuf}
        LinComb* y_mat = out_desc + 1;                 // {base = ybuf, t = y->t}, written on the device
        fe_y->dense_output_dev(A.dev, y, F.tape, ybuf->p, y_mat, out_desc);
        y = y_mat;
      }
      ev.vjp(y, in, nullptr, in, -1.0f, nullptr, in, DB, -1.0f, 0.0f, done);
    };
    A.body = [&]() {
      if (la) {
        la->attempt(A.dev);
        controller_kernel<<<1, 32, 0, st>>>(A.dev);
        LR_COUNT(ctx);
        LR_CHECK_LAUNCH();
      } else lr_step_body(A, rhs);
    };
    mark("latent setup");
    A.build_graphs(o.loop_mode);
    A.upload();
    mark("graphs");
    // z(t2) = [dL/du(t2); 0]
    LR_CUDA(cudaMemsetAsync(A.tape, 0, sizeof(float) * len, st));
    std::vector<const float*> blocks;
    cot_blocks(t2, blocks);
    for (auto b : blocks) {
      axpy_kernel<<<lr_ew_blocks(DB), 256, 0, st>>>(A.tape, b, 1.0f, DB);
      LR_COUNT(ctx);
    }
    lr_solver_start(A, rhs, 1);
    mark("solver start");
    // data-parallel group: the replicated global mu of the latent-space engine starts at mu(t2) = 0 (ring slot 0)
    if (la && A.muglob) LR_CUDA(cudaMemsetAsync(A.muglob, 0, sizeof(float) * P, st));
    if (la) latent_begin();
    mark("latent begin");
    if (la && getenv("LRNDE_PROFILE_ADJ")) lr_profile_adjoint(ctx, *la, A.dev, std::max(1, atoi(getenv("LRNDE_PROFILE_ADJ"))), timing);
    for (size_t si = 0; si < stops.size(); ++si) {
      A.run_segment();
      mark("segment");
      if (si + 1 < stops.size()) {
        cot_blocks(stops[si], blocks);
        for (auto b : blocks) {
          jump_kernel<<<lr_ew_blocks(DB), 256, 0, st>>>(A.dev, b, DB);
          LR_COUNT(ctx);
        }
        k1_desc_kernel<<<1, 32, 0, st>>>(A.dev);
        LR_COUNT(ctx);
        if (la) latent_begin();
        else rhs(&A.dev->st[6], &A.dev->yint[6], &A.dev->failed, nullptr, false);
        segment_begin_kernel<<<1, 32, 0, st>>>(A.dev, stops[si + 1], 1);
        LR_COUNT(ctx);
        nbwd_stops++;
      }
    }
    LR_CHECK_LAUNCH();
    A.download();
    lr_copy_log(A, T, 1);
    const float* z = A.tape + (size_t)A.h.slot * 7 * len;
    LR_CUDA(cudaMemcpyAsync(dx_dev, z, sizeof(float) * DB, cudaMemcpyDeviceToDevice, st));
    LR_CUDA(cudaMemcpyAsync(dps_dev, z + DB, sizeof(float) * P, cudaMemcpyDeviceToDevice, st));
    cot_blocks(t0, blocks);
    for (auto b : blocks) {
      axpy_kernel<<<lr_ew_blocks(DB), 256, 0, st>>>(dx_dev, b, 1.0f, DB);
      LR_COUNT(ctx);
    }
    retcode_bwd = A.h.c.retcode;
    nacc_b = A.h.c.naccept;
    nrej_b = A.h.c.nreject;
    body_launches = A.body_nodes * (long)A.h.nlog;
    LR_CUDA(cudaStreamSynchronize(st));
  } else {
    LR_CUDA(cudaMemsetAsync(dx_dev, 0, sizeof(float) * DB, st));
    LR_CUDA(cudaMemsetAsync(dps_dev, 0, sizeof(float) * P, st));
  }

  const long tb_adj = lr_now_us();
  // ---- reverse pass of the regulariser step: gradient w.r.t. ps only
  if (T->reg && d_reg != 0.0f) {
    if (route.reg_hidden) lr_reg_pullback_hidden(ctx, m, T, ev, d_reg, dps_dev);
    else lr_reg_pullback_layers(ctx, m, T, ev, d_reg, dps_dev);
  }
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  if (ev.conv) ctx->bn_check();
  if (stats) {
    stats->nf_bwd = (nsteps >= 1) ? 3 + 6 * (nacc_b + nrej_b) + nbwd_stops : 0;
    stats->naccept_bwd = nacc_b;
    stats->nreject_bwd = nrej_b;
    stats->retcode_bwd = retcode_bwd;
    stats->gpu_launches = (int)((ctx->launches - launches0) + body_launches);
    stats->reserved[3] = (int32_t)(tb_adj - tb_start);
    stats->reserved[5] = (int32_t)(tb_start - tb_call);
    stats->reserved[4] = (int32_t)(lr_now_us() - tb_adj);
  }
  LR_API_END
}

// ------------------------------------------------------------------------------------------
// profiling hook: one Tsit5 attempt of the latent-space engine, repeated (same descriptors: the controller
// does not run), timed with CUDA events on the library's stream.  us[0] = chain kernel, us[1] = kgemm kernel,
// us[2] = the attempt as the solve loop runs it (chain + kgemm + controller arithmetic excluded)
// ------------------------------------------------------------------------------------------
extern "C" int lrnde_profile_step(lrnde_ctx* ctx, const lrnde_model* m, const lrnde_opts* o, const float* ps,
                                  const float* x, int64_t B, int32_t iters, float* us) {
  LR_API_BEGIN
  if (!ctx || !m || !o || !ps || !x || !us || B < 1 || iters < 1) lr_fail(LRNDE_EINVAL, "lrnde_profile_step: bad args");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t DB = (size_t)m->D * B;
  const OdeRoute route = lr_ode_route(ctx, m, o, B);
  if (!route.fused) lr_fail(LRNDE_EINVAL, "lrnde_profile_step: the model / precision does not use the latent-space engine");
  MlpEval ev(ctx, m, ps, B, route, false);
  ev.prepare();
  Solver F(ctx, DB, DB, 3, 0, 8);
  F.init_ctrl(o->t0, o->t2, o->t2, o->maxiters, o->pow_mode, o->abstol, o->reltol);
  F.enable_latent(ev.fe->zlen(), o->keep_tape != 0);   // keep_tape: the training configuration (hidden tape, lean D-tape)
  if (F.htape) LR_CUDA(cudaMemsetAsync(F.htape, 0, sizeof(float) * ev.fe->zlen(), st));
  ev.fe->lean = route.lean ? 1 : 0;
  LR_CUDA(cudaMemcpyAsync(F.tape, x, sizeof(float) * DB, cudaMemcpyDeviceToDevice, st));
  F.h.use_cond = 0;
  F.upload();
  ev.latent_of(F.tape, F.ztape);
  auto eval = [&](const LinComb* in, const LinComb*, const int* done, const LinComb* out, bool) {
    ev.fe->eval(F.dev, in, out, done, 1);
  };
  lr_solver_start(F, eval, 1);
  cudaEvent_t e[4];
  for (auto& ev_ : e) LR_CUDA(cudaEventCreate(&ev_));
  for (int w = 0; w < 2; ++w) ev.fe->step(F.dev, 0);
  LR_CUDA(cudaEventRecord(e[0], st));
  for (int i = 0; i < iters; ++i) ev.fe->step_chain(F.dev, 0);
  LR_CUDA(cudaEventRecord(e[1], st));
  for (int i = 0; i < iters; ++i) ev.fe->step_kgemm(F.dev);
  LR_CUDA(cudaEventRecord(e[2], st));
  for (int i = 0; i < iters; ++i) ev.fe->step(F.dev, 0);
  LR_CUDA(cudaEventRecord(e[3], st));
  LR_CUDA(cudaEventSynchronize(e[3]));
  for (int k = 0; k < 3; ++k) {
    float ms = 0.0f;
    LR_CUDA(cudaEventElapsedTime(&ms, e[k], e[k + 1]));
    us[k] = 1000.0f * ms / (float)iters;
  }
  for (auto& ev_ : e) cudaEventDestroy(ev_);
  LR_API_END
}

// ------------------------------------------------------------------------------------------
// One gradient evaluation of the MNIST classifier Chain(FlattenLayer, NeuralODE, diffeqsol_to_array, Dense(D => C))
// (experiments/src/construct.jl:180-200) under the training loss logitcrossentropy + w_reg * reg_val
// (construct.jl:19-31), i.e. what Zygote.pullback does in run_training_step (experiments/src/utils.jl:106-115) --
// with u(t2) and its cotangent kept on the device: only x, the labels and the parameters go in, only the loss and
// the parameter gradients come out.
// ------------------------------------------------------------------------------------------
__global__ void scale_kernel(float* v, float s, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) v[i] *= s;
}
// The next batch's inputs, copied host -> device on a separate copy stream while the current call computes: the
// input pipeline of a training loop (the reference's DataLoader + `gpu` transfer, experiments/src/utils.jl:106-115).
// lrnde_classifier_grad (host_buffers) then finds the staged copy by the host pointers instead of copying again.
static void lr_flush_prefetch(lrnde_ctx* ctx) {
  if (!ctx->pending.valid) return;
  const float* x = ctx->pending.x; const int32_t* labels = ctx->pending.y;
  const int64_t B = ctx->pending.B; const int32_t D = ctx->pending.D;
  ctx->pending.valid = false;
  if (!ctx->copy_stream) LR_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  // the slot that is free, else the older one
  int pick = 0;
  if (ctx->staged[0].ready && (!ctx->staged[1].ready || ctx->staged[1].seq < ctx->staged[0].seq)) pick = 1;
  lrnde_ctx::Staged& sg = ctx->staged[pick];
  const size_t nx = (size_t)D * (size_t)B, ny = (size_t)B;
  if (sg.cap_x < nx) { if (sg.x) cudaFree(sg.x); LR_CUDA(cudaMalloc((void**)&sg.x, 4 * nx)); sg.cap_x = nx; }
  if (sg.cap_y < ny) { if (sg.y) cudaFree(sg.y); LR_CUDA(cudaMalloc((void**)&sg.y, 4 * ny)); sg.cap_y = ny; }
  if (!sg.ev) LR_CUDA(cudaEventCreateWithFlags(&sg.ev, cudaEventDisableTiming));
  LR_CUDA(cudaMemcpyAsync(sg.x, x, 4 * nx, cudaMemcpyHostToDevice, ctx->copy_stream));
  LR_CUDA(cudaMemcpyAsync(sg.y, labels, 4 * ny, cudaMemcpyHostToDevice, ctx->copy_stream));
  LR_CUDA(cudaEventRecord(sg.ev, ctx->copy_stream));
  sg.key_x = x; sg.key_y = labels; sg.nx = nx; sg.ny = ny; sg.seq = ++ctx->staged_seq; sg.ready = true;
}

extern "C" int lrnde_prefetch_inputs(lrnde_ctx* ctx, const float* x, const int32_t* labels, int64_t B, int32_t D) {
  LR_API_BEGIN
  if (!ctx || !x || !labels || B < 1 || D < 1) lr_fail(LRNDE_EINVAL, "lrnde_prefetch_inputs: bad args");
  LR_CUDA(cudaSetDevice(ctx->device));
  lr_flush_prefetch(ctx);   // an earlier request nobody flushed: its copy starts now
  ctx->pending.x = x; ctx->pending.y = labels; ctx->pending.B = B; ctx->pending.D = D; ctx->pending.valid = true;
  LR_API_END
}

extern "C" int lrnde_classifier_grad(lrnde_ctx* ctx, const lrnde_model* m, const lrnde_opts* o, const float* ps,
                                     const float* Wc, const float* x, const int32_t* labels, int64_t B, int32_t Cn,
                                     float w_reg, float grad_scale, float* loss_ce, float* d_ps, float* d_Wc,
                                     lrnde_stats* stats) {
  LR_API_BEGIN
  if (!ctx || !m || !o || !ps || !Wc || !x || !labels || !loss_ce || !d_ps || !d_Wc || !stats || B < 1 || Cn < 1)
    lr_fail(LRNDE_EINVAL, "lrnde_classifier_grad: bad args");
  LR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int D = m->D;
  const size_t DB = (size_t)D * B, P = (size_t)m->nparams, PW = (size_t)Cn * (D + 1);
  CallerBufs io(ctx, o->host_buffers);
  const float* psv = io.in(ps, P);
  const float* wcv = io.in(Wc, PW);
  const float* xv = x; const int32_t* yv = labels;
  // host x and labels: the copy lrnde_prefetch_inputs staged on the copy stream (oldest matching slot, waited for
  // through its event), else copied here.  Device x and labels are used in place.
  if (o->host_buffers) {
    if (ctx->pending.valid && ctx->pending.x == x && ctx->pending.y == labels) lr_flush_prefetch(ctx);   // this very batch
    lrnde_ctx::Staged* hit = nullptr;
    for (auto& sg : ctx->staged)
      if (sg.ready && sg.key_x == x && sg.key_y == labels && sg.nx == DB && sg.ny == (size_t)B && (!hit || sg.seq < hit->seq)) hit = &sg;
    if (hit) {
      LR_CUDA(cudaStreamWaitEvent(st, hit->ev, 0));
      xv = hit->x; yv = hit->y;
      hit->ready = false;   // consumed: this call synchronises before returning, so the slot is free afterwards
    } else {
      xv = io.in(x, DB);
      yv = io.in(labels, (size_t)B);
    }
    lr_flush_prefetch(ctx);   // the next batch's copy, queued behind this call's own host -> device copies
  }
  float* dpsv = io.out(d_ps, P);
  float* dwv = io.out(d_Wc, PW);
  DevBuf ud(ctx, DB), dud(ctx, DB);
  const bool timing = getenv("LRNDE_TIMING") != nullptr;
  long tmark = lr_now_us();
  auto mark = [&](const char* what) {
    if (!timing) return;
    cudaStreamSynchronize(st);
    const long now = lr_now_us();
    fprintf(stderr, "[lrnde] classifier_grad %-10s %8ld us\n", what, now - tmark);
    tmark = now;
  };
  mark("stage in");
  lrnde_opts od = *o;
  od.host_buffers = 0; od.keep_tape = 1; od.last_only = 1; od.no_dx = 1;
  lrnde_tape* T = nullptr;
  lrnde_stats s1, s2;
  memset(&s2, 0, sizeof(s2));
  int rc = lrnde_ode_forward(ctx, m, &od, psv, xv, B, ud.p, 1, nullptr, &s1, &T);
  mark("forward");
  if (rc == LRNDE_OK) rc = lrnde_head_ce(ctx, wcv, ud.p, yv, B, D, Cn, 0, loss_ce, dud.p, dwv);
  mark("head");
  if (rc == LRNDE_OK && grad_scale != 1.0f) {
    scale_kernel<<<lr_ew_blocks(DB), 256, 0, st>>>(dud.p, grad_scale, DB);
    scale_kernel<<<lr_ew_blocks(PW), 256, 0, st>>>(dwv, grad_scale, PW);
    LR_COUNT(ctx); LR_COUNT(ctx);
  }
  if (rc == LRNDE_OK) rc = lrnde_ode_backward(ctx, m, T, dud.p, w_reg, dpsv, nullptr, &s2);
  mark("backward");
  if (T) lrnde_tape_free(T);
  if (rc != LRNDE_OK) throw LrError(rc);   // the failing call already set the error text
  io.finish();
  LR_CUDA(cudaStreamSynchronize(st));
  mark("stage out");
  *stats = s1;
  stats->nf_bwd = s2.nf_bwd; stats->naccept_bwd = s2.naccept_bwd; stats->nreject_bwd = s2.nreject_bwd;
  stats->retcode_bwd = s2.retcode_bwd;
  stats->gpu_launches = s1.gpu_launches + s2.gpu_launches + 8;
  stats->reserved[3] = s2.reserved[3]; stats->reserved[4] = s2.reserved[4];
  LR_API_END
}

#include "lrnde_extra.cuh"
#include "lrnde_sde.cuh"
#include "lrnde_latent.cuh"
#include "lrnde_conv_ops.cuh"
