// CPU build of the scalar step-size logic (lrnde_controller.h) and of the save plan
// (lrnde_saveplan.h) for the no-GPU test-suite.
// Not part of the product path: libLRNDE.so runs the same functions inside its controller
// kernels and its forward call; this library only lets pytest compare them with the oracle.
#include "lrnde_controller.h"
#include "lrnde_saveplan.h"

extern "C" {

float lrhc_fastpow(float x, float y, int mode) { return lr_fastpow(x, y, mode); }
float lrhc_spacing(float x) { return lr_spacing(x); }
void lrhc_interp_weights(float theta, float* b) { lr_tsit5_interp(theta, b); }
float lrhc_tsit5_a(int row, int i) { return lr_tsit5_a(row, i); }
float lrhc_tsit5_c(int row) { return lr_tsit5_c(row); }
float lrhc_tsit5_btilde(int i) { return lr_tsit5_btilde(i); }
int lrhc_locate(const float* ts, int nsteps, int tdir, float tval) {
  return lr_locate(ts, nsteps, tdir, tval);
}
float lrhc_initdt(float d0, float d1, float d2_rms_of, int f_equal, float dtmax, float dtmin,
                  int tdir, float* dt0_out) {
  float dt0 = lr_initdt_a(d0, d1, dtmax, tdir);
  if (dt0_out) *dt0_out = dt0;
  return lr_initdt_b(dt0, d1, d2_rms_of, f_equal, dtmax, dtmin, tdir);
}

// Replays a whole controller trajectory: given the EEst the solver measured at every attempt,
// reproduces (t, dt, accepted) of every attempt.  Returns the number of attempts consumed.
int lrhc_replay(float t0, float tend, const float* tstops, int nstops, float dt0, float dtmin,
                int maxiters, int pow_mode, const float* eest, int n_eest, float* t_out,
                float* dt_out, unsigned char* acc_out, int* retcode) {
  LrCtrl c;
  lr_ctrl_init(c, t0, tend, dt0, dtmin, maxiters, pow_mode);
  int k = 0;
  for (int s = 0; s <= nstops; ++s) {
    c.tstop = (s < nstops) ? tstops[s] : tend;
    while (lr_ctrl_header(c, 0)) {
      if (k >= n_eest) { *retcode = -1; return k; }
      t_out[k] = c.t;
      dt_out[k] = c.dt;
      float taken;
      acc_out[k] = (unsigned char)lr_ctrl_footer(c, eest[k], &taken);
      ++k;
    }
    if (c.retcode != LR_RET_SUCCESS) break;
  }
  *retcode = c.retcode;
  return k;
}

// The save plan of a forward call (lrnde_saveplan.h) whose solve accepted the times fts[0..nfts-1].  Writes up to cap
// times and output blocks, t1 and the number of output blocks; returns the number of times.
int lrhc_save_plan(int reg_mode, float t0, float t2, float t1, float u01, const float* saveat, int nsave,
                   int save_start, int last_only, const float* fts, int nfts, float* times, int* out, int cap,
                   float* t1_out, int* nout) {
  lrnde_opts o;
  memset(&o, 0, sizeof(o));
  o.reg_mode = reg_mode; o.t0 = t0; o.t2 = t2; o.t1 = t1; o.u01 = u01;
  o.saveat = saveat; o.nsave = nsave; o.save_start = save_start; o.last_only = last_only;
  const SavePlan p = lr_save_plan(o, std::vector<float>(fts, fts + nfts));
  for (int i = 0; i < (int)p.times.size() && i < cap; ++i) { times[i] = p.times[i]; out[i] = p.out[i]; }
  *t1_out = p.t1;
  *nout = p.nout;
  return (int)p.times.size();
}
}
