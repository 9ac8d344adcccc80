// wave.cuh — kernel W: the warp-per-voice back-end.  One warp owns one voice and walks its timeline in blocks of
// (up to) 32 frames, lane = frame.  Within a block
//   * every linear time-invariant recurrence (one-poles, all-pass sections of the half-band oversampler, TPT / Chamberlin
//     state-variable filters, RBJ biquads, DC blocker) is evaluated as a Kogge-Stone prefix scan over the lanes:
//     y[n] = a y[n-1] + b[n] for scalars, s[n] = M s[n-1] + f[n] over 2x2 state matrices for second-order sections;
//   * every memoryless stage between them (tanh waveshaping at 4x rate, gain compensation, sine lookups of phase-
//     modulated oscillators, mixes) is plain SIMT work, one frame per lane;
//   * the few genuinely nonlinear / integer recurrences (xorshift RNGs, f32 phase accumulators, the envelope follower's
//     data-dependent coefficient, the hi-hat's asymmetric smoother) are replayed in the reference's exact operation order
//     over the block (a handful of instructions per frame; every lane runs the same loop and keeps its own frame).
// This turns the serial tail that bounds kernel C (1024 voices = 32 warps on 148 SMs, IPC 0.19) into 1024 warps of mostly
// data-parallel work.  Scans re-associate the f32 sums, so W is not bit-identical to the per-sample order (C / S are);
// the difference is the rounding noise of the recurrence itself (measured <= 3e-6 through the 4x oversampler at drive 40),
// inside the 1e-5 parity bar.  State is the same Aud struct the serial paths use, so calls can alternate between them.
//
// One voice per whole warp.  Splitting a warp into groups of 16 or 8 lanes, one voice each, cuts the replay cost per
// voice-frame but also the warp count; measured on B200 (C2, r1): 32 lanes -> 82 ms / step, 16 -> 105 ms, 8 -> 150 ms.
// These kernels are bound by the dependent-issue latency of each warp's timeline, not by issue slots.
#pragma once
#include "kernels.cuh"

namespace gd { namespace wave {

// Warp-wide cross-lane operations (coop.cuh uses them too).
__device__ __forceinline__ float shup(float v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }
__device__ __forceinline__ float shl(float v, int n) { return __shfl_sync(0xffffffffu, v, n); }
__device__ __forceinline__ bool gall(bool p) { return __all_sync(0xffffffffu, p); }
__device__ __forceinline__ unsigned gballot(bool p) { return __ballot_sync(0xffffffffu, p); }
__device__ __forceinline__ void gsync() { __syncwarp(); }

// ---- first-order scans -----------------------------------------------------------------------------------
// Per-lane constants of the recurrence y[n] = a y[n-1] + b[n] over 32 lanes.
struct Geo1 { float m[5]; float ap; };            // m[i] = lane >= 2^i ? a^(2^i) : 0 ;  ap = a^(lane+1)
// Two frames per lane (64-long sequence, lane holds elements 2l and 2l+1): lane ratio a^2.
struct Geo2 { float a; float m[5]; float ap; };   // m[i] = lane >= 2^i ? (a^2)^(2^i) : 0 ;  ap = (a^2)^lane

__device__ __forceinline__ Geo1 make_geo1(float a, int lane) {
  Geo1 g; float p = a, ap = 1.0f; const int e = lane + 1;
#pragma unroll
  for (int i = 0; i < 5; i++) { g.m[i] = lane >= (1 << i) ? p : 0.0f; if (e & (1 << i)) ap *= p; p *= p; }
  if (e & 32) ap *= p;
  g.ap = ap;
  return g;
}
__device__ __forceinline__ Geo2 make_geo2(float a, int lane) {
  Geo2 g; g.a = a; float p = a * a, ap = 1.0f;
#pragma unroll
  for (int i = 0; i < 5; i++) { g.m[i] = lane >= (1 << i) ? p : 0.0f; if (lane & (1 << i)) ap *= p; p *= p; }
  g.ap = ap;
  return g;
}
__device__ __forceinline__ float scan1(float b, const Geo1& g, float y_prev) {
#pragma unroll
  for (int i = 0; i < 5; i++) { float t = shup(b, 1 << i); b = __fmaf_rn(g.m[i], t, b); }
  return __fmaf_rn(g.ap, y_prev, b);
}
__device__ __forceinline__ void scan2(float& b0, float& b1, const Geo2& g, float y_prev, int lane) {
  float B = __fmaf_rn(g.a, b0, b1);
#pragma unroll
  for (int i = 0; i < 5; i++) { float t = shup(B, 1 << i); B = __fmaf_rn(g.m[i], t, B); }
  float yp = shup(B, 1);
  if (lane == 0) yp = 0.0f;
  yp = __fmaf_rn(g.ap, y_prev, yp);
  b0 = __fmaf_rn(g.a, yp, b0);
  b1 = __fmaf_rn(g.a, b0, b1);
}
__device__ __forceinline__ float prev_lane(float v, float carry, int lane) { float t = shup(v, 1); return lane == 0 ? carry : t; }

// Shared-memory table of the per-lane constants that do not depend on the voice.
enum { GT_HB = 0, GT_CLICK = 8, GT_DC = 9, GT_PINK = 10, GT_RING = 13, GT_N1 = 14 };
struct GeoTables {
  float g1[GT_N1][6][32];   // half-band sections at the section's own rate (ratio -c_i), then the fixed one-poles
  float g2[8][7][32];       // the half-band sections over two frames per lane
};
__device__ __forceinline__ void geo_tables_init(GeoTables& T, const RateCtx& rc, int tid, int nthreads) {
  for (int idx = tid; idx < GT_N1 * 32; idx += nthreads) {
    const int i = idx >> 5, lane = idx & 31;
    float ratio;
    if (i < 8) ratio = -c_hb[i];
    else if (i == GT_CLICK) ratio = 1.0f - rc.click_alpha;
    else if (i == GT_DC) ratio = 0.995f;
    else if (i == GT_PINK) ratio = rc.pink.p0;
    else if (i == GT_PINK + 1) ratio = rc.pink.p1;
    else if (i == GT_PINK + 2) ratio = rc.pink.p2;
    else ratio = 0.999f;
    const Geo1 a = make_geo1(ratio, lane);
#pragma unroll
    for (int k = 0; k < 5; k++) T.g1[i][k][lane] = a.m[k];
    T.g1[i][5][lane] = a.ap;
    if (i < 8) {
      const Geo2 b = make_geo2(ratio, lane);
#pragma unroll
      for (int k = 0; k < 5; k++) T.g2[i][1 + k][lane] = b.m[k];
      T.g2[i][0][lane] = b.a; T.g2[i][6][lane] = b.ap;
    }
  }
}
__device__ __forceinline__ Geo1 load_geo1(const GeoTables& T, int i, int lane) {
  Geo1 g;
#pragma unroll
  for (int k = 0; k < 5; k++) g.m[k] = T.g1[i][k][lane];
  g.ap = T.g1[i][5][lane];
  return g;
}
__device__ __forceinline__ Geo2 load_geo2(const GeoTables& T, int i, int lane) {
  Geo2 g; g.a = T.g2[i][0][lane];
#pragma unroll
  for (int k = 0; k < 5; k++) g.m[k] = T.g2[i][1 + k][lane];
  g.ap = T.g2[i][6][lane];
  return g;
}

// One all-pass section y[n] = c (x[n] - y[n-1]) + x[n-1] (dsp.cuh hb_run) over a block; (xs, ys) = section state.
__device__ __forceinline__ float ap_sec1(float x, float c, const Geo1& g, float& xs, float& ys, int lane, int last) {
  const float xp = prev_lane(x, xs, lane);
  const float y = scan1(__fmaf_rn(c, x, xp), g, ys);
  xs = shl(x, last); ys = shl(y, last);
  return y;
}
// two frames per lane; `last` = last valid lane, both of its frames valid
__device__ __forceinline__ void ap_sec2(float& x0, float& x1, float c, const Geo2& g, float& xs, float& ys, int lane, int last) {
  const float xp = prev_lane(x1, xs, lane);
  float b0 = __fmaf_rn(c, x0, xp), b1 = __fmaf_rn(c, x1, x0);
  const float nx = shl(x1, last);
  scan2(b0, b1, g, ys, lane);
  xs = nx; ys = shl(b1, last);
  x0 = b0; x1 = b1;
}
// hb_run over a block at the stage's own rate: path 0 through coefficients 0,2,4,6, path 1 through 1,3,5,7
__device__ __forceinline__ void hb_run1(Hb8& s, float& p0, float& p1, const GeoTables& T, int lane, int last) {
#pragma unroll
  for (int i = 0; i < 8; i += 2) {
    p0 = ap_sec1(p0, c_hb[i], load_geo1(T, i, lane), s.x[i], s.y[i], lane, last);
    p1 = ap_sec1(p1, c_hb[i + 1], load_geo1(T, i + 1, lane), s.x[i + 1], s.y[i + 1], lane, last);
  }
}
__device__ __forceinline__ void hb_run2(Hb8& s, float& a0, float& a1, float& b0, float& b1, const GeoTables& T, int lane, int last) {
#pragma unroll
  for (int i = 0; i < 8; i += 2) {
    ap_sec2(a0, a1, c_hb[i], load_geo2(T, i, lane), s.x[i], s.y[i], lane, last);
    ap_sec2(b0, b1, c_hb[i + 1], load_geo2(T, i + 1, lane), s.x[i + 1], s.y[i + 1], lane, last);
  }
}
// Oversampler::process over a block (utils/oversampler.rs:38-113; dsp.cuh os_process); f is the memoryless nonlinearity
template <class F> __device__ __forceinline__ float os_scan(Oversamp& o, float in, F f, const GeoTables& T, int lane, int last) {
  if (o.mode == 0) return f(in);
  float s0 = in, s1 = in;
  hb_run1(o.outer_up, s0, s1, T, lane, last);          // 2x stream: s0, s1 per frame
  if (o.mode == 2) {
    float a = f(s1), b = f(s0);
    hb_run1(o.outer_down, a, b, T, lane, last);
    return 0.5f * (a + b);
  }
  float i00 = s0, i01 = s1, i10 = s0, i11 = s1;        // inner_up path 0 / path 1 over the 2x stream
  hb_run2(o.inner_up, i00, i01, i10, i11, T, lane, last);
  // 4x stream per frame: i00, i10, i01, i11.  inner_down takes (second, first) of each pair
  float a0 = f(i10), a1 = f(i11), b0 = f(i00), b1 = f(i01);
  hb_run2(o.inner_down, a0, a1, b0, b1, T, lane, last);
  const float d0 = 0.5f * (a0 + b0), d1 = 0.5f * (a1 + b1);
  float a = d1, b = d0;
  hb_run1(o.outer_down, a, b, T, lane, last);
  return 0.5f * (a + b);
}

// ---- second-order LTI scans: s[n] = M s[n-1] + f[n],  M = [m0 m1; m2 m3] ------------------------------------
struct Lin2 {            // per-warp, in shared memory
  float P[5][4];         // M^(2^i)
  float L[4][32];        // M^(lane+1)
};
__device__ __forceinline__ void mat_mul(const float* a, const float* b, float* c) {
  c[0] = a[0] * b[0] + a[1] * b[2]; c[1] = a[0] * b[1] + a[1] * b[3];
  c[2] = a[2] * b[0] + a[3] * b[2]; c[3] = a[2] * b[1] + a[3] * b[3];
}
__device__ __forceinline__ void lin2_init(Lin2& S, float m0, float m1, float m2, float m3, int lane) {
  float p[4] = {m0, m1, m2, m3}, acc[4] = {1.0f, 0.0f, 0.0f, 1.0f}, t[4];
  const int e = lane + 1;
#pragma unroll
  for (int i = 0; i < 5; i++) {
    if (lane == 0) { S.P[i][0] = p[0]; S.P[i][1] = p[1]; S.P[i][2] = p[2]; S.P[i][3] = p[3]; }
    if (e & (1 << i)) { mat_mul(p, acc, t); acc[0] = t[0]; acc[1] = t[1]; acc[2] = t[2]; acc[3] = t[3]; }
    mat_mul(p, p, t); p[0] = t[0]; p[1] = t[1]; p[2] = t[2]; p[3] = t[3];
  }
  if (e & 32) { mat_mul(p, acc, t); acc[0] = t[0]; acc[1] = t[1]; acc[2] = t[2]; acc[3] = t[3]; }
  S.L[0][lane] = acc[0]; S.L[1][lane] = acc[1]; S.L[2][lane] = acc[2]; S.L[3][lane] = acc[3];
  gsync();
}
// in: forcing (f0, f1) per lane; out: state after each frame.  (s0p, s1p) = state before the block.
__device__ __forceinline__ void lin2_scan(const Lin2& S, float& f0, float& f1, float s0p, float s1p, int lane) {
#pragma unroll
  for (int i = 0; i < 5; i++) {
    const float t0 = shup(f0, 1 << i), t1 = shup(f1, 1 << i);
    if (lane >= (1 << i)) {
      f0 = __fmaf_rn(S.P[i][0], t0, __fmaf_rn(S.P[i][1], t1, f0));
      f1 = __fmaf_rn(S.P[i][2], t0, __fmaf_rn(S.P[i][3], t1, f1));
    }
  }
  f0 = __fmaf_rn(S.L[0][lane], s0p, __fmaf_rn(S.L[1][lane], s1p, f0));
  f1 = __fmaf_rn(S.L[2][lane], s0p, __fmaf_rn(S.L[3][lane], s1p, f1));
}

// Per-warp read-only tables in shared memory (written by span_setup, then only read).
struct WaveScratch { Lin2 lin[3]; float stash[8][32]; };

// The Aud state is held in REGISTERS, replicated in every lane (all lanes compute the same state updates from
// shuffled values), so there are no shared-memory hazards; the exact-order serial sections below are executed by all
// lanes redundantly, which costs the same issue slots as running them on one lane.

// tanh for the memoryless saturators of the scan back end:  1 - 2 / (exp(2|x|) + 1)  through ex2.approx / rcp.approx.
// Absolute error <= 3e-7 (ex2.approx is 2 ulp; |d tanh / d e| <= 1/2), against ~90 instructions of the bit-exact
// fdlibm port (gm::g_tanhf) that the per-sample paths keep.  These stages feed bounded-gain filters only (half-band
// decimators, DC blocker, dry/wet mix), never a recurrence, so the error stays at that level in the output: well inside
// the 1e-5 parity bar (tests/test_voices_gpu.py measures the total).
__device__ __forceinline__ float w_tanh(float x) {
  const float ax = fabsf(x);
  const float e = __expf(2.0f * ax);                       // +inf for large |x| -> t = 1; NaN propagates
  const float t = 1.0f - __fdividef(2.0f, e + 1.0f);
  return copysignf(t, x);
}
// (A sin.approx variant of the hi-hat / tom oscillators was tried and rejected: the tom alone ends 1e-4 away from the
// oracle — its sines are multiplied together and drive the high-Q membrane — for a 3 % gain.)
// FeedbackWaveshaper::gain_compensation (dsp.cuh fbws_gain_comp) with the fast tanh: a gain, relative error 3e-7
__device__ __forceinline__ float w_gain_comp(FbShaper& w, float env) {
  const float reference = fmaxf(env, 0.05f);
  const float driven = fmaxf(fabsf(w_tanh(reference * w.drive)), 1e-6f);
  const float comp_no_fb = w_tanh(reference) / driven;
  const float makeup = fbws_makeup(w);
  const float taming = 1.0f / (1.0f + comp_no_fb * w.feedback * 0.25f);
  return fminf(comp_no_fb * taming * makeup, 3.0f);
}
__device__ __forceinline__ float wrap01(float x) { return x < 1.0f ? x : (x < 2.0f ? x - 1.0f : fmodf(x, 1.0f)); }   // fmodf(x, 1) for x >= 0, exact

// TPT SVF as a linear map of (ic1, ic2) (state_variable_tpt.rs:56-69, resonant_lowpass.rs:49-103):
//   v1 = (g (in - ic2) + ic1) h ; v2 = ic2 + g v1 ; ic1' = 2 v1 - ic1 ; ic2' = 2 v2 - ic2
struct TptLin { float in0, in1; };
__device__ __forceinline__ TptLin tpt_lin_init(Lin2& S, const Tpt& f, int lane) {
  const float g = f.g, h = f.h, gh = g * h, g2h = g * gh;
  lin2_init(S, 2.0f * h - 1.0f, -2.0f * gh, 2.0f * gh, 1.0f - 2.0f * g2h, lane);
  TptLin t; t.in0 = 2.0f * gh; t.in1 = 2.0f * g2h;
  return t;
}
// runs the filter over the block; returns this lane's PRE-state so the caller can form the outputs exactly as the
// serial code does from it
__device__ __forceinline__ void tpt_scan(const Lin2& S, const TptLin& t, Tpt& f, float in, float& ic1_pre, float& ic2_pre, int lane, int last) {
  float s0 = t.in0 * in, s1 = t.in1 * in;
  lin2_scan(S, s0, s1, f.ic1, f.ic2, lane);
  ic1_pre = prev_lane(s0, f.ic1, lane); ic2_pre = prev_lane(s1, f.ic2, lane);
  f.ic1 = shl(s0, last); f.ic2 = shl(s1, last);
}
// RBJ biquad, direct form I (dsp.cuh biquad_process): y[n] = b0 x[n] + b1 x[n-1] + b2 x[n-2] - a1 y[n-1] - a2 y[n-2]
__device__ __forceinline__ void biquad_lin_init(Lin2& S, const Biquad& b, int lane) { lin2_init(S, -b.a1, -b.a2, 1.0f, 0.0f, lane); }
__device__ __forceinline__ float biquad_scan(const Lin2& S, Biquad& b, float x, int lane, int last) {
  const float xm1 = prev_lane(x, b.x1, lane);
  float xm2 = shup(x, 2);
  xm2 = lane == 0 ? b.x2 : (lane == 1 ? b.x1 : xm2);
  float f0 = b.b0 * x + b.b1 * xm1 + b.b2 * xm2, f1 = 0.0f;
  lin2_scan(S, f0, f1, b.y1, b.y2, lane);
  const float nx1 = shl(x, last), nx2 = shl(xm1, last);
  const float ny1 = shl(f0, last), ny2 = shl(f1, last);
  b.x1 = nx1; b.x2 = nx2; b.y1 = ny1; b.y2 = ny2;
  return fabsf(f0) < 1e-15f ? 0.0f : f0;
}

// Replay helper: value of `v` held by lane n, for a loop index n that is uniform across the warp.
#define LANE_VAL(v, n) shl((v), (n))
// Replay loops read the block's per-frame inputs from shared memory instead of shuffling them out of lane n: a uniform
// LDS has no convergence requirement, so ptxas may hoist it across iterations, whereas a SHFL inside a loop with a
// data-dependent branch is fenced by BSSY / BRA.DIV / BSYNC and exposes its ~25-cycle latency on every iteration
// (ncu source page, r1_h: the tom band-pass replay spent its stalls on the FMUL that consumes the shuffled sample).
#define STASH_PUT(slot, v) (sc.stash[slot][lane] = (v))
#define STASH_GET(slot, n) (sc.stash[slot][n])

// ---- kick ------------------------------------------------------------------------------------------------
struct KickW {
  using V = KickV;
  struct Span2 { bool noise, shaper, serial; };
  static __device__ __forceinline__ int active_end(const KickV::Run& r) { return r.j_act; }
  static __device__ __forceinline__ void span_setup(KickAud& a, const KickV::Run& r, Span2& w, WaveScratch&, const RateCtx& rc, int) {
    w.noise = r.d.noise_amount > 0.001f;
    a.ws.drive = r.d.drive; a.ws.feedback = r.d.feedback;
    fbws_set_cutoff(a.ws, rc.sr, r.d.fb_cutoff);
    w.shaper = !(a.ws.mix <= 0.0001f || a.ws.drive <= 1.0f);
    w.serial = w.shaper && a.ws.feedback != 0.0f;     // tanh inside the feedback loop: no scan (feedback_waveshaper.rs:122-159)
    if (w.noise) rlp_set(a.noise_lp, rc.sr, r.d.noise_cut, r.d.noise_res);
  }
  // one block: lanes [0, nl) hold frames j .. j+nl-1.  p[] = this lane's front planes.  Returns the output sample.
  static __device__ __forceinline__ float block(KickAud& a, const KickV::Run& r, const Span2& w, WaveScratch& sc, const GeoTables& T,
                                                const float* p, int, int& nl, const RateCtx& rc, int lane) {
    const int last = nl - 1;
    const float p1 = p[0], raw_click = p[1], ne = p[2], amp = p[3];
    // click high-pass and the pink-noise layer: cheap recurrences, replayed in the reference's order (kick.rs:1171-1193)
    float hp_l = 0.0f, fn_l = 0.0f;
    gsync(); STASH_PUT(0, raw_click); gsync();
#pragma unroll 4
    for (int n = 0; n < nl; n++) {
      const float raw = STASH_GET(0, n);
      const float hp = raw - a.click_hp;
      a.click_hp += rc.click_alpha * hp;
      float fn = 0.0f;
      if (w.noise) fn = rlp_process(a.noise_lp, pink_tick(a.pink, rc.pink));
      if (n == lane) { hp_l = hp; fn_l = fn; }
    }
    const float filt_click = hp_l * (1.0f + 4.0f * 0.1f);
    const float noise_out = w.noise ? fn_l * ne * r.d.noise_amount * 0.5f : 0.0f;
    const float total = p1 + filt_click + noise_out;
    float od = total;
    const bool finite = gall(isfinite(total));
    if (w.serial || (w.shaper && !finite)) {       // feedback > 0 (or a non-finite input): the reference's per-sample order
#pragma unroll 4
      for (int n = 0; n < nl; n++) {
        const float y = fbws_process(a.ws, LANE_VAL(total, n));
        if (n == lane) od = y;
      }
    } else if (w.shaper) {
      FbShaper& ws = a.ws;
      const float fb_in = ws.drive * total + ws.feedback * ws.last_out;   // feedback == 0
      const float shaped = os_scan(ws.os, fb_in, [](float x) { return w_tanh(x); }, T, lane, last);
      // envelope follower: the coefficient depends on a comparison with the running state -> replay
      const float rect_l = fabsf(total);
      float env_l = 0.0f;
      gsync(); STASH_PUT(1, rect_l); gsync();
#pragma unroll 4
      for (int n = 0; n < nl; n++) {
        const float rect = STASH_GET(1, n);
        const float coeff = rect > ws.env ? ws.env_att : ws.env_rel;
        ws.env += (1.0f - coeff) * (rect - ws.env);
        if (fabsf(ws.env) < 1e-15f) ws.env = 0.0f;
        if (n == lane) env_l = ws.env;
      }
      const float comp = w_gain_comp(ws, env_l);
      const float compensated = shaped * comp;
      // DC blocker and the one-pole that feeds last_out (feedback_waveshaper.rs:262-271, 151-159): replay
      float out_l = 0.0f;
      gsync(); STASH_PUT(2, compensated); gsync();
#pragma unroll 4
      for (int n = 0; n < nl; n++) {
        const float c = STASH_GET(2, n);
        const float out = c - ws.dc_x1 + 0.995f * ws.dc_y1;
        ws.dc_x1 = c;
        ws.dc_y1 = fabsf(out) < 1e-15f ? 0.0f : out;
        ws.filter_state += ws.filter_coeff * (out - ws.filter_state);
        if (fabsf(ws.filter_state) < 1e-15f) ws.filter_state = 0.0f;
        if (n == lane) out_l = out;
      }
      ws.last_out = ws.filter_state;
      od = total * (1.0f - ws.mix) + out_l * ws.mix;
    }
    return od * amp * r.d.va * r.d.volume;
  }
};

// ---- snare -----------------------------------------------------------------------------------------------
struct SnareW {
  using V = SnareV;
  struct Span2 { float comp; bool shaper; };
  static __device__ __forceinline__ int active_end(const SnareV::Run& r) { return r.j_act; }
  static __device__ __forceinline__ void span_setup(SnareAud& a, const SnareV::Run& r, Span2& w, WaveScratch&, const RateCtx& rc, int) {
    chamb_set(a.filt, rc.sr, r.d.cutoff, r.d.res);
    a.ws.drive = r.d.drive;
    w.shaper = !(a.ws.mix <= 0.0001f || a.ws.drive <= 1.0f);
    w.comp = w.shaper ? gm::g_tanhf(0.5f) / gm::g_tanhf(0.5f * a.ws.drive) : 1.0f;
  }
  static __device__ __forceinline__ float block(SnareAud& a, const SnareV::Run& r, const Span2& w, WaveScratch& sc, const GeoTables& T,
                                                const float* p, int, int& nl, const RateCtx&, int lane) {
    const int last = nl - 1;
    const float tonal_out = p[0], raw_noise = p[1], cne = p[2], crack_out = p[3], amp = p[4];
    // Chamberlin SVF: replayed exactly (it is unstable for high cutoff x low resonance, and the reference's
    // blow-up -> NaN -> Waveshaper guard -> 0 sequence has to be reproduced sample for sample)
    float low_l = 0.0f, band_l = 0.0f, high_l = 0.0f;
    {
      const float f = a.filt.f, q = a.filt.q;
      float low = a.filt.low, band = a.filt.band;
      gsync(); STASH_PUT(0, raw_noise); gsync();
#pragma unroll 4
      for (int n = 0; n < nl; n++) {
        const float in = STASH_GET(0, n);
        float high = 0.0f;
#pragma unroll
        for (int i = 0; i < 2; i++) { low = low + f * band; high = in - low - q * band; band = f * high + band; }
        if (n == lane) { low_l = low; band_l = band; high_l = high; }
      }
      a.filt.low = low; a.filt.band = band;
    }
    const float filtered = svf_pick(low_l, band_l, high_l, r.d.filter_type);
    const float noise_out = filtered * cne * r.d.noise_mix;
    const float total = tonal_out + noise_out + crack_out;
    float od = total;
    const bool finite = gall(isfinite(total));
    if (!finite) {          // waveshaper.rs:49-53 resets its oversampler on a non-finite input: per-sample order
#pragma unroll 4
      for (int n = 0; n < nl; n++) {
        const float y = ws_process(a.ws, LANE_VAL(total, n));
        if (n == lane) od = y;
      }
    } else if (w.shaper) {
      const float d = a.ws.drive, comp = w.comp;
      const float sat = os_scan(a.ws.os, total, [d, comp](float x) { return w_tanh(x * d) * comp; }, T, lane, last);
      od = total * (1.0f - a.ws.mix) + sat * a.ws.mix;
    }
    return od * amp * r.d.va * r.d.volume;
  }
};

// ---- hi-hat ----------------------------------------------------------------------------------------------
struct HatW {
  using V = HatV;
  struct Span2 { TptLin svf; };
  static __device__ __forceinline__ int active_end(const HatV::Run&) { return 0x7fffffff; }
  static __device__ __forceinline__ void span_setup(HatAud& a, const HatV::Run& r, Span2& w, WaveScratch& sc, const RateCtx& rc, int lane) {
    hp_set(a.hp1, rc.sr, r.d.pitch_hz, 1.0f);
    biquad_lin_init(sc.lin[0], a.hp1, lane);
    if (r.d.db24) { hp_set(a.hp2, rc.sr, r.d.pitch_hz, 1.0f); biquad_lin_init(sc.lin[1], a.hp2, lane); }
    tpt_set(a.svf, rc.sr, r.d.tone_hz, 0.5f);
    w.svf = tpt_lin_init(sc.lin[2], a.svf, lane);
  }
  // j = frame of lane 0.  May shorten nl when the voice deactivates inside the block (frames after it are silent).
  static __device__ __forceinline__ float block(HatAud& a, const HatV::Run& r, const Span2& w, WaveScratch& sc, const GeoTables&,
                                                const float* p, int j, int& nl, const RateCtx& rc, int lane) {
    const float sr = rc.sr;
    // envelope through the asymmetric smoother and the deactivation test (hihat2.rs:489-506): replay
    const float env_l = (j + lane) < r.j_env ? p[0] : r.env_final;
    float es_l = 0.0f;
    int nv = nl;
    gsync(); STASH_PUT(0, env_l); gsync();
    if (j + nl <= r.j_env) {     // the envelope is still running through the whole block: the voice cannot deactivate here
#pragma unroll 4
      for (int n = 0; n < nl; n++) {
        const float e = STASH_GET(0, n);
        if (e >= a.env_smooth) a.env_smooth = e; else a.env_smooth += rc.asym_down * (e - a.env_smooth);
        if (n == lane) es_l = a.env_smooth;
      }
    } else {
#pragma unroll 4
      for (int n = 0; n < nl; n++) {
        const float e = STASH_GET(0, n);
        if (e >= a.env_smooth) a.env_smooth = e; else a.env_smooth += rc.asym_down * (e - a.env_smooth);
        if (n == lane) es_l = a.env_smooth;
        if ((j + n) >= r.j_env && a.env_smooth < 1e-4f) { nv = n + 1; a.active = 0; break; }
      }
    }
    nl = nv;
    // noise and the two phase accumulators: replay
    float noise = 0.0f, mph = 0.0f, nph = 0.0f;
    const float inc_mod = fmaxf(r.d.pitch_hz * 0.1f, 0.0f) / sr, inc_main = fmaxf(r.d.pitch_hz, 0.0f) / sr;
    // fmodf(x, 1) of x = phase + inc with phase in [0, 1) and inc < 1 is x or x - 1 (exact): no fmodf path needed then
    const bool small_inc = inc_main < 1.0f && a.mod_phase < 1.0f && a.main_phase < 1.0f;
    if (!r.d.pink_on && small_inc) {
      // white noise: only the xorshift state is a recurrence; its multiply / conversion happens once per lane afterwards
      uint64_t st_l = 0;
#pragma unroll 4
      for (int n = 0; n < nv; n++) {
        uint64_t x = a.white;
        x ^= x >> 12; x ^= x << 25; x ^= x >> 27;
        a.white = x;
        float pm = a.mod_phase + inc_mod; a.mod_phase = pm < 1.0f ? pm : pm - 1.0f;
        float pn = a.main_phase + inc_main; a.main_phase = pn < 1.0f ? pn : pn - 1.0f;
        if (n == lane) { st_l = x; mph = a.mod_phase; nph = a.main_phase; }
      }
      const float u = u64_to_f32(st_l * 0x2545f4914f6cdd1dull) / 18446744073709551616.0f;
      noise = (u * 2.0f) - 1.0f;
    } else {
#pragma unroll 4
      for (int n = 0; n < nv; n++) {
        float x;
        if (r.d.pink_on) x = pink_tick(a.pink, rc.pink);
        else { float u = u64_to_f32(xorshift64s_next(a.white)) / 18446744073709551616.0f; x = (u * 2.0f) - 1.0f; }
        a.mod_phase = wrap01(a.mod_phase + inc_mod);
        a.main_phase = wrap01(a.main_phase + inc_main);
        if (n == lane) { noise = x; mph = a.mod_phase; nph = a.main_phase; }
      }
    }
    // PhaseModOsc outputs are memoryless given the phases (hihat2.rs:277-286): one frame per lane
    float ph = mph + noise * 0.25f; ph -= floorf(ph);
    const float mod_out = gm::g_sinf(2.0f * PI_F * ph);
    ph = nph + mod_out * 0.75f; ph -= floorf(ph);
    const float main_out = gm::g_sinf(2.0f * PI_F * ph);
    // two RBJ high-passes (Q = 1), envelope, TPT high-pass (Q = 0.5): well damped LTI sections -> 2x2 scans
    const int last = nv - 1;
    float filtered = biquad_scan(sc.lin[0], a.hp1, main_out, lane, last);
    if (r.d.db24) filtered = biquad_scan(sc.lin[1], a.hp2, filtered, lane, last) * 0.8f;
    const float out = filtered * es_l * r.d.vel035 * 0.35f;
    float ic1p, ic2p;
    tpt_scan(sc.lin[2], w.svf, a.svf, out, ic1p, ic2p, lane, last);
    const float v1 = (a.svf.g * (out - ic2p) + ic1p) * a.svf.h;
    const float v2 = ic2p + a.svf.g * v1;
    const float hi = out - (a.svf.r * v1 + v2);
    return hi * r.d.volume;
  }
};

// ---- tom -------------------------------------------------------------------------------------------------
// A block of the tom (tom2.rs:450-585) is cut by what depends on history:
//   * the three f32 phase accumulators, the rand~ sample-and-hold and the band-pass's coefficient-change detector
//     (biquad_bandpass.rs:73-87, a chain through last_freq only) are replayed in the reference's order; the detector
//     leaves the block's UPDATE MASK;
//   * sines / triangles / morph mix and the band-pass coefficient sets of the frames that update are per-lane work; every
//     lane picks the set in effect at its frame and forms the FEED-FORWARD half of the direct-form-I section,
//     (b0 x[n] + b1 x[n-1]) + b2 x[n-2] — inputs only, same operation order as biquad_process;
//   * only the FEEDBACK half, out = (ffwd - a1 y1) - a2 y2, is replayed (4 flops per frame instead of the whole section with
//     its coefficient selects); the five membrane resonators are split the same way and replayed on five lanes at once;
//   * ringing TAIL (main oscillator done, envelope complete, membrane > 0): only membrane / tanh / ring level run.  What the
//     reference keeps ticking there (phases, click, band-pass memory) is reset by the next trigger before it can be
//     observed; the band-pass coefficient memory, which survives a trigger, is brought to where the per-sample bp_set calls
//     would leave it.  Everything else that is done (no membrane but a stale ring level, completion by pitch instead of
//     envelope, foreign phase state) takes the reference's whole tick per frame (generic()).
struct TomW {
  using V = TomV;
  struct Span2 { int dummy; };
  static __device__ __forceinline__ int active_end(const TomV::Run&) { return 0x7fffffff; }
  static __device__ __forceinline__ void span_setup(TomAud&, const TomV::Run&, Span2&, WaveScratch&, const RateCtx&, int) {}
  // the reference's per-sample order over the block (all lanes replicate the state)
  static __device__ __forceinline__ float generic(TomAud& a, const TomV::Run& r, WaveScratch& sc, float env_l, float noise_l, float rnd_l,
                                                  int j, int& nl, const RateCtx& rc, int lane) {
    float y_l = 0.0f;
    int nv = nl;
    gsync(); STASH_PUT(0, env_l); STASH_PUT(1, noise_l); STASH_PUT(2, rnd_l); gsync();
#pragma unroll 2
    for (int n = 0; n < nl; n++) {
      TomFront f; f.env = STASH_GET(0, n); f.noise = STASH_GET(1, n); f.rnd = STASH_GET(2, n);
      const float y = tom_back(a, r.d, f, (j + n) >= r.j_env, rc);
      if (n == lane) y_l = y;
      if (!a.active) { nv = n + 1; break; }
    }
    nl = nv;
    return y_l;
  }
  // membrane resonators over a block whose membrane input is mi_l: feed-forward halves per lane, feedback halves replayed
  // on lanes 0..4 (lane i owns filter i), summed per frame in the reference's order; returns tanh(sum)
  static __device__ __forceinline__ float membrane(TomAud& a, WaveScratch& sc, float mi_l, int nv, int lane) {
    const float u1 = shup(mi_l, 1), u2 = shup(mi_l, 2);
    gsync();
#pragma unroll
    for (int f = 0; f < 5; f++) {
      const Biquad& m = a.mem[f];
      const float xm1 = lane == 0 ? m.x1 : u1, xm2 = lane == 0 ? m.x2 : (lane == 1 ? m.x1 : u2);
      sc.stash[f][lane] = m.b0 * mi_l + m.b1 * xm1 + m.b2 * xm2;
    }
    const float nx1 = shl(mi_l, nv - 1), nx2 = nv >= 2 ? shl(mi_l, nv - 2) : a.mem[0].x1;   // the five filters share their input history
#pragma unroll
    for (int f = 0; f < 5; f++) { a.mem[f].x2 = nv >= 2 ? nx2 : a.mem[f].x1; a.mem[f].x1 = nx1; }
    float a1 = a.mem[4].a1, a2 = a.mem[4].a2, y1 = a.mem[4].y1, y2 = a.mem[4].y2;
#pragma unroll
    for (int f = 0; f < 4; f++) if (lane == f) { a1 = a.mem[f].a1; a2 = a.mem[f].a2; y1 = a.mem[f].y1; y2 = a.mem[f].y2; }
    const int row = lane < 5 ? lane : 4;
    gsync();
#pragma unroll 4
    for (int n = 0; n < nv; n++) {
      const float out = sc.stash[row][n] - a1 * y1 - a2 * y2;
      y2 = y1; y1 = out;
      if (lane < 5) sc.stash[row][n] = fabsf(out) < 1e-15f ? 0.0f : out;
    }
    gsync();
    float acc = 0.0f;
#pragma unroll
    for (int i = 0; i < 5; i++) acc += sc.stash[i][lane];
#pragma unroll
    for (int i = 0; i < 5; i++) { a.mem[i].y1 = shl(y1, i); a.mem[i].y2 = shl(y2, i); }
    return w_tanh(acc);
  }
  static __device__ __forceinline__ float block(TomAud& a, const TomV::Run& r, const Span2&, WaveScratch& sc, const GeoTables&,
                                                const float* p, int j, int& nl, const RateCtx& rc, int lane) {
    const TomDer& d = r.d;
    const float sr = rc.sr;
    const float env_l = (j + lane) < r.j_env ? p[0] : r.env_final;
    const float noise_l = p[1], rnd_l = p[2];
    const bool complete_l = (j + lane) >= r.j_env;
    const unsigned valid = nl >= 32 ? 0xffffffffu : ((1u << nl) - 1u);
    const unsigned le = (2u << lane) - 1u;     // lanes 0..lane
    // pure per-frame quantities (tom2.rs:455-489)
    const float eb = env_l * d.bend_scaled;
    const float raw_freq = d.base_frequency * (1.0f + eb * eb);
    const unsigned m_att = gballot(env_l > 0.9f) & valid;
    const bool past_l = a.past_attack || (m_att & le) != 0u;
    const unsigned m_done = gballot(complete_l || (past_l && raw_freq < 20.0f)) & valid;
    const int first_done = a.main_done ? 0 : (m_done ? __ffs(m_done) - 1 : 32);
    const bool merged = a.tri_phase == a.main_sine_phase && a.tri_phase == a.mtri_phase && a.tri_phase == a.gated_sine_phase;
    if (first_done == 0) {
      if (d.membrane > 0.0f && j >= r.j_env) {
        // ---- ringing tail ----
        a.main_done = 1;
        const float eb0 = r.env_final * d.bend_scaled;
        bp_set(a.bp, sr, fmaxf(fmaxf(d.base_frequency * (1.0f + eb0 * eb0), 40.0f), 20.0f), d.fq, 1.1f);
        const float clipped = membrane(a, sc, 0.0f, nl, lane);
        gsync(); STASH_PUT(5, fabsf(clipped) * 0.001f); gsync();
        float lev_l = 0.0f;
        int nv = nl;
        for (int n = 0; n < nl; n++) {
          if (!(a.ring_level > 0.0001f)) { nv = n; a.active = 0; break; }      // tom2.rs:488-493, tested before the frame's membrane tick
          a.ring_level = a.ring_level * 0.999f + STASH_GET(5, n);
          if (n == lane) lev_l = a.ring_level;
        }
        nl = nv;
        const float fd = lev_l >= 0.005f ? 1.0f : (lev_l <= 0.0001f ? 0.0f : (lev_l - 0.0001f) / (0.005f - 0.0001f));
        return clipped * d.mm * fd * 0.7f * d.vol;
      }
      if (!(d.membrane > 0.0f) && !(a.ring_level > 0.0001f)) {   // no tail: the voice ends at this frame
        a.main_done = 1; a.active = 0; if (m_att & 1u) a.past_attack = 1;
        nl = 0;
        return 0.0f;
      }
      return generic(a, r, sc, env_l, noise_l, rnd_l, j, nl, rc, lane);
    }
    if (!merged) return generic(a, r, sc, env_l, noise_l, rnd_l, j, nl, rc, lane);
    // ---- main oscillator running over frames [0, nv); a block that ends at its last frame is followed by a tail block ----
    const int nv = first_done < nl ? first_done : nl;
    a.past_attack = a.past_attack || (m_att & (nv >= 32 ? 0xffffffffu : ((1u << nv) - 1u))) != 0u;
    nl = nv;
    const float fade = (past_l && raw_freq < 40.0f) ? (raw_freq - 20.0f) / (40.0f - 20.0f) : 1.0f;
    const float mf_l = fmaxf(raw_freq, 40.0f);
    float click = 0.0f;
    if (a.click_playing) {
      const uint32_t idx = a.click_pos + (uint32_t)lane;
      if (idx < 64u) click = c_tom_impulse[idx];
      a.click_pos = min(64u, a.click_pos + (uint32_t)nv);
      if (a.click_pos >= 64u) a.click_playing = 0;
    }
    const float ff_l = fmaxf(mf_l, 20.0f);
    // phase accumulators, rand~ sample-and-hold, coefficient-change detector: replay (morph_osc.rs:137-202, biquad_bandpass.rs:73-87)
    const float inc_fixed = 190.0f / sr, inc_rand = d.rand_freq / sr;
    gsync(); STASH_PUT(0, mf_l / sr); STASH_PUT(1, rnd_l); STASH_PUT(2, ff_l); gsync();
    unsigned mask = 0u;
    {
      float ph = a.tri_phase, fx = a.fixed_sine_phase, rph = a.rand_phase, rcu = a.rand_current, rtg = a.rand_target, lf = a.bp.last_freq;
      bool qg_ok = fabsf(d.fq - a.bp.last_q) < 0.001f && fabsf(1.1f - a.bp.last_gain) < 0.001f;   // an update makes both terms true
#pragma unroll 4
      for (int n = 0; n < nv; n++) {
        const float inc = STASH_GET(0, n), rnd = STASH_GET(1, n), ffn = STASH_GET(2, n);
        sc.stash[3][n] = ph; sc.stash[4][n] = fx;
        ph += inc; if (ph >= 1.0f) ph -= 1.0f;
        fx += inc_fixed; if (fx >= 1.0f) fx -= 1.0f;
        const float prev = rph;
        rph += inc_rand; if (rph >= 1.0f) rph -= 1.0f;
        const bool wrap = rph < prev;
        rcu = wrap ? rtg : rcu; rtg = wrap ? rnd : rtg;
        sc.stash[5][n] = rcu + (rtg - rcu) * rph;
        const bool upd = !(fabsf(ffn - lf) < 0.01f && qg_ok);   // !bp_unchanged
        lf = upd ? ffn : lf; qg_ok = qg_ok || upd;
        mask |= upd ? (1u << n) : 0u;
      }
      a.tri_phase = a.main_sine_phase = a.mtri_phase = a.gated_sine_phase = ph;
      a.fixed_sine_phase = fx; a.rand_phase = rph; a.rand_current = rcu; a.rand_target = rtg;
      a.bp.last_freq = lf;
      if (mask) { a.bp.last_q = d.fq; a.bp.last_gain = 1.1f; }
    }
    gsync();
    const float tp = sc.stash[3][lane], fsp = sc.stash[4][lane], rand_value = sc.stash[5][lane];
    const float click_out = click * 1.1f;
    const float tri_out = a.tri_enabled ? tri_wave(tp) * 0.5f : 0.0f;
    const float us = unit_sine(tp);
    const float main_sine = us * 0.5f;
    const float mtri = tri_wave(tp) * 0.5f;
    const float fixed_sine = unit_sine(fsp) * 0.5f;
    const float noise = noise_l * 0.2f;
    const float noise_combined = (noise + rand_value) * 0.4f;
    const float gated = d.tone < 99.0f ? us * 0.2f : 0.0f;
    const float ch1 = main_sine * fixed_sine, ch2 = mtri + noise_combined, ch3 = noise_combined + gated;
    const float morph_out = ch1 * d.w1 + ch2 * d.w2 + ch3 * d.w3;
    const float x = click_out + tri_out + morph_out;
    // band-pass: coefficient set in effect at this frame = the set of the latest update frame <= lane, else the carried one
    float b0 = a.bp.b0, b1 = a.bp.b1, b2 = a.bp.b2, a1 = a.bp.a1, a2 = a.bp.a2;
    if (mask) {
      Biquad spec;
      bp_compute(spec, sr, ff_l, d.fq, 1.1f);
      const unsigned m = mask & le;
      const int src = m ? 31 - __clz(m) : 0;
      const float sb0 = shl(spec.b0, src), sb1 = shl(spec.b1, src), sb2 = shl(spec.b2, src), sa1 = shl(spec.a1, src), sa2 = shl(spec.a2, src);
      if (m) { b0 = sb0; b1 = sb1; b2 = sb2; a1 = sa1; a2 = sa2; }
    }
    float xm1 = shup(x, 1), xm2 = shup(x, 2);
    if (lane == 0) { xm1 = a.bp.x1; xm2 = a.bp.x2; } else if (lane == 1) xm2 = a.bp.x1;
    const float ffwd = b0 * x + b1 * xm1 + b2 * xm2;
    gsync(); STASH_PUT(0, ffwd); STASH_PUT(1, a1); STASH_PUT(2, a2); gsync();
    {   // state after the block's last frame
      const int last = nv - 1;
      a.bp.b0 = shl(b0, last); a.bp.b1 = shl(b1, last); a.bp.b2 = shl(b2, last); a.bp.a1 = shl(a1, last); a.bp.a2 = shl(a2, last);
      a.bp.x1 = shl(x, last); a.bp.x2 = shl(xm1, last);
    }
    {
      float y1 = a.bp.y1, y2 = a.bp.y2;
#pragma unroll 4
      for (int n = 0; n < nv; n++) {
        const float out = STASH_GET(0, n) - STASH_GET(1, n) * y1 - STASH_GET(2, n) * y2;
        y2 = y1; y1 = out;
        sc.stash[3][n] = fabsf(out) < 1e-15f ? 0.0f : out;
      }
      a.bp.y1 = y1; a.bp.y2 = y2;
    }
    gsync();
    const float filtered = sc.stash[3][lane];
    float mem_out = 0.0f;
    if (d.membrane > 0.0f) {  // MembraneResonator::process (membrane_resonator.rs:189-200); main_done is false here
      mem_out = membrane(a, sc, filtered * env_l, nv, lane);
      gsync(); STASH_PUT(5, fabsf(mem_out) * 0.001f); gsync();            // the product of membrane_resonator.rs:196 is per frame; only the sum is a recurrence
#pragma unroll 4
      for (int n = 0; n < nv; n++) a.ring_level = a.ring_level * 0.999f + STASH_GET(5, n);
    }
    const float dry_gain = 1.0f - d.mm;
    const float dry = filtered * env_l;
    const float fs = dry * dry_gain + mem_out * d.mm;
    return fs * fade * 0.7f * d.vol;
  }
};

// ---- the kernel ----------------------------------------------------------------------------------------------
// One voice per one-warp CTA.
template <class W>
__global__ void __launch_bounds__(32, 1) wave_kernel(const VoiceLaunch L) {
  using V = typename W::V; using Span = typename V::Span; using Aud = typename V::Aud;
  constexpr int WC = sizeof(typename V::Ctl) / 4;
  __shared__ GeoTables T;
  __shared__ WaveScratch sc;
  const int lane = threadIdx.x & 31;   // lane = frame within the block
  geo_tables_init(T, L.rc, threadIdx.x, 32);
  __syncthreads();
  const int v = blockIdx.x;
  const bool alive = v < L.n && L.mode[v] == 0;
  const int sv = alive ? (L.slots ? (int)L.slots[v] : v) : 0;
  Aud a;
  const Span* spans = nullptr;
  uint32_t ns = 0, cur = 0xffffffffu;
  typename V::Run run;
  typename W::Span2 w2;
  bool ready = false;
  int next_j0 = 0x7fffffff;
  float* out = nullptr;
  const float* planes = nullptr;
  if (alive) {
    load_words(a, L.state, sv, L.n_pad, WC);
    spans = reinterpret_cast<const Span*>(L.spans) + L.span_off[v];
    ns = L.n_spans[v];
    cur = L.span_cursor[v];
    if (cur != 0xffffffffu) V::span_resume(spans[cur], run);
    next_j0 = cur + 1u < ns ? spans[cur + 1u].j0 : 0x7fffffff;
    const long long row = L.rows ? (long long)L.rows[v] : (long long)(L.row0 + v);
    out = L.out + row * L.stride;
    planes = L.planes + (size_t)v * L.pitch;
  }
  const int c1 = L.chunk0 + min(L.chunk_frames, L.frames - L.chunk0);
  int j = L.chunk0;
  while (alive && j < c1) {
    while (j == next_j0) {
      cur += 1u;
      V::span_begin(a, spans[cur], run, L.rc.sr);
      ready = false;
      next_j0 = cur + 1u < ns ? spans[cur + 1u].j0 : 0x7fffffff;
    }
    const int span_end = min(next_j0, c1);
    const int act_end = min(span_end, W::active_end(run));
    if (cur == 0xffffffffu || !V::is_active(a, run, j) || j >= act_end) {      // silent until the next span: zero-fill
      for (int k = j + lane; k < span_end; k += 32) out[k] = 0.0f;
      j = span_end;
      continue;
    }
    if (!ready) { gsync(); W::span_setup(a, run, w2, sc, L.rc, lane); ready = true; }
    int nl = min(32, act_end - j);
    float p[V::NPL];
    const int jj = j + min(lane, nl - 1);       // lanes past the block re-read its last frame: finite, never stored
#pragma unroll
    for (int q = 0; q < V::NPL; q++) p[q] = planes[(size_t)q * L.plane_stride + (jj - L.chunk0)];
    const float y = W::block(a, run, w2, sc, T, p, j, nl, L.rc, lane);
    // block() shortens nl when the voice ended inside the block, or the tom's main oscillator did and a tail block
    // follows; the next iteration either zero-fills the silent stretch or takes the next block from there
    if (lane < nl) out[j + lane] = y;
    j += nl;
  }
  if (alive && lane == 0) {
    store_words(a, L.state, sv, L.n_pad, WC);
    L.span_cursor[v] = cur;
  }
}

#undef LANE_VAL
} }  // namespace gd::wave
