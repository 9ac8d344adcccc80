// dsp.cuh — device-side DSP building blocks for the batched offline renderer.
//
// One voice (or one engine) per thread; every struct here is a flat POD that
// lives in registers / local memory for the duration of a launch and is
// loaded/stored word-interleaved (SoA) from HBM at launch boundaries.
// Arithmetic follows the reference's f32 evaluation order exactly (compile with
// -fmad=false); transcendental calls that feed phase arguments go through the
// bit-exact gm:: routines (gmath.cuh).  Reference citations are relative to
// /root/reference/src.
#pragma once
#include "gmath.cuh"

#ifdef __CUDACC__
#define G_HD __host__ __device__ __forceinline__
#define G_D __device__ __forceinline__
#else
#define G_HD inline
#define G_D inline
#endif

namespace gd {

constexpr float PI_F = 3.14159265358979323846f;

G_HD float clampf(float x, float lo, float hi) { return x < lo ? lo : (x > hi ? hi : x); }
G_HD float denorm(float n, float mn, float mx) { return mn + clampf(n, 0.0f, 1.0f) * (mx - mn); }
G_HD float fract(float x) { return x - truncf(x); }

// u64 -> f32 round-to-nearest-even (Rust `as f32`)
G_HD float u64_to_f32(uint64_t h) {
#ifdef __CUDA_ARCH__
  return __ull2float_rn(h);
#else
  return (float)h;
#endif
}
G_HD uint64_t f32_to_u64_sat(float x) {  // Rust `as u64`
  if (!(x == x) || x <= 0.0f) return 0;
  if (x >= 18446744073709551616.0f) return 0xffffffffffffffffull;
  return (uint64_t)x;
}

// utils/smoother.rs:120-137 — settled <=> cur == tgt (see DESIGN.md).
G_HD void smooth_tick(float& cur, float tgt, float coeff) {
  if (cur != tgt) {
    cur += coeff * (tgt - cur);
    if (fabsf(cur - tgt) < 1e-4f) cur = tgt;
  }
}
G_HD float smooth_coeff(float sr, float ms) {  // :69-77
  if (ms <= 0.0f) return 1.0f;
  float n = (ms / 1000.0f) * sr;
  return 1.0f - gm::g_expf(-1.0f / n);
}
G_HD float tuning_to_multiplier(float n) {  // utils/mod.rs:14-17
  float semis = (clampf(n, 0.0f, 1.0f) - 0.5f) * 24.0f;
  return gm::g_powf(2.0f, semis / 12.0f);
}

// ---- envelope.rs ---------------------------------------------------------------------
struct Env {
  float attack, decay, sustain, release;
  float acurve, dcurve;   // exponent; < 0 encodes EnvelopeCurve::Linear
  double trig, rel_start;
  uint32_t flags;         // bit0 active, bit1 release latched
};
constexpr float CURVE_LINEAR = -1.0f;
G_HD float curve_apply(float c, float p) { return c < 0.0f ? p : gm::g_powf(p, clampf(c, 0.1f, 10.0f)); }
G_HD void env_init(Env& e) {  // Envelope::new() = ADSRConfig::default() (0.01, 0.3, 0.7, 0.5)
  e.attack = 0.01f; e.decay = 0.3f; e.sustain = 0.7f; e.release = 0.5f;
  e.acurve = CURVE_LINEAR; e.dcurve = CURVE_LINEAR; e.trig = 0.0; e.rel_start = 0.0; e.flags = 0;
}
// ADSRConfig::new floors (envelope.rs:40-49) + set_config
G_HD void env_config(Env& e, float a, float d, float s, float r, float ac = CURVE_LINEAR, float dc = CURVE_LINEAR) {
  e.attack = fmaxf(a, 0.001f); e.decay = fmaxf(d, 0.001f); e.sustain = clampf(s, 0.0f, 1.0f); e.release = fmaxf(r, 0.001f);
  e.acurve = ac; e.dcurve = dc;
}
G_HD void env_config_raw(Env& e, float a, float d, float s, float r, float ac, float dc) {  // struct-literal (bass.rs)
  e.attack = a; e.decay = d; e.sustain = s; e.release = r; e.acurve = ac; e.dcurve = dc;
}
G_HD void env_trigger(Env& e, double t) { e.flags = 1; e.trig = t; }
G_HD void env_release(Env& e, double t) { if ((e.flags & 3) == 1) { e.flags |= 2; e.rel_start = t; } }
G_HD bool env_active(const Env& e) { return e.flags & 1; }
G_HD float env_shape(const Env& e, float elapsed) {
  if (elapsed < e.attack) return curve_apply(e.acurve, elapsed / e.attack);
  if (elapsed < e.attack + e.decay) {
    float de = elapsed - e.attack;
    float dp = de / e.decay;
    float cp = curve_apply(e.dcurve, dp);
    return 1.0f - (1.0f - e.sustain) * cp;
  }
  return e.sustain;
}
// Envelope::get_amplitude (envelope.rs:154-211) split into its pure value and its latch side effects so that
// the time-parallel front-end can evaluate the value from a span-start snapshot (see DESIGN.md "A/B/C").
G_HD float env_value(const Env& e, double now) {
  if (!(e.flags & 1)) return 0.0f;
  float elapsed = (float)(now - e.trig);
  if (e.flags & 2) {
    float rel_el = (float)(now - e.rel_start);
    if (rel_el < e.release) {
      float ra = env_shape(e, elapsed);
      float rp = rel_el / e.release;
      return ra * (1.0f - rp);
    }
    return 0.0f;
  }
  if (elapsed < e.attack + e.decay || elapsed < e.attack) return env_shape(e, elapsed);
  return e.sustain;
}
G_HD void env_latch(Env& e, double now) {
  if (!(e.flags & 1)) return;
  if (e.flags & 2) {
    float rel_el = (float)(now - e.rel_start);
    if (!(rel_el < e.release)) e.flags &= ~1u;
    return;
  }
  float elapsed = (float)(now - e.trig);
  if (elapsed < e.attack + e.decay || elapsed < e.attack) return;
  if (e.sustain == 0.0f) { e.flags |= 2; e.rel_start = now; }
}
G_HD float env_amp(Env& e, double now) { float v = env_value(e, now); env_latch(e, now); return v; }

// ---- analytic advance of the latches over a frame range (planner, kernel A) -----------------------------------------
// tt[k] is the engine clock after k additions of 1/sr (bounce.rs:48-53); frame j of the call has k = kbase + j.
constexpr int J_NONE = 0x7fffffff;
// smallest j in [ja, jb) with pred(tt[kbase + j]) (pred monotone false->true); jb if none
template <class P> G_HD int first_true(const double* tt, uint32_t kbase, int ja, int jb, const P& pred) {
  int lo = ja, hi = jb;
  while (lo < hi) { int mid = lo + ((hi - lo) >> 1); if (pred(tt[kbase + mid])) hi = mid; else lo = mid + 1; }
  return lo;
}
struct EnvPastDecay { const Env* e; float ad; G_HD bool operator()(double now) const { float el = (float)(now - e->trig); return !(el < ad || el < e->attack); } };
struct EnvPastRelease { const Env* e; G_HD bool operator()(double now) const { float r = (float)(now - e->rel_start); return !(r < e->release); } };
// Applies to `e` exactly the latch transitions that ticking frames [ja, jb) would; returns the frame at whose tick
// the envelope became inactive (J_NONE if it does not within the range).
G_HD int env_advance(Env& e, const double* tt, uint32_t kbase, int ja, int jb) {
  if (!(e.flags & 1) || ja >= jb) return J_NONE;
  int j = ja;
  if (!(e.flags & 2)) {
    if (e.sustain != 0.0f) return J_NONE;
    EnvPastDecay p{&e, e.attack + e.decay};
    int j1 = first_true(tt, kbase, ja, jb, p);
    if (j1 >= jb) return J_NONE;
    e.flags |= 2; e.rel_start = tt[kbase + j1];
    j = j1 + 1;
  }
  EnvPastRelease q{&e};
  int j2 = first_true(tt, kbase, j, jb, q);
  if (j2 >= jb) return J_NONE;
  e.flags &= ~1u;
  return j2;
}

// ---- max_curve.rs ----------------------------------------------------------------------
// The factors of the curve > 0 branch of :21-48 that depend only on |curve|: fp and expm1f(fp).  A span stores them per
// envelope segment, so that the front end evaluates one expm1f per frame instead of powf + 2 expm1f.
struct CurveK { float fp, den, rcp_den; };
G_HD CurveK curve_k(float curve) {
  float hp = gm::g_powf((fabsf(curve) + 1e-20f) * 1.2f, 0.41f) * 0.91f;
  float fp = hp / (1.0f - hp);
  float den = gm::g_expm1f(fp);
  return {fp, den, 1.0f / den};
}
// expm1f(fp * progress) / expm1f(fp) through the reciprocal: every curve of the instruments (|curve| = 0.3, 0.8, 0.83) gives
// fp in [1.4, 10] and a quotient in [0, 1] that is 0 or above 1e-26 (progress is 0 or above 1e-22, see maxenv_value), never
// subnormal, so g_div_by returns the IEEE quotient.
G_HD float max_curve_pos(float progress, CurveK k) {
  if (fabsf(k.fp) < 1e-6f) return progress;
  return gm::g_div_by(gm::g_expm1f(k.fp * progress), k.den, k.rcp_den);
}
G_HD float max_curve(float progress, float curve, CurveK k) {  // k = curve_k(curve)
  progress = clampf(progress, 0.0f, 1.0f);
  if (fabsf(curve) < 1e-6f) return progress;
  if (curve < 0.0f) {
    // reference computes gp for the negative curve first, discards it, then recurses
    float q = clampf(1.0f - progress, 0.0f, 1.0f);
    return 1.0f - max_curve_pos(q, k);
  }
  return max_curve_pos(progress, k);
}
G_HD float max_curve(float progress, float curve) { return max_curve(progress, curve, curve_k(curve)); }
// Two-segment MaxCurveEnvelope (all users: hihat2.rs:442, tom2.rs:443) from initial value 0.
struct MaxEnv2 {
  float target[2], dur[2], curve[2];
  double seg_start;
  float seg_start_val, cur_val;
  uint32_t seg;     // current segment (2 = past the end)
  uint32_t active;
};
G_HD void maxenv_init(MaxEnv2& e, float t0, float d0ms, float c0, float t1, float d1ms, float c1) {
  e.target[0] = t0; e.dur[0] = d0ms / 1000.0f; e.curve[0] = c0;
  e.target[1] = t1; e.dur[1] = d1ms / 1000.0f; e.curve[1] = c1;
  e.seg_start = 0.0; e.seg_start_val = 0.0f; e.cur_val = 0.0f; e.seg = 0; e.active = 0;
}
G_HD void maxenv_trigger(MaxEnv2& e, double t) { e.active = 1; e.seg = 0; e.seg_start = t; e.seg_start_val = 0.0f; e.cur_val = 0.0f; }
G_HD void maxenv_set_dur_ms(MaxEnv2& e, int i, float ms) { e.dur[i] = fmaxf(ms / 1000.0f, 0.0f); }
G_HD bool maxenv_complete(const MaxEnv2& e) { return !e.active && e.seg >= 2; }
// The constants of one segment that depend only on its duration and curve.  The planner stores both segments' in the
// span, so that the front end does not recompute them every frame.
struct SegK { float rcp_dur; CurveK ck; };
G_HD SegK maxenv_seg_k(const MaxEnv2& e, bool s1) {
  const float dur = s1 ? e.dur[1] : e.dur[0];
  return {dur > 0.0f ? 1.0f / dur : 0.0f, curve_k(s1 ? e.curve[1] : e.curve[0])};
}
// max_curve.rs:133-174; kf(s1) gives the SegK of segment s1 (segments are picked by select, so that a copy of the
// envelope stays in registers)
template <class KF> G_HD float maxenv_value_k(MaxEnv2& e, double now, const KF& kf) {
  if (!e.active) return e.cur_val;
  for (;;) {
    if (e.seg >= 2) { e.active = 0; return e.cur_val; }
    const bool s1 = e.seg != 0;
    float el = (float)(now - e.seg_start);
    const float dur = s1 ? e.dur[1] : e.dur[0], target = s1 ? e.target[1] : e.target[0];
    if (el >= dur) {
      e.seg_start_val = target;
      e.cur_val = target;
      e.seg_start += (double)dur;
      e.seg += 1;
      continue;
    }
    const SegK k = kf(s1);
    // el / dur through the reciprocal.  Here 0 <= el < dur, and el is 0 or a difference of two clock values of which the
    // smaller is at least 1 / sr (or 0 and then el >= 1 / sr): el >= 2^-70, dur <= 4 s, so the quotient is 0 or far above the
    // subnormal range and g_div_by returns the IEEE quotient.
    float progress = dur > 0.0f ? gm::g_div_by(el, dur, k.rcp_dur) : 1.0f;
    float cp = max_curve(progress, s1 ? e.curve[1] : e.curve[0], k.ck);
    float range = target - e.seg_start_val;
    e.cur_val = e.seg_start_val + range * cp;
    return e.cur_val;
  }
}
G_HD float maxenv_value(MaxEnv2& e, double now) { return maxenv_value_k(e, now, [&](bool s1) { return maxenv_seg_k(e, s1); }); }
// both segments' constants, for a span (the durations and curves do not change within one)
struct MaxEnvK { SegK s[2]; };
G_HD MaxEnvK maxenv_k(const MaxEnv2& e) { return {{maxenv_seg_k(e, false), maxenv_seg_k(e, true)}}; }
G_HD float maxenv_value(MaxEnv2& e, double now, const MaxEnvK& k) { return maxenv_value_k(e, now, [&](bool s1) { return s1 ? k.s[1] : k.s[0]; }); }

// ---- SipHash-1-3(k=0) of one u64 (Rust DefaultHasher; oscillator.rs:187-196, morph_osc.rs:42-47)
G_HD uint64_t rotl64(uint64_t x, int b) { return (x << b) | (x >> (64 - b)); }
#define G_SIPROUND \
  v0 += v1; v1 = rotl64(v1, 13); v1 ^= v0; v0 = rotl64(v0, 32); \
  v2 += v3; v3 = rotl64(v3, 16); v3 ^= v2;                       \
  v0 += v3; v3 = rotl64(v3, 21); v3 ^= v0;                       \
  v2 += v1; v1 = rotl64(v1, 17); v1 ^= v2; v2 = rotl64(v2, 32);
G_HD uint64_t siphash13_u64(uint64_t m) {
  uint64_t v0 = 0x736f6d6570736575ull, v1 = 0x646f72616e646f6dull, v2 = 0x6c7967656e657261ull, v3 = 0x7465646279746573ull;
  v3 ^= m; G_SIPROUND v0 ^= m;
  const uint64_t b = 8ull << 56;
  v3 ^= b; G_SIPROUND v0 ^= b;
  v2 ^= 0xff; G_SIPROUND G_SIPROUND G_SIPROUND
  return v0 ^ v1 ^ v2 ^ v3;
}
G_HD float hash_noise(uint64_t idx) {
  float n = u64_to_f32(siphash13_u64(idx)) / 18446744073709551616.0f;
  return n * 2.0f - 1.0f;
}

// ---- gen/oscillator.rs: time-based waveforms ----------------------------------------------
// idx = f32(elapsed) * sr ; sine = sin(idx * freq * 2pi / sr), left-to-right in f32 (:42-46)
// 1 / (i * i) for odd i = 2 k + 1 < 2 INV_SQ_N, evaluated on the host with the expression of oscillator.rs:118 (an IEEE
// division costs ~10 instructions per harmonic otherwise); filled next to c_hb.
constexpr int INV_SQ_N = 1024;
#ifdef __CUDACC__
__constant__ float c_inv_sq[INV_SQ_N];
#endif
// FAST = the ~1-ulp sine (gm::g_sinf_fast) instead of the bit-exact glibc port: the time-parallel front end only
template <bool FAST = false> G_HD float osc_sine(float idx, float freq, float sr) {
  const float two_pi = 2.0f * PI_F;
  const float x = idx * freq * two_pi / sr;
  if (FAST) return gm::g_sinf_fast(x);
  return gm::g_sinf(x);
}
// the same with the reciprocal of the sample rate hoisted by the caller (additive oscillators: one division per harmonic)
G_HD float osc_sine_fast(float idx, float freq, float sr, float rcp_sr) {
  const float two_pi = 2.0f * PI_F;
  return gm::g_sinf_fast(gm::g_div_by(idx * freq * two_pi, sr, rcp_sr));
}
// 1 / (i * i) for odd i < 2 INV_SQ_N: the same f32 quotient, tabulated on the device (i is uniform across the warp)
G_HD float inv_sq_odd(int i, float fi) {
#ifdef __CUDA_ARCH__
  return c_inv_sq[i >> 1];
#else
  return 1.0f / (fi * fi);
#endif
}
template <bool FAST> G_HD float tri_partial(float idx, float hf, float sr, float rcp_sr) {
  return FAST ? osc_sine_fast(idx, hf, sr, rcp_sr) : osc_sine<false>(idx, hf, sr);
}
// additive "triangle": odd harmonics, gain 1/i^2 (powf(i,2) is exact so 1/(i*i) matches), Gibbs taper (:106-131).
// The reference's loop adds harmonic i = 1, 3, ... in increasing order and stops at the first with freq * i > nyquist; the
// taper is 1 while freq * i <= 0.7 nyquist (below that hf / nyquist cannot round above 0.75).  For freq > 0 and sr > 0,
// freq * i only grows with i, so the harmonics fall into three runs, each summed by a loop of its own with the reference's
// operations in the reference's order:
//   1. freq * i <= 0.7 nyquist and i < 2 INV_SQ_N: no taper (gain * 1 == gain), gain from the table;
//   2. the tapered top with i < 2 INV_SQ_N, where hf > 0.7 nyquist always holds;
//   3. i >= 2 INV_SQ_N (freq < nyquist / 2047, about 11 Hz at 44.1 kHz) or any other input: the reference's loop as written.
template <bool FAST = false> G_HD float osc_triangle(float idx, float freq, float sr) {
  float output = 0.0f;
  const float nyquist = sr / 2.0f;
  const float rcp_sr = 1.0f / sr;
  const float rcp_nyq = 2.0f * rcp_sr;      // == RN(1 / nyquist): both are scaled by exactly 2
  const float lim = 0.7f * nyquist;
  float q = nyquist / freq;
  int max_h = !(q == q) ? 0 : (q >= 2147483648.0f ? 2147483647 : (q <= -2147483648.0f ? (-2147483647 - 1) : (int)q));
  const int cap = (freq > 0.0f && sr > 0.0f) ? (max_h < 2 * INV_SQ_N - 1 ? max_h : 2 * INV_SQ_N - 1) : 0;   // last odd i runs 1 and 2 may take
  // n1 = number of harmonics of run 1 (i = 1, 3, ..., 2 n1 - 1): the guess from q is off by at most one harmonic
  int n1 = 0;
  if (cap >= 1) {
    n1 = ((int)fminf(q * 0.7f, (float)cap) + 1) >> 1;
    while (n1 > 0 && freq * (float)(2 * n1 - 1) > lim) n1--;
    while (2 * n1 + 1 <= cap && !(freq * (float)(2 * n1 + 1) > lim)) n1++;
  }
#ifdef __CUDA_ARCH__
#pragma unroll 4
#endif
  for (int h = 0; h < n1; h++) {
    const int i = 2 * h + 1;
    const float fi = (float)i;
    output += inv_sq_odd(i, fi) * tri_partial<FAST>(idx, freq * fi, sr, rcp_sr);
  }
  int i = 2 * n1 + 1;
  for (; i <= cap; i += 2) {
    const float fi = (float)i;
    const float hf = freq * fi;
    if (hf > nyquist) return output;
    // hf is in (0.7 nyquist, nyquist]: the quotient is near 1, never subnormal, so the hoisted reciprocal gives its exact bits
    const float ratio = gm::g_div_by(hf, nyquist, rcp_nyq);
    const float t = (ratio - 0.75f) / 0.25f;
    const float taper = ratio > 0.75f ? 1.0f - t * t : 1.0f;
    output += inv_sq_odd(i, fi) * taper * tri_partial<FAST>(idx, hf, sr, rcp_sr);
  }
  for (; i <= max_h; i += 2) {
    float fi = (float)i;
    if (freq * fi > nyquist) break;
    float gain = 1.0f / (fi * fi);
    float hf = freq * fi;
    float taper = 1.0f;
    if (hf > 0.7f * nyquist) {
      float ratio = hf / nyquist;
      if (ratio > 0.75f) { float t = (ratio - 0.75f) / 0.25f; taper = 1.0f - t * t; }
    }
    output += gain * taper * tri_partial<FAST>(idx, hf, sr, rcp_sr);
  }
  return output;
}

// ---- gen/pink_noise.rs ------------------------------------------------------------------------
constexpr uint64_t XS_SEED = 0x123456789abcdef0ull;
G_HD uint64_t xorshift64s_next(uint64_t& s) {
  uint64_t x = s;
  x ^= x >> 12; x ^= x << 25; x ^= x >> 27;
  s = x;
  return x * 0x2545f4914f6cdd1dull;
}
struct Pink { uint64_t rng; float f0, f1, f2; };
struct PinkCoef { float p0, p1, p2, g0, g1, g2; };
G_HD void pink_reset(Pink& p) { p.rng = XS_SEED; p.f0 = p.f1 = p.f2 = 0.0f; }
G_HD PinkCoef pink_coefs(float sr) {  // :24-46
  const float RP[3] = {0.99765f, 0.96300f, 0.57000f};
  const float RG[3] = {0.0990460f, 0.2965164f, 1.0526913f};
  sr = fmaxf(sr, 1.0f);
  float ratio = 44100.0f / sr;
  float po[3], ga[3];
  for (int i = 0; i < 3; i++) {
    po[i] = gm::g_powf(RP[i], ratio);
    ga[i] = RG[i] * sqrtf((1.0f - po[i] * po[i]) / (1.0f - RP[i] * RP[i]));
  }
  return {po[0], po[1], po[2], ga[0], ga[1], ga[2]};
}
G_HD float pink_tick(Pink& p, const PinkCoef& c) {  // :56-79
  uint64_t h = xorshift64s_next(p.rng);
#ifdef __CUDA_ARCH__
  // a / 16777215 through the rounded reciprocal (gm::g_div_by): bit-identical to the IEEE quotient for EVERY a in [0, 2^24)
  // (all 16 777 216 cases checked on the host), 3 instructions instead of div.rn's ~9 — the division was 9 % of a kick block
  float w = gm::g_div_by((float)(uint32_t)(h >> 40), 16777215.0f, 0x1.000002p-24f);
#else
  float w = (float)(uint32_t)(h >> 40) / 16777215.0f;
#endif
  w = w * 2.0f - 1.0f;
  p.f0 = c.p0 * p.f0 + c.g0 * w;
  p.f1 = c.p1 * p.f1 + c.g1 * w;
  p.f2 = c.p2 * p.f2 + c.g2 * w;
  float s = 0.0f + p.f0;
  s += p.f1;
  s += p.f2;
  return (s + w * 0.1848f) * 0.11f;
}

// ---- TPT SVF (filters/state_variable_tpt.rs, resonant_lowpass.rs share the core) -----------------
struct Tpt { float cutoff, res, g, r, h, ic1, ic2; };
G_HD void tpt_update(Tpt& f, float sr) {  // state_variable_tpt.rs:42-53
  float cutoff = clampf(f.cutoff, 20.0f, sr * 0.45f);
  float q = fmaxf(f.res, 0.5f);
  float g = gm::g_tanf(PI_F * cutoff / sr);
  float r = 1.0f / q;
  f.g = g; f.r = r; f.h = 1.0f / (1.0f + r * g + g * g);
}
G_HD void tpt_init(Tpt& f, float sr, float cutoff, float res) {
  f.cutoff = clampf(cutoff, 20.0f, 20000.0f); f.res = fmaxf(res, 0.5f); f.ic1 = f.ic2 = 0.0f; tpt_update(f, sr);
}
G_HD void tpt_set(Tpt& f, float sr, float cutoff, float res) {  // :83-92
  float nc = clampf(cutoff, 20.0f, sr * 0.45f);
  float nr = fmaxf(res, 0.5f);
  if (fabsf(nc - f.cutoff) > 0.001f || fabsf(nr - f.res) > 0.001f) { f.cutoff = nc; f.res = nr; tpt_update(f, sr); }
}
G_HD void tpt_process(Tpt& f, float in, float& lo, float& bd, float& hi) {  // :56-69
  float v1 = (f.g * (in - f.ic2) + f.ic1) * f.h;
  float v2 = f.ic2 + f.g * v1;
  f.ic1 = 2.0f * v1 - f.ic1;
  f.ic2 = 2.0f * v2 - f.ic2;
  lo = v2; bd = v1; hi = in - (f.r * v1 + v2);
}
G_HD float svf_pick(float lo, float bd, float hi, uint32_t type) {
  return type == 0 ? lo : (type == 2 ? hi : (type == 3 ? lo + hi : bd));
}
// ResonantLowpassFilter (resonant_lowpass.rs): clamps res to [0.5,10], cutoff to [20,20000]
G_HD void rlp_update(Tpt& f, float sr) {
  float s = fmaxf(sr, 1.0f);
  float cutoff = clampf(f.cutoff, 20.0f, s * 0.45f);
  float q = clampf(f.res, 0.5f, 10.0f);
  f.g = gm::g_tanf(PI_F * cutoff / s);
  f.r = 1.0f / q;
  f.h = 1.0f / (1.0f + f.r * f.g + f.g * f.g);
}
G_HD void rlp_init(Tpt& f, float sr, float cutoff, float res) {
  f.cutoff = clampf(cutoff, 20.0f, 20000.0f); f.res = clampf(res, 0.5f, 10.0f); f.ic1 = f.ic2 = 0.0f; rlp_update(f, sr);
}
G_HD void rlp_set(Tpt& f, float sr, float cutoff, float res) {
  cutoff = clampf(cutoff, 20.0f, 20000.0f);
  res = clampf(res, 0.5f, 10.0f);
  if (fabsf(cutoff - f.cutoff) > 0.001f || fabsf(res - f.res) > 0.001f) { f.cutoff = cutoff; f.res = res; rlp_update(f, sr); }
}
G_HD float rlp_process(Tpt& f, float in) {
  float v1 = (f.g * (in - f.ic2) + f.ic1) * f.h;
  float v2 = f.ic2 + f.g * v1;
  f.ic1 = 2.0f * v1 - f.ic1;
  f.ic2 = 2.0f * v2 - f.ic2;
  return fabsf(v2) < 1e-15f ? 0.0f : v2;
}

// ---- Chamberlin SVF (filters/state_variable.rs) -------------------------------------------------------
struct Chamb { float cutoff, res, f, q, low, band; };
G_HD void chamb_set(Chamb& s, float sr, float cutoff, float res) {  // set_params :131-135 (unconditional)
  float c = clampf(cutoff, 20.0f, 20000.0f), r = fmaxf(res, 0.5f);
  if (c == s.cutoff && r == s.res) return;  // same inputs -> same coefficients (pure function)
  s.cutoff = c; s.res = r;
  float nf = fminf(c / sr, 0.45f);
  s.f = 2.0f * gm::g_sinf(PI_F * nf);
  s.q = 1.0f / r;
}
G_HD void chamb_init(Chamb& s, float sr, float cutoff, float res) { s.cutoff = -1.0f; s.res = -1.0f; s.low = s.band = 0.0f; chamb_set(s, sr, cutoff, res); }
G_HD float chamb_process(Chamb& s, float in, uint32_t type) {  // :78-105
  float high = 0.0f;
  for (int i = 0; i < 2; i++) {
    s.low = s.low + s.f * s.band;
    high = in - s.low - s.q * s.band;
    s.band = s.f * high + s.band;
  }
  return svf_pick(s.low, s.band, high, type);
}

// ---- RBJ biquads, direct form I (filters/biquad_{bandpass,highpass}.rs) ---------------------------------
struct Biquad { float b0, b1, b2, a1, a2, x1, x2, y1, y2, last_freq, last_q, last_gain; };
G_HD void biquad_reset(Biquad& b) { b.x1 = b.x2 = b.y1 = b.y2 = 0.0f; }
G_HD float biquad_process(Biquad& b, float in) {
  float out = b.b0 * in + b.b1 * b.x1 + b.b2 * b.x2 - b.a1 * b.y1 - b.a2 * b.y2;
  b.x2 = b.x1; b.x1 = in; b.y2 = b.y1; b.y1 = out;
  return fabsf(out) < 1e-15f ? 0.0f : out;
}
G_HD void bp_compute(Biquad& b, float sr, float freq, float q, float gain) {  // coefficient formulas of biquad_bandpass.rs:88-119
  float nyq = sr * 0.5f;
  freq = clampf(freq, 20.0f, nyq * 0.95f);
  q = clampf(q, 0.1f, 100.0f);
  float w0 = 2.0f * PI_F * freq / sr;
  float sn = gm::g_sinf(w0), cs = gm::g_cosf(w0);
  float alpha = sn / (2.0f * q);
  float B0 = q * alpha * gain, B1 = 0.0f, B2 = -q * alpha * gain;
  float A0 = 1.0f + alpha, A1 = -2.0f * cs, A2 = 1.0f - alpha;
  b.b0 = B0 / A0; b.b1 = B1 / A0; b.b2 = B2 / A0; b.a1 = A1 / A0; b.a2 = A2 / A0;
}
G_HD bool bp_unchanged(const Biquad& b, float freq, float q, float gain) {  // :73-87
  return fabsf(freq - b.last_freq) < 0.01f && fabsf(q - b.last_q) < 0.001f && fabsf(gain - b.last_gain) < 0.001f;
}
G_HD void bp_set(Biquad& b, float sr, float freq, float q, float gain) {  // biquad_bandpass.rs:73-119
  if (bp_unchanged(b, freq, q, gain)) return;
  b.last_freq = freq; b.last_q = q; b.last_gain = gain;
  bp_compute(b, sr, freq, q, gain);
}
G_HD void bp_init(Biquad& b, float sr) { b.last_freq = b.last_q = b.last_gain = -1.0f; biquad_reset(b); bp_set(b, sr, 1000.0f, 1.0f, 1.0f); }
G_HD void hp_set(Biquad& b, float sr, float freq, float q) {  // biquad_highpass.rs:68-96
  if (fabsf(freq - b.last_freq) < 0.01f && fabsf(q - b.last_q) < 0.001f) return;
  b.last_freq = freq; b.last_q = q;
  float nyq = sr * 0.5f;
  freq = clampf(freq, 20.0f, nyq * 0.95f);
  q = clampf(q, 0.1f, 100.0f);
  float w0 = 2.0f * PI_F * freq / sr;
  float sn = gm::g_sinf(w0), cs = gm::g_cosf(w0);
  float alpha = sn / (2.0f * q);
  float B0 = (1.0f + cs) / 2.0f, B1 = -(1.0f + cs), B2 = (1.0f + cs) / 2.0f;
  float A0 = 1.0f + alpha, A1 = -2.0f * cs, A2 = 1.0f - alpha;
  b.b0 = B0 / A0; b.b1 = B1 / A0; b.b2 = B2 / A0; b.a1 = A1 / A0; b.a2 = A2 / A0;
}
G_HD void hp_init(Biquad& b, float sr) { b.last_freq = b.last_q = -1.0f; b.last_gain = 0.0f; biquad_reset(b); hp_set(b, sr, 1000.0f, 1.0f); }

// ---- halfband (third-party crate, reconstructed; see DESIGN.md "halfband") --------------------------------
// 8 polyphase allpass sections: even-index coefficients on path 0, odd on path 1,
// section: y[n] = c*(x[n]-y[n-1]) + x[n-1].  Coefficients are designed on the host
// (csrc/halfband_design.h) and live in constant memory.
#ifdef __CUDACC__
__constant__ float c_hb[8];
#define G_HB(i) c_hb[i]
#else
extern float g_hb_host[8];
#define G_HB(i) g_hb_host[i]
#endif
struct Hb8 { float x[8], y[8]; };
G_HD void hb_clear(Hb8& s) { for (int i = 0; i < 8; i++) s.x[i] = s.y[i] = 0.0f; }
G_D void hb_run(Hb8& s, float& p0, float& p1) {
#pragma unroll
  for (int i = 0; i < 8; i += 2) {
    float t0 = (p0 - s.y[i]) * G_HB(i) + s.x[i];
    float t1 = (p1 - s.y[i + 1]) * G_HB(i + 1) + s.x[i + 1];
    s.x[i] = p0; s.x[i + 1] = p1; s.y[i] = t0; s.y[i + 1] = t1;
    p0 = t0; p1 = t1;
  }
}
G_D void hb_up(Hb8& s, float in, float& o0, float& o1) { o0 = in; o1 = in; hb_run(s, o0, o1); }
G_D float hb_down(Hb8& s, float i0, float i1) { float a = i1, b = i0; hb_run(s, a, b); return 0.5f * (a + b); }

// utils/oversampler.rs:38-175.  mode: 0 Off, 2 X2, 4 X4.  X2 shares the outer pair's storage: a mode
// change resets every stage (:150-155) and only the active mode's stages ever run.
struct Oversamp { Hb8 outer_up, inner_up, inner_down, outer_down; uint32_t mode; };
G_HD void os_reset(Oversamp& o) { hb_clear(o.outer_up); hb_clear(o.inner_up); hb_clear(o.inner_down); hb_clear(o.outer_down); }
G_HD void os_init(Oversamp& o) { os_reset(o); o.mode = 4; }
template <class F> G_D float os_process(Oversamp& o, float in, F f) {
  if (o.mode == 0) return f(in);
  if (o.mode == 2) { float s0, s1; hb_up(o.outer_up, in, s0, s1); float a = f(s0), b = f(s1); return hb_down(o.outer_down, a, b); }
  float o0, o1, i0, i1, i2, i3;
  hb_up(o.outer_up, in, o0, o1);
  hb_up(o.inner_up, o0, i0, i1);
  float fa = f(i0), fb = f(i1);
  float d0 = hb_down(o.inner_down, fa, fb);
  hb_up(o.inner_up, o1, i2, i3);
  float fc = f(i2), fd = f(i3);
  float d1 = hb_down(o.inner_down, fc, fd);
  return hb_down(o.outer_down, d0, d1);
}

// ---- effects/waveshaper.rs:48-72 -----------------------------------------------------------------------------
struct WShaper { float drive, mix; Oversamp os; };
G_HD void ws_init(WShaper& w, float drive, float mix) { w.drive = clampf(drive, 1.0f, 10.0f); w.mix = clampf(mix, 0.0f, 1.0f); os_init(w.os); }
G_D float ws_core(float drive, float mix, Oversamp& os, float in) {
  if (!isfinite(in)) { os_reset(os); return 0.0f; }
  if (mix <= 0.0001f || drive <= 1.0f) return in;
  float d = drive;
  float comp = gm::g_tanhf(0.5f) / gm::g_tanhf(0.5f * d);
  float sat = os_process(os, in, [&](float x) { return gm::g_tanhf(x * d) * comp; });
  return in * (1.0f - mix) + sat * mix;
}
G_D float ws_process(WShaper& w, float in) { return ws_core(w.drive, w.mix, w.os, in); }

// ---- effects/feedback_waveshaper.rs ---------------------------------------------------------------------------
struct FbShaper {
  float drive, mix, feedback, cutoff, filter_coeff, env_att, env_rel;
  float last_out, filter_state, dc_x1, dc_y1, env;
  float memo_drive, memo_fb, memo_makeup;   // makeup gain is a pure function of (drive, feedback): cached, bit-identical
  Oversamp os;
};
G_HD float fbws_filter_coeff(float c, float sr) { float g = 1.0f - gm::g_expf(-2.0f * PI_F * c / sr); return clampf(g, 0.0f, 0.9f); }
G_HD void fbws_init(FbShaper& w, float sr, float drive, float fb, float cutoff, float mix) {
  w.drive = clampf(drive, 1.0f, 100.0f); w.mix = clampf(mix, 0.0f, 1.0f); w.feedback = clampf(fb, 0.0f, 0.98f);
  w.cutoff = clampf(cutoff, 200.0f, 20000.0f);
  w.filter_coeff = fbws_filter_coeff(w.cutoff, sr);
  w.env_att = gm::g_expf(-1.0f / (1.0f / 1000.0f * sr));
  w.env_rel = gm::g_expf(-1.0f / (120.0f / 1000.0f * sr));
  w.last_out = w.filter_state = w.dc_x1 = w.dc_y1 = w.env = 0.0f;
  w.memo_drive = -1.0f; w.memo_fb = -1.0f; w.memo_makeup = 1.0f;
  os_init(w.os);
}
G_HD void fbws_reset(FbShaper& w) { w.last_out = w.filter_state = w.dc_x1 = w.dc_y1 = w.env = 0.0f; os_reset(w.os); }
G_HD void fbws_set_cutoff(FbShaper& w, float sr, float c) {
  c = clampf(c, 200.0f, 20000.0f);
  if (c != w.cutoff) { w.cutoff = c; w.filter_coeff = fbws_filter_coeff(c, sr); }  // pure function of (c, sr)
}
// The functions below are templates over the state struct: FbShaper (a voice's own shaper, oversampler inside) and mix.cuh's
// FbSmall (an effect slot, whose oversampler history lives in the slot's ring arena) share field names.
template <class S> G_D float fbws_makeup(S& w) {  // the level-independent factor of gain_compensation (:252-256)
  if (w.drive != w.memo_drive || w.feedback != w.memo_fb) {
    float drive_norm = clampf((w.drive - 1.0f) / 99.0f, 0.0f, 1.0f);
    float fb_norm = clampf(w.feedback / 0.98f, 0.0f, 1.0f);
    float high_end = gm::g_powf(drive_norm, 1.35f) * gm::g_powf(fb_norm, 2.0f);
    w.memo_makeup = gm::g_powf(10.0f, 5.1f * high_end / 20.0f);
    w.memo_drive = w.drive; w.memo_fb = w.feedback;
  }
  return w.memo_makeup;
}
template <class S> G_D float fbws_gain_comp(S& w, float env) {  // :247-259
  float reference = fmaxf(env, 0.05f);
  float driven = fmaxf(fabsf(gm::g_tanhf(reference * w.drive)), 1e-6f);
  float comp_no_fb = gm::g_tanhf(reference) / driven;
  float makeup = fbws_makeup(w);
  float taming = 1.0f / (1.0f + comp_no_fb * w.feedback * 0.25f);
  return fminf(comp_no_fb * taming * makeup, 3.0f);
}
template <class S> G_D float fbws_core(S& w, Oversamp& os, float in) {  // :109-169
  if (!isfinite(in)) { w.last_out = w.filter_state = w.dc_x1 = w.dc_y1 = w.env = 0.0f; os_reset(os); return 0.0f; }
  if (w.mix <= 0.0001f || w.drive <= 1.0f) return in;
  float fb_in = w.drive * in + w.feedback * w.last_out;
  float shaped = os_process(os, fb_in, [](float x) { return gm::g_tanhf(x); });
  float rect = fabsf(in);
  float coeff = rect > w.env ? w.env_att : w.env_rel;
  w.env += (1.0f - coeff) * (rect - w.env);
  if (fabsf(w.env) < 1e-15f) w.env = 0.0f;
  float comp = fbws_gain_comp(w, w.env);
  float compensated = shaped * comp;
  float out = compensated - w.dc_x1 + 0.995f * w.dc_y1;
  w.dc_x1 = compensated;
  w.dc_y1 = fabsf(out) < 1e-15f ? 0.0f : out;
  w.filter_state += w.filter_coeff * (out - w.filter_state);
  if (fabsf(w.filter_state) < 1e-15f) w.filter_state = 0.0f;
  w.last_out = w.filter_state;
  if (!isfinite(w.last_out) || fabsf(w.last_out) > 50.0f) { w.last_out = w.filter_state = w.dc_x1 = w.dc_y1 = w.env = 0.0f; os_reset(os); return in; }
  return in * (1.0f - w.mix) + out * w.mix;
}
G_D float fbws_process(FbShaper& w, float in) { return fbws_core(w, w.os, in); }

// ---- instruments/fm_snap.rs:102-169 -----------------------------------------------------------------------------
struct PhaseMod { double trig; uint32_t active; };
G_HD float phasemod_value(const PhaseMod& m, double now) {
  if (!m.active) return 0.0f;
  float el = (float)(now - m.trig);
  const float attack = 0.001f, decay = 0.005f;
  float total = attack + decay;
  if (el > total) return 0.0f;
  if (el < attack) return gm::g_powf(el / attack, 0.3f);
  float de = el - attack;
  return 1.0f - gm::g_powf(de / decay, 0.4f);
}
G_HD void phasemod_latch(PhaseMod& m, double now) {
  if (!m.active) return;
  float el = (float)(now - m.trig);
  if (el > 0.001f + 0.005f) m.active = 0;
}
G_HD float phasemod_tick(PhaseMod& m, double now) { float v = phasemod_value(m, now); phasemod_latch(m, now); return v; }
struct PmPast { const PhaseMod* m; G_HD bool operator()(double now) const { float el = (float)(now - m->trig); return el > 0.001f + 0.005f; } };
G_HD int phasemod_advance(PhaseMod& m, const double* tt, uint32_t kbase, int ja, int jb) {
  if (!m.active || ja >= jb) return J_NONE;
  PmPast p{&m};
  int j = first_true(tt, kbase, ja, jb, p);
  if (j >= jb) return J_NONE;
  m.active = 0;
  return j;
}

// MaxCurveEnvelope transitions are path independent (each depends only on `now`), so the value at any frame can be
// computed from a span-start snapshot, and the state after a range is the state after its last frame.
G_HD float maxenv_value_pure(const MaxEnv2& e, double now) { MaxEnv2 t = e; return maxenv_value(t, now); }
G_HD float maxenv_value_pure(const MaxEnv2& e, const MaxEnvK& k, double now) { MaxEnv2 t = e; return maxenv_value(t, now, k); }
struct MaxEnvDone { const MaxEnv2* e; G_HD bool operator()(double now) const { MaxEnv2 t = *e; maxenv_value(t, now); return t.seg >= 2; } };
// first frame in [ja, jb) whose tick leaves the envelope complete (seg >= 2); jb if none
G_HD int maxenv_complete_frame(const MaxEnv2& e, const double* tt, uint32_t kbase, int ja, int jb) {
  if (!e.active) return e.seg >= 2 ? ja : jb;
  MaxEnvDone p{&e};
  return first_true(tt, kbase, ja, jb, p);
}

}  // namespace gd
