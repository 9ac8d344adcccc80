// voices.cuh — the drum voices (kick, snare, hi-hat, tom).
//
// Every voice is split into a CONTROL half (Ctl: smoothed parameters, envelopes, trigger bookkeeping —
// everything that is a pure function of time once the parameters are settled) and an AUDIO half (Aud: filter
// memories, RNGs, phase accumulators, oversampler history — the true sample-to-sample recurrences).
//
//   <v>_event(Ctl&, e, tt, resets)   host-resolved event (events.h) applied to the control half; audio-side
//                                    resets are returned as bits and applied by <v>_span_begin().
//   <v>_front(Ctl, Der, now) -> planes   PURE: oscillators, hash noise, envelope values.  Kernel B evaluates it for
//                                    thousands of frames of one voice at once (time-parallel).
//   <v>_back(Aud&, Der, planes)      the recurrences; kernel C runs it one voice per thread.
//   <v>_plan(Ctl&, ..., Span&)       kernel A: advances the control half analytically over a span of frames
//                                    (envelope latches by binary search on the engine clock table) and snapshots it.
//   <v>_tick(State&)                 the reference's per-sample tick, composed from the same pieces; used for
//                                    voices whose parameters are still gliding (general path, kernel S).
//
// Reference: src/instruments/{kick,snare,hihat2,tom2}.rs; citations inline.  Time: frame k of an engine has
// now = tt[k], the f64 clock after k additions of 1/sr (src/bounce.rs:48-53, src/ffi.rs:1096,1379).
#pragma once
#include "dsp.cuh"
#include "events.h"

namespace gd {

// Per-launch constants derived from the sample rate (uniform across a batch).
struct RateCtx {
  float sr;
  double dt;          // 1.0 / (sr as f64)
  float smooth15;     // SmoothedParam coeff, 15 ms (DEFAULT_SMOOTH_TIME_MS)
  float smooth10, smooth30, smooth50;
  float click_alpha;  // kick click HP: 1 - exp(-2pi*8000/sr) (resonant_highpass.rs:44-45)
  float asym_down;    // hihat AsymmetricSmoother(100 samples) (hihat2.rs:295-305)
  PinkCoef pink;
};
G_HD RateCtx make_rate_ctx(float sr) {
  RateCtx c;
  c.sr = sr;
  c.dt = 1.0 / (double)sr;
  c.smooth15 = smooth_coeff(sr, 15.0f);
  c.smooth10 = smooth_coeff(sr, 10.0f);
  c.smooth30 = smooth_coeff(sr, 30.0f);
  c.smooth50 = smooth_coeff(sr, 50.0f);
  c.click_alpha = 1.0f - gm::g_expf(-2.0f * PI_F * 8000.0f / sr);
  c.asym_down = 1.0f - gm::g_expf(-1.0f / 100.0f);
  c.pink = pink_coefs(sr);
  return c;
}

enum : uint32_t { RST_TRIGGER = 1u };   // audio-side reset requested by a trigger event

// Common smoothed-parameter event handling (cur/tgt arrays of NP entries).
template <int NP> G_HD bool params_settled(const float* cur, const float* tgt) {
  bool ok = true;
#pragma unroll
  for (int i = 0; i < NP; i++) ok &= (cur[i] == tgt[i]);
  return ok;
}
template <int NP> G_HD void params_set_target(float* tgt, uint32_t p, float v) {
  // compare-select over every slot instead of tgt[p]: a dynamic index would force the whole state into local memory
  const float c = clampf(v, 0.0f, 1.0f);
#pragma unroll
  for (int i = 0; i < NP; i++) if ((uint32_t)i == p && fabsf(tgt[i] - c) > 1e-8f) tgt[i] = c;
}
template <int NP> G_HD void params_snap(float* cur, const float* tgt) {
#pragma unroll
  for (int i = 0; i < NP; i++) cur[i] = tgt[i];
}

// =========================================== Kick ===========================================
enum { K_FREQ, K_PUNCH, K_SUB, K_CLICK, K_OSC_DECAY, K_PITCH_ENV_AMT, K_PITCH_ENV_CURVE, K_VOLUME,
       K_PITCH_START_RATIO, K_PHASE_MOD, K_NOISE_AMT, K_NOISE_CUTOFF, K_NOISE_RES, K_OVERDRIVE,
       K_FEEDBACK, K_FB_CUTOFF, K_AMP_DECAY, K_AMP_DECAY_CURVE, K_TUNING, K_NP };

struct KickCtl {
  float cur[K_NP], tgt[K_NP];
  uint32_t os_mode;   // FeedbackWaveshaper oversampling mode (0/2/4)
  Env sub_env, punch_env, click_env, pitch_env, noise_env, amp_env;
  PhaseMod pm;
  float tpm;          // triggered_pitch_multiplier
  float velocity;
  uint32_t active;
  float saved_freq; uint32_t has_saved;   // VoiceStrip.saved_global_freq (ffi.rs:596, 1176-1194)
  uint32_t k;         // engine clock index of the next frame
};
struct KickAud {
  float click_hp;     // ResonantHighpassFilter.filter_state
  uint32_t pad0;
  Pink pink;
  Tpt noise_lp;
  FbShaper ws;
};
struct KickState { KickCtl c; KickAud a; };
struct KickDer {      // per-tick derived values (constant while the parameters are settled)
  float sub_vol, punch_vol, click_vol, base_frequency, pma, noise_amount, noise_cut, noise_res, drive, feedback, fb_cutoff, va, volume;
};
struct KickFront { float p1, raw_click, ne, amp; };
enum { KICK_PLANES = 4 };

G_HD float overdrive_to_drive(float a) { return 1.0f + a * a * a * 40.0f; }

// KickDrum::with_config (kick.rs:712-775) + configure_oscillators (:777-817); cfg = 18 normalized values
G_HD void kick_init(KickState& s, const float* cfg, float sr) {
  KickCtl& c = s.c; KickAud& a = s.a;
  for (int i = 0; i < 18; i++) { float v = clampf(cfg[i], 0.0f, 1.0f); c.cur[i] = c.tgt[i] = v; }
  c.cur[K_TUNING] = c.tgt[K_TUNING] = 0.5f;
  c.os_mode = 4;
  float ratio = denorm(c.cur[K_PITCH_START_RATIO], 1.0f, 10.0f);
  c.tpm = 1.0f + (ratio - 1.0f) * c.cur[K_PITCH_ENV_AMT];
  float decay = denorm(c.cur[K_OSC_DECAY], 0.01f, 4.0f);
  env_init(c.sub_env); env_init(c.punch_env); env_init(c.click_env); env_init(c.pitch_env); env_init(c.noise_env); env_init(c.amp_env);
  env_config(c.sub_env, 0.001f, decay, 0.0f, decay * 0.2f);
  env_config(c.punch_env, 0.001f, decay, 0.0f, decay * 0.2f);
  env_config(c.click_env, 0.001f, decay * 0.2f, 0.0f, decay * 0.02f);
  float pd = decay * 0.6f;
  env_config(c.pitch_env, 0.001f, pd, 0.0f, pd * 0.1f);
  env_config(c.noise_env, 0.001f, decay, 0.0f, decay * 0.2f);
  c.pm.trig = 0.0; c.pm.active = 0;
  c.velocity = 1.0f; c.active = 0; c.saved_freq = 0.0f; c.has_saved = 0; c.k = 0;
  a.click_hp = 0.0f; a.pad0 = 0;
  pink_reset(a.pink);
  rlp_init(a.noise_lp, sr, denorm(c.cur[K_NOISE_CUTOFF], 20.0f, 10000.0f), denorm(c.cur[K_NOISE_RES], 0.0f, 5.0f));
  fbws_init(a.ws, sr, overdrive_to_drive(c.cur[K_OVERDRIVE]), c.cur[K_FEEDBACK] * 0.98f, 200.0f + c.cur[K_FB_CUTOFF] * 3800.0f, 1.0f);
}

// KickDrum::trigger_with_velocity (kick.rs:971-1086), control half
G_HD void kick_trigger(KickCtl& c, float velocity, double time) {
  c.velocity = clampf(velocity, 0.0f, 1.0f);
  c.active = 1;
  float vel = c.velocity, vel2 = vel * vel;
  float decay_scale = 1.0f - (0.5f * vel2);
  float base_decay = denorm(c.cur[K_OSC_DECAY], 0.01f, 4.0f) * decay_scale;
  float psr = denorm(c.cur[K_PITCH_START_RATIO], 1.0f, 10.0f);
  c.tpm = 1.0f + (psr - 1.0f) * c.cur[K_PITCH_ENV_AMT];
  float pcv = denorm(c.cur[K_PITCH_ENV_CURVE], 0.1f, 4.0f);
  float dc = fabsf(pcv - 1.0f) < 0.01f ? CURVE_LINEAR : pcv;
  env_config(c.pitch_env, 0.001f, base_decay, 0.0f, base_decay * 0.2f, CURVE_LINEAR, dc);
  env_config(c.sub_env, 0.001f, base_decay, 0.0f, base_decay * 0.2f);
  env_config(c.punch_env, 0.001f, base_decay, 0.0f, base_decay * 0.2f);
  env_config(c.click_env, 0.001f, base_decay * 0.2f, 0.0f, base_decay * 0.02f);
  env_trigger(c.sub_env, time); env_trigger(c.punch_env, time); env_trigger(c.click_env, time);
  env_trigger(c.pitch_env, time);
  if (c.cur[K_PHASE_MOD] > 0.001f) { c.pm.trig = time; c.pm.active = 1; }
  env_config(c.noise_env, 0.001f, base_decay, 0.0f, base_decay * 0.2f);
  env_trigger(c.noise_env, time);
  float amp_decay = denorm(c.cur[K_AMP_DECAY], 0.0f, 4.0f) * decay_scale;
  float adc = denorm(c.cur[K_AMP_DECAY_CURVE], 0.1f, 10.0f);
  float adcv = fabsf(adc - 1.0f) < 0.01f ? CURVE_LINEAR : adc;
  env_config(c.amp_env, 0.001f, amp_decay, 0.0f, amp_decay * 0.2f, 0.5f, adcv);
  env_trigger(c.amp_env, time);
}

G_HD void kick_event(KickCtl& c, const VoiceEvent& e, const double* tt, uint32_t& resets) {
  switch (e.kind) {
    case EV_TRIGGER: kick_trigger(c, e.value, tt[c.k]); resets |= RST_TRIGGER; break;
    case EV_SET_TARGET: params_set_target<K_NP>(c.tgt, e.param, e.value); break;
    case EV_SNAP: params_snap<K_NP>(c.cur, c.tgt); break;
    case EV_SET_AUX: if (e.param == AUX_OVERSAMPLING) c.os_mode = (uint32_t)e.value; break;
    case EV_SET_TIME: c.k = e.aux; break;
    case EV_NOTE_FREQ:
      if (!c.has_saved) { c.saved_freq = c.cur[K_FREQ]; c.has_saved = 1; }
      params_set_target<K_NP>(c.tgt, K_FREQ, e.value);
      params_snap<K_NP>(c.cur, c.tgt);
      break;
    case EV_RESTORE_FREQ:
      if (c.has_saved) { c.has_saved = 0; params_set_target<K_NP>(c.tgt, K_FREQ, c.saved_freq); params_snap<K_NP>(c.cur, c.tgt); }
      break;
    default: break;
  }
}
// audio-side consequences of events (kick.rs:1082-1085; the FeedbackWaveshaper is NOT reset by a trigger)
G_HD void kick_span_begin(KickAud& a, const KickCtl& c, uint32_t resets) {
  if (resets & RST_TRIGGER) { a.click_hp = 0.0f; a.noise_lp.ic1 = a.noise_lp.ic2 = 0.0f; pink_reset(a.pink); }
  if (a.ws.os.mode != c.os_mode) { a.ws.os.mode = c.os_mode; os_reset(a.ws.os); }
}

// live decay re-application (kick.rs:1111-1136), no floors
G_HD void kick_live(KickCtl& c) {
  float vel2 = c.velocity * c.velocity;
  float decay_scale = 1.0f - (0.5f * vel2);
  float base_decay = denorm(c.cur[K_OSC_DECAY], 0.01f, 4.0f) * decay_scale;
  c.sub_env.decay = base_decay; c.sub_env.release = base_decay * 0.2f;
  c.punch_env.decay = base_decay; c.punch_env.release = base_decay * 0.2f;
  c.click_env.decay = base_decay * 0.2f; c.click_env.release = base_decay * 0.02f;
  c.noise_env.decay = base_decay; c.noise_env.release = base_decay * 0.2f;
  c.pitch_env.decay = base_decay; c.pitch_env.release = base_decay * 0.2f;
}
G_HD KickDer kick_derive(const KickCtl& c) {
  KickDer d;
  float cvs = 0.6f + 0.4f * c.velocity;   // apply_params (:820-835)
  d.sub_vol = clampf(c.cur[K_SUB], 0.0f, 1.0f);
  d.punch_vol = clampf(c.cur[K_PUNCH] * 0.7f, 0.0f, 1.0f);
  d.click_vol = clampf(c.cur[K_CLICK] * 0.15f * cvs, 0.0f, 1.0f);
  d.base_frequency = denorm(c.cur[K_FREQ], 30.0f, 120.0f) * tuning_to_multiplier(c.cur[K_TUNING]);
  d.pma = c.cur[K_PHASE_MOD];
  d.noise_amount = c.cur[K_NOISE_AMT];
  d.noise_cut = denorm(c.cur[K_NOISE_CUTOFF], 20.0f, 10000.0f);
  d.noise_res = denorm(c.cur[K_NOISE_RES], 0.0f, 5.0f);
  d.drive = clampf(overdrive_to_drive(c.cur[K_OVERDRIVE]), 1.0f, 100.0f);
  d.feedback = clampf(c.cur[K_FEEDBACK] * 0.98f, 0.0f, 0.98f);
  d.fb_cutoff = 200.0f + c.cur[K_FB_CUTOFF] * 3800.0f;
  d.va = sqrtf(c.velocity);
  d.volume = c.cur[K_VOLUME];
  return d;
}
// Oscillator::tick x3 (oscillator.rs:242-286) + envelope values.  An oscillator whose envelope amplitude or volume
// is exactly 0 contributes raw*0 = +-0, so its waveform is skipped (raw is always finite).
template <bool FAST = false> G_HD KickFront kick_front(const KickCtl& c, const KickDer& d, double now, float sr) {
  KickFront f;
  float pev = env_value(c.pitch_env, now);
  float fm = 1.0f + (c.tpm - 1.0f) * pev;
  if (d.pma > 0.001f) {
    float pm = phasemod_value(c.pm, now);
    fm *= 1.0f + (pm * d.pma * 2.0f);
  }
  float sub_f = d.base_frequency * fm;
  float punch_f = d.base_frequency * 2.5f * fm;
  float sub_out = 0.0f, punch_out = 0.0f;
  f.raw_click = 0.0f;
  {
    float idx = env_active(c.sub_env) ? (float)(now - c.sub_env.trig) * sr : 0.0f;
    float amp = env_value(c.sub_env, now);
    if (amp != 0.0f && d.sub_vol != 0.0f) sub_out = osc_sine<FAST>(idx, sub_f, sr) * amp * d.sub_vol;
  }
  {
    float idx = env_active(c.punch_env) ? (float)(now - c.punch_env.trig) * sr : 0.0f;
    float amp = env_value(c.punch_env, now);
    if (amp != 0.0f && d.punch_vol != 0.0f) punch_out = osc_triangle<FAST>(idx, punch_f, sr) * amp * d.punch_vol;
  }
  {
    float idx = env_active(c.click_env) ? (float)(now - c.click_env.trig) * sr : 0.0f;
    float amp = env_value(c.click_env, now);
    if (amp != 0.0f && d.click_vol != 0.0f) f.raw_click = hash_noise(f32_to_u64_sat(idx)) * amp * d.click_vol;
  }
  f.p1 = sub_out + punch_out;
  f.ne = d.noise_amount > 0.001f ? env_value(c.noise_env, now) : 0.0f;
  f.amp = env_value(c.amp_env, now);
  return f;
}
G_HD void kick_latch(KickCtl& c, const KickDer& d, double now) {
  env_latch(c.pitch_env, now);
  if (d.pma > 0.001f) phasemod_latch(c.pm, now);
  env_latch(c.sub_env, now); env_latch(c.punch_env, now); env_latch(c.click_env, now);
  if (d.noise_amount > 0.001f) env_latch(c.noise_env, now);
  env_latch(c.amp_env, now);
}
G_D float kick_back(KickAud& a, const KickDer& d, const KickFront& f, const RateCtx& rc) {
  const float sr = rc.sr;
  // click HP (resonant_highpass.rs:22-54), resonance 4.0
  float hp = f.raw_click - a.click_hp;
  a.click_hp += rc.click_alpha * hp;
  float filt_click = hp * (1.0f + 4.0f * 0.1f);
  float noise_out = 0.0f;
  if (d.noise_amount > 0.001f) {
    float pn = pink_tick(a.pink, rc.pink);
    rlp_set(a.noise_lp, sr, d.noise_cut, d.noise_res);
    float fn = rlp_process(a.noise_lp, pn);
    noise_out = fn * f.ne * d.noise_amount * 0.5f;
  }
  float total = f.p1 + filt_click + noise_out;
  a.ws.drive = d.drive;
  a.ws.feedback = d.feedback;
  fbws_set_cutoff(a.ws, sr, d.fb_cutoff);
  float od = fbws_process(a.ws, total);
  return od * f.amp * d.va * d.volume;
}
// KickDrum::tick (kick.rs:1097-1232)
G_D float kick_tick(KickState& s, const double* tt, const RateCtx& rc) {
  KickCtl& c = s.c;
  const double now = tt[c.k];
  c.k += 1;
#pragma unroll
  for (int i = 0; i < K_NP; i++) smooth_tick(c.cur[i], c.tgt[i], rc.smooth15);
  if (!c.active) return 0.0f;
  kick_live(c);
  const KickDer d = kick_derive(c);
  // the per-sample path carries gliding (FFI-edited) and LFO-routed voices; on the device its additive oscillators use the same
  // ~1-ulp sine under the same drive rule as the time-parallel front end (kernels.cuh KickV::front) — 89 harmonics x ~100
  // instructions of the bit-exact port were two thirds of a gliding kick's tick.  Host builds (tests/emu) keep the exact port.
#ifdef __CUDA_ARCH__
  const KickFront f = d.drive <= 8.0f ? kick_front<true>(c, d, now, rc.sr) : kick_front<false>(c, d, now, rc.sr);
#else
  const KickFront f = kick_front(c, d, now, rc.sr);
#endif
  kick_latch(c, d, now);
  float out = kick_back(s.a, d, f, rc);
  if (!env_active(c.amp_env)) c.active = 0;
  return out;
}

// One span of a call: frames [j0, j1) with settled parameters and no event inside.
struct KickSpan {
  int j0, j1, j_act;     // frames [j0, j_act) tick an active voice; [j_act, j1) output 0 and touch nothing
  uint32_t kbase;        // clock index of frame j is kbase + j
  uint32_t resets, pad;
  KickDer d;
  KickCtl c;             // snapshot at j0 (after live decay re-application)
};
G_HD void kick_plan(KickCtl& c, uint32_t resets, const double* tt, int ja, int jb, KickSpan& sp) {
  sp.j0 = ja; sp.j1 = jb; sp.kbase = c.k - (uint32_t)ja; sp.resets = resets; sp.pad = 0;
  if (!c.active) { sp.j_act = ja; sp.c.os_mode = c.os_mode; c.k += (uint32_t)(jb - ja); return; }
  kick_live(c);
  sp.d = kick_derive(c);
  sp.c = c;
  const uint32_t kb = sp.kbase;
  int jd = env_advance(c.amp_env, tt, kb, ja, jb);
  int je = jd == J_NONE ? jb : jd + 1;
  env_advance(c.pitch_env, tt, kb, ja, je);
  if (sp.d.pma > 0.001f) phasemod_advance(c.pm, tt, kb, ja, je);
  env_advance(c.sub_env, tt, kb, ja, je); env_advance(c.punch_env, tt, kb, ja, je); env_advance(c.click_env, tt, kb, ja, je);
  if (sp.d.noise_amount > 0.001f) env_advance(c.noise_env, tt, kb, ja, je);
  if (jd != J_NONE) c.active = 0;
  sp.j_act = je;
  c.k += (uint32_t)(jb - ja);
}

// =========================================== Snare ===========================================
enum { S_FREQ, S_DECAY, S_BRIGHTNESS, S_VOLUME, S_TONAL, S_NOISE, S_PITCH_DROP, S_TONAL_DECAY, S_TONAL_DECAY_CURVE,
       S_NOISE_DECAY, S_NOISE_TAIL_DECAY, S_FILTER_CUTOFF, S_FILTER_RES, S_XFADE, S_PHASE_MOD, S_OVERDRIVE,
       S_AMP_DECAY, S_AMP_DECAY_CURVE, S_TUNING, S_NP };

struct SnareCtl {
  float cur[S_NP], tgt[S_NP];
  uint32_t filter_type;
  Env tonal_osc_env, noise_osc_env, crack_env, pitch_env, tail_env, tonal_env, main_noise_env, amp_env;
  PhaseMod pm;
  float tonal_vol, noise_vol, crack_vol;   // Oscillator.volume (only refreshed while params move, snare.rs:1052-1055)
  float psm;                               // pitch_start_multiplier
  float velocity;
  uint32_t active;
  uint32_t os_mode;
  uint32_t k;
};
struct SnareAud { Chamb filt; WShaper ws; };
struct SnareState { SnareCtl c; SnareAud a; };
struct SnareDer { float base_frequency, pma, cutoff, res, tonal_mix, noise_mix, drive, va, volume; uint32_t filter_type; };
struct SnareFront { float tonal_out, raw_noise, cne, crack_out, amp; };
enum { SNARE_PLANES = 5 };

// SnareDrum::with_config (snare.rs:769-809); cfg = 18 normalized values in S_* order
G_HD void snare_init(SnareState& s, const float* cfg, uint32_t filter_type, float sr) {
  SnareCtl& c = s.c;
  for (int i = 0; i < 18; i++) { float v = clampf(cfg[i], 0.0f, 1.0f); c.cur[i] = c.tgt[i] = v; }
  c.cur[S_TUNING] = c.tgt[S_TUNING] = 0.5f;
  c.filter_type = filter_type > 3 ? 3 : filter_type;
  env_init(c.tonal_osc_env); env_init(c.noise_osc_env); env_init(c.crack_env); env_init(c.pitch_env);
  env_init(c.tail_env); env_init(c.tonal_env); env_init(c.main_noise_env); env_init(c.amp_env);
  c.tonal_vol = c.noise_vol = c.crack_vol = 1.0f;  // Oscillator::new volume
  c.psm = 1.0f + c.cur[S_PITCH_DROP] * 1.5f;
  c.pm.trig = 0.0; c.pm.active = 0;
  c.velocity = 0.5f; c.active = 0; c.os_mode = 4; c.k = 0;
  chamb_init(s.a.filt, sr, denorm(c.cur[S_FILTER_CUTOFF], 100.0f, 10000.0f), denorm(c.cur[S_FILTER_RES], 0.5f, 10.0f));
  ws_init(s.a.ws, 1.0f, 1.0f);
}

// SnareDrum::trigger_with_velocity (snare.rs:873-1027)
G_HD void snare_trigger(SnareCtl& c, float velocity, double time) {
  c.velocity = clampf(velocity, 0.0f, 1.0f);
  c.active = 1;
  float vel = c.velocity, vel2 = vel * vel;
  float decay_scale = 1.0f - (0.45f * vel2);
  float pitch_decay_scale = 1.0f - (0.5f * vel2);
  float base_decay = denorm(c.cur[S_DECAY], 0.05f, 3.5f);
  float tonal_decay = denorm(c.cur[S_TONAL_DECAY], 0.0f, 3.5f);
  float tonal_decay_curve = denorm(c.cur[S_TONAL_DECAY_CURVE], 0.1f, 10.0f);
  float noise_decay = denorm(c.cur[S_NOISE_DECAY], 0.0f, 3.5f);
  float noise_tail_decay = denorm(c.cur[S_NOISE_TAIL_DECAY], 0.0f, 3.5f);
  float amp_decay = denorm(c.cur[S_AMP_DECAY], 0.0f, 4.0f);
  float amp_decay_curve = denorm(c.cur[S_AMP_DECAY_CURVE], 0.1f, 10.0f);
  float scaled_decay = base_decay * decay_scale;
  c.psm = 1.0f + c.cur[S_PITCH_DROP] * 1.5f;
  float pdt = fminf(scaled_decay * 0.3f * pitch_decay_scale, scaled_decay * 0.25f);
  env_config(c.pitch_env, 0.001f, pdt, 0.0f, pdt * 0.1f);
  c.tonal_vol = clampf(c.cur[S_TONAL], 0.0f, 1.0f);
  env_config(c.tonal_osc_env, 0.001f, 0.001f, 1.0f, scaled_decay * 0.4f);
  c.noise_vol = clampf(c.cur[S_NOISE] * 0.8f, 0.0f, 1.0f);
  env_config(c.noise_osc_env, 0.001f, 0.001f, 1.0f, scaled_decay * 0.3f);
  float cvs = 0.7f + 0.3f * vel;
  c.crack_vol = clampf(c.cur[S_BRIGHTNESS] * 0.4f * cvs, 0.0f, 1.0f);
  env_config(c.crack_env, 0.001f, scaled_decay * 0.2f, 0.0f, scaled_decay * 0.1f);
  float std_ = tonal_decay * decay_scale;
  env_config(c.tonal_env, 0.001f, std_, 0.0f, std_ * 0.2f, CURVE_LINEAR, tonal_decay_curve);
  float snd = noise_decay * decay_scale;
  env_config(c.main_noise_env, 0.001f, snd, 0.0f, snd * 0.2f);
  float stl = noise_tail_decay * decay_scale;
  env_config(c.tail_env, 0.001f, stl, 0.0f, stl * 0.3f);
  float sad = amp_decay * decay_scale;
  env_config(c.amp_env, 0.001f, sad, 0.0f, sad * 0.2f, CURVE_LINEAR, amp_decay_curve);
  env_trigger(c.tonal_osc_env, time); env_trigger(c.noise_osc_env, time); env_trigger(c.crack_env, time);
  env_trigger(c.pitch_env, time); env_trigger(c.tonal_env, time); env_trigger(c.main_noise_env, time);
  env_trigger(c.tail_env, time); env_trigger(c.amp_env, time);
  if (c.cur[S_PHASE_MOD] > 0.001f) { c.pm.trig = time; c.pm.active = 1; }
}

G_HD void snare_event(SnareCtl& c, const VoiceEvent& e, const double* tt, uint32_t& resets) {
  switch (e.kind) {
    case EV_TRIGGER: snare_trigger(c, e.value, tt[c.k]); resets |= RST_TRIGGER; break;
    case EV_SET_TARGET: params_set_target<S_NP>(c.tgt, e.param, e.value); break;
    case EV_SNAP: params_snap<S_NP>(c.cur, c.tgt); break;
    case EV_SET_TIME: c.k = e.aux; break;
    case EV_SET_AUX:
      if (e.param == AUX_SNARE_FILTER_TYPE) { uint32_t t = (uint32_t)e.value; c.filter_type = t > 3 ? 3 : t; }
      else if (e.param == AUX_OVERSAMPLING) c.os_mode = (uint32_t)e.value;
      else if (e.param == AUX_SNARE_PITCH_START) c.psm = e.value;  // SnareDrum::set_config (:820)
      break;
    default: break;
  }
}
G_HD void snare_span_begin(SnareAud& a, const SnareCtl& c, uint32_t resets) {
  if (resets & RST_TRIGGER) { a.filt.low = a.filt.band = 0.0f; }   // noise_filter.reset() (:1026)
  if (a.ws.os.mode != c.os_mode) { a.ws.os.mode = c.os_mode; os_reset(a.ws.os); }
}
G_HD void snare_live(SnareCtl& c) {  // snare.rs:1062-1104
  float vel2 = c.velocity * c.velocity;
  float decay_scale = 1.0f - (0.45f * vel2);
  float pitch_decay_scale = 1.0f - (0.5f * vel2);
  float scaled_decay = denorm(c.cur[S_DECAY], 0.05f, 3.5f) * decay_scale;
  float pdt = fminf(scaled_decay * 0.3f * pitch_decay_scale, scaled_decay * 0.25f);
  c.pitch_env.decay = pdt; c.pitch_env.release = pdt * 0.1f;
  c.tonal_osc_env.release = scaled_decay * 0.4f;
  c.noise_osc_env.release = scaled_decay * 0.3f;
  c.crack_env.decay = scaled_decay * 0.2f; c.crack_env.release = scaled_decay * 0.1f;
  float std_ = denorm(c.cur[S_TONAL_DECAY], 0.0f, 3.5f) * decay_scale;
  c.tonal_env.decay = std_; c.tonal_env.release = std_ * 0.2f;
  float snd = denorm(c.cur[S_NOISE_DECAY], 0.0f, 3.5f) * decay_scale;
  c.main_noise_env.decay = snd; c.main_noise_env.release = snd * 0.2f;
  float stl = denorm(c.cur[S_NOISE_TAIL_DECAY], 0.0f, 3.5f) * decay_scale;
  c.tail_env.decay = stl; c.tail_env.release = stl * 0.3f;
  float sad = denorm(c.cur[S_AMP_DECAY], 0.0f, 4.0f) * decay_scale;
  c.amp_env.decay = sad; c.amp_env.release = sad * 0.2f;
}
G_HD SnareDer snare_derive(const SnareCtl& c) {
  SnareDer d;
  d.base_frequency = denorm(c.cur[S_FREQ], 100.0f, 600.0f) * tuning_to_multiplier(c.cur[S_TUNING]);
  d.pma = c.cur[S_PHASE_MOD];
  d.cutoff = denorm(c.cur[S_FILTER_CUTOFF], 100.0f, 10000.0f);
  d.res = denorm(c.cur[S_FILTER_RES], 0.5f, 10.0f);
  float xfade = c.cur[S_XFADE];
  d.tonal_mix = 1.0f - xfade; d.noise_mix = xfade;
  d.drive = clampf(1.0f + (c.cur[S_OVERDRIVE] * 9.0f), 1.0f, 10.0f);
  d.va = sqrtf(c.velocity);
  d.volume = c.cur[S_VOLUME];
  d.filter_type = c.filter_type;
  return d;
}
template <bool FAST = false> G_HD SnareFront snare_front(const SnareCtl& c, const SnareDer& d, double now, float sr) {
  SnareFront f;
  float pev = env_value(c.pitch_env, now);
  float fm = 1.0f + (c.psm - 1.0f) * pev;
  if (d.pma > 0.001f) {
    float pm = phasemod_value(c.pm, now);
    fm *= 1.0f + (pm * d.pma * 1.0f);
  }
  float tonal_f = d.base_frequency * fm;
  // tonal: osc (sustain-1 envelope) * tonal_env * mix.  The heavy additive sum is skipped whenever any
  // factor of the product is exactly 0 (result would be +-0).
  float idx_t = env_active(c.tonal_osc_env) ? (float)(now - c.tonal_osc_env.trig) * sr : 0.0f;
  float osc_amp = env_value(c.tonal_osc_env, now);
  float tonal_env = env_value(c.tonal_env, now);
  f.tonal_out = 0.0f;
  if (osc_amp != 0.0f && c.tonal_vol != 0.0f && tonal_env != 0.0f && d.tonal_mix != 0.0f)
    f.tonal_out = osc_triangle<FAST>(idx_t, tonal_f, sr) * osc_amp * c.tonal_vol * tonal_env * d.tonal_mix;
  float idx_n = env_active(c.noise_osc_env) ? (float)(now - c.noise_osc_env.trig) * sr : 0.0f;
  float namp = env_value(c.noise_osc_env, now);
  f.raw_noise = 0.0f;
  if (namp != 0.0f && c.noise_vol != 0.0f) f.raw_noise = hash_noise(f32_to_u64_sat(idx_n)) * namp * c.noise_vol;
  float ne = env_value(c.main_noise_env, now);
  float te = env_value(c.tail_env, now);
  f.cne = (ne * 0.7f) + (te * 0.3f);
  float idx_c = env_active(c.crack_env) ? (float)(now - c.crack_env.trig) * sr : 0.0f;
  float camp = env_value(c.crack_env, now);
  f.crack_out = 0.0f;
  if (camp != 0.0f && c.crack_vol != 0.0f) f.crack_out = hash_noise(f32_to_u64_sat(idx_c)) * camp * c.crack_vol;
  f.amp = env_value(c.amp_env, now);
  return f;
}
G_HD void snare_latch(SnareCtl& c, const SnareDer& d, double now) {
  env_latch(c.pitch_env, now);
  if (d.pma > 0.001f) phasemod_latch(c.pm, now);
  env_latch(c.tonal_osc_env, now); env_latch(c.tonal_env, now); env_latch(c.noise_osc_env, now);
  env_latch(c.main_noise_env, now); env_latch(c.tail_env, now); env_latch(c.crack_env, now); env_latch(c.amp_env, now);
}
G_HD bool snare_still_active(const SnareCtl& c) {
  bool classic = env_active(c.tonal_osc_env) || env_active(c.noise_osc_env) || env_active(c.crack_env);
  bool ds = env_active(c.tonal_env) || env_active(c.main_noise_env) || env_active(c.tail_env) || env_active(c.amp_env) || c.pm.active;
  return classic || ds;
}
G_D float snare_back(SnareAud& a, const SnareDer& d, const SnareFront& f, const RateCtx& rc) {
  chamb_set(a.filt, rc.sr, d.cutoff, d.res);
  float filtered = chamb_process(a.filt, f.raw_noise, d.filter_type);
  float noise_out = filtered * f.cne * d.noise_mix;
  float total = f.tonal_out + noise_out + f.crack_out;
  a.ws.drive = d.drive;
  float od = ws_process(a.ws, total);
  return od * f.amp * d.va * d.volume;
}
// SnareDrum::tick (snare.rs:1044-1198)
G_D float snare_tick(SnareState& s, const double* tt, const RateCtx& rc) {
  SnareCtl& c = s.c;
  const double now = tt[c.k];
  c.k += 1;
  bool changing = false;
#pragma unroll
  for (int i = 0; i < S_NP; i++) { smooth_tick(c.cur[i], c.tgt[i], rc.smooth15); changing |= (c.cur[i] != c.tgt[i]); }
  if (!c.active) return 0.0f;
  if (changing) {  // apply_params (:1206-1220)
    float cvs = 0.7f + 0.3f * c.velocity;
    c.tonal_vol = clampf(c.cur[S_TONAL], 0.0f, 1.0f);
    c.noise_vol = clampf(c.cur[S_NOISE] * 0.8f, 0.0f, 1.0f);
    c.crack_vol = clampf(c.cur[S_BRIGHTNESS] * 0.4f * cvs, 0.0f, 1.0f);
  }
  snare_live(c);
  const SnareDer d = snare_derive(c);
#ifdef __CUDA_ARCH__
  const SnareFront f = snare_front<true>(c, d, now, rc.sr);      // as SnareV::front (the snare's waveshaper drive is at most 10)
#else
  const SnareFront f = snare_front(c, d, now, rc.sr);
#endif
  snare_latch(c, d, now);
  float out = snare_back(s.a, d, f, rc);
  if (!snare_still_active(c)) c.active = 0;
  return out;
}
struct SnareSpan {
  int j0, j1, j_act;
  uint32_t kbase;
  uint32_t resets, pad;
  SnareDer d;
  SnareCtl c;
};
G_HD int j_max(int a, int b) { return a > b ? a : b; }
G_HD void snare_plan(SnareCtl& c, uint32_t resets, const double* tt, int ja, int jb, SnareSpan& sp) {
  sp.j0 = ja; sp.j1 = jb; sp.kbase = c.k - (uint32_t)ja; sp.resets = resets; sp.pad = 0;
  if (!c.active) { sp.j_act = ja; sp.c.os_mode = c.os_mode; c.k += (uint32_t)(jb - ja); return; }
  snare_live(c);
  sp.d = snare_derive(c);
  sp.c = c;
  const uint32_t kb = sp.kbase;
  // the voice stays active while ANY envelope (or the phase modulator) is; every envelope is ticked until then,
  // so each can be advanced independently over the whole range and the last one to finish ends the voice.
  Env* envs[8] = {&c.tonal_osc_env, &c.noise_osc_env, &c.crack_env, &c.pitch_env, &c.tail_env, &c.tonal_env, &c.main_noise_env, &c.amp_env};
  int jd = -1;
  for (int i = 0; i < 8; i++) {
    if (!env_active(*envs[i])) continue;
    int j = env_advance(*envs[i], tt, kb, ja, jb);
    jd = j_max(jd, j);
  }
  if (c.pm.active) {
    int j = sp.d.pma > 0.001f ? phasemod_advance(c.pm, tt, kb, ja, jb) : J_NONE;
    jd = j_max(jd, j);
  }
  // jd < 0: nothing was active at j0 — the first tick finds that out and deactivates the voice
  int je;
  if (jd == J_NONE) je = jb;
  else { je = (jd < 0 ? ja : jd) + 1; if (je > jb) je = jb; c.active = 0; }
  sp.j_act = je;
  c.k += (uint32_t)(jb - ja);
}

// =========================================== HiHat2 ===========================================
enum { H_PITCH, H_DECAY, H_ATTACK, H_TONE, H_VOLUME, H_TUNING, H_NP };
struct HatCtl {
  float cur[H_NP], tgt[H_NP];
  uint32_t pink_on, db24;
  MaxEnv2 env;
  float velocity;
  uint32_t k;
};
struct HatAud {
  float mod_phase, main_phase, env_smooth;
  uint32_t active;
  Biquad hp1, hp2;
  Tpt svf;
  uint64_t white;
  Pink pink;
};
struct HatState { HatCtl c; HatAud a; };
struct HatDer { float pitch_hz, tone_hz, vel035, volume; uint32_t pink_on, db24; MaxEnvK ek; };   // ek = maxenv_k(c.env)
struct HatFront { float env; };
enum { HAT_PLANES = 1 };
G_HD float hat_pitch_hz(float p) { return denorm(p * p, 3500.0f, 10000.0f); }

// HiHat2::with_config (hihat2.rs:354-376); cfg = pitch, decay, attack, tone, volume
G_HD void hat_init(HatState& s, const float* cfg, uint32_t pink_on, uint32_t db24, float sr) {
  HatCtl& c = s.c; HatAud& a = s.a;
  for (int i = 0; i < 5; i++) { float v = clampf(cfg[i], 0.0f, 1.0f); c.cur[i] = c.tgt[i] = v; }
  c.cur[H_TUNING] = c.tgt[H_TUNING] = 0.5f;
  c.pink_on = pink_on; c.db24 = db24;
  c.env.target[0] = c.env.target[1] = 0; c.env.dur[0] = c.env.dur[1] = 0; c.env.curve[0] = c.env.curve[1] = 0;
  c.env.seg_start = 0.0; c.env.seg_start_val = 0; c.env.cur_val = 0; c.env.seg = 2; c.env.active = 0;  // MaxCurveEnvelope::new(vec![])
  c.velocity = 1.0f; c.k = 0;
  a.mod_phase = a.main_phase = 0.0f; a.env_smooth = 0.0f; a.active = 0;
  hp_init(a.hp1, sr); hp_init(a.hp2, sr);
  tpt_init(a.svf, sr, denorm(c.cur[H_TONE], 500.0f, 10000.0f), 0.5f);
  a.white = XS_SEED;
  pink_reset(a.pink);
}
G_HD void hat_trigger(HatCtl& c, float velocity, double time) {  // :434-451
  c.velocity = clampf(velocity, 0.0f, 1.0f);
  float attack_ms = denorm(c.cur[H_ATTACK], 0.5f, 200.0f);
  float decay_ms = denorm(c.cur[H_DECAY], 0.5f, 4000.0f);
  maxenv_init(c.env, 1.0f, attack_ms, -0.3f, 0.0f, decay_ms, -0.8f);
  maxenv_trigger(c.env, time);
}
G_HD void hat_event(HatCtl& c, const VoiceEvent& e, const double* tt, uint32_t& resets) {
  switch (e.kind) {
    case EV_TRIGGER: hat_trigger(c, e.value, tt[c.k]); resets |= RST_TRIGGER; break;
    case EV_SET_TARGET: params_set_target<H_NP>(c.tgt, e.param, e.value); break;
    case EV_SNAP: params_snap<H_NP>(c.cur, c.tgt); break;
    case EV_SET_TIME: c.k = e.aux; break;
    case EV_SET_AUX:
      if (e.param == AUX_HAT_PINK) c.pink_on = e.value != 0.0f;
      else if (e.param == AUX_HAT_DB24) c.db24 = e.value != 0.0f;
      break;
    default: break;
  }
}
G_HD void hat_span_begin(HatAud& a, const HatCtl&, uint32_t resets) {
  if (resets & RST_TRIGGER) {
    a.active = 1;
    a.env_smooth = 0.0f;
    a.mod_phase = a.main_phase = 0.0f;
    biquad_reset(a.hp1); biquad_reset(a.hp2);
    a.svf.ic1 = a.svf.ic2 = 0.0f;
  }
}
G_HD void hat_live(HatCtl& c) {  // hihat2.rs:460-463
  maxenv_set_dur_ms(c.env, 0, denorm(c.cur[H_ATTACK], 0.5f, 200.0f));
  maxenv_set_dur_ms(c.env, 1, denorm(c.cur[H_DECAY], 0.5f, 4000.0f));
}
G_HD HatDer hat_derive(const HatCtl& c) {
  HatDer d;
  d.pitch_hz = hat_pitch_hz(c.cur[H_PITCH]) * tuning_to_multiplier(c.cur[H_TUNING]);
  d.tone_hz = denorm(c.cur[H_TONE], 500.0f, 10000.0f);
  d.vel035 = c.velocity;
  d.volume = c.cur[H_VOLUME];
  d.pink_on = c.pink_on; d.db24 = c.db24;
  d.ek = maxenv_k(c.env);   // after hat_live: the durations are current
  return d;
}
G_HD HatFront hat_front(const HatCtl& c, const HatDer& d, double now, float) { HatFront f; f.env = maxenv_value_pure(c.env, d.ek, now); return f; }
G_D float hat_osc(float& phase_cycle, float freq, float sr, float pm) {  // PhaseModOsc::tick (:277-286); set_frequency floors at 0
  float inc = fmaxf(freq, 0.0f) / sr;
  phase_cycle = fmodf(phase_cycle + inc, 1.0f);
  float ph = phase_cycle + pm;
  ph -= floorf(ph);
  return gm::g_sinf(2.0f * PI_F * ph);
}
// everything of HiHat2::tick after the envelope value (hihat2.rs:466-508); env_complete = maxenv_complete after this tick
G_D float hat_back(HatAud& a, const HatDer& d, const HatFront& f, bool env_complete, const RateCtx& rc) {
  const float sr = rc.sr;
  float noise;
  if (d.pink_on) noise = pink_tick(a.pink, rc.pink);
  else { float n = u64_to_f32(xorshift64s_next(a.white)) / 18446744073709551616.0f; noise = (n * 2.0f) - 1.0f; }
  float mod_out = hat_osc(a.mod_phase, d.pitch_hz * 0.1f, sr, noise * 0.25f);
  float main_out = hat_osc(a.main_phase, d.pitch_hz, sr, mod_out * 0.75f);
  hp_set(a.hp1, sr, d.pitch_hz, 1.0f);
  float filtered = biquad_process(a.hp1, main_out);
  if (d.db24) { hp_set(a.hp2, sr, d.pitch_hz, 1.0f); filtered = biquad_process(a.hp2, filtered) * 0.8f; }
  float env = f.env;
  if (env >= a.env_smooth) a.env_smooth = env; else a.env_smooth += rc.asym_down * (env - a.env_smooth);
  env = a.env_smooth;
  float out = filtered * env * d.vel035 * 0.35f;
  tpt_set(a.svf, sr, d.tone_hz, 0.5f);
  float lo, bd, hi;
  tpt_process(a.svf, out, lo, bd, hi);
  float o = hi * d.volume;
  if (env_complete && a.env_smooth < 1e-4f) a.active = 0;
  return o;
}
// HiHat2::tick (hihat2.rs:453-508)
G_D float hat_tick(HatState& s, const double* tt, const RateCtx& rc) {
  HatCtl& c = s.c;
  const double now = tt[c.k];
  c.k += 1;
#pragma unroll
  for (int i = 0; i < H_NP; i++) smooth_tick(c.cur[i], c.tgt[i], rc.smooth15);
  if (!s.a.active) return 0.0f;
  hat_live(c);
  const HatDer d = hat_derive(c);
  HatFront f;
  f.env = maxenv_value(c.env, now);
  return hat_back(s.a, d, f, maxenv_complete(c.env), rc);
}
struct HatSpan {
  int j0, j1, j_env;     // frames [j0, j_env) read the envelope plane; from j_env on the envelope is complete (value env_final)
  uint32_t kbase;
  uint32_t resets; float env_final;
  HatDer d;
  HatCtl c;
};
G_HD void hat_plan(HatCtl& c, uint32_t resets, const double* tt, int ja, int jb, HatSpan& sp) {
  sp.j0 = ja; sp.j1 = jb; sp.kbase = c.k - (uint32_t)ja; sp.resets = resets;
  hat_live(c);   // idempotent; an inactive voice's envelope is complete or empty, so the durations do not matter
  sp.d = hat_derive(c);
  sp.c = c;
  int jc = maxenv_complete_frame(c.env, tt, sp.kbase, ja, jb);   // first frame whose tick completes the envelope
  sp.j_env = jc;
  sp.env_final = jc < jb ? maxenv_value_pure(sp.c.env, tt[sp.kbase + (uint32_t)jc]) : 0.0f;
  if (jb > ja) maxenv_value(c.env, tt[sp.kbase + (uint32_t)(jb - 1)]);   // state after the range == state after its last frame
  c.k += (uint32_t)(jb - ja);
}

// =========================================== Tom2 ===========================================
enum { T_TUNE, T_BEND, T_TONE, T_COLOR, T_DECAY, T_MEMBRANE, T_MEMBRANE_Q, T_VOLUME, T_TUNING, T_NP };
struct TomCtl {
  float p[T_NP];      // plain f32 parameters, 0-100 (tuning 0-1), applied instantly (tom2.rs:66-79)
  uint32_t trig_k;    // clock index of the last trigger (MorphOsc noise counter = k - trig_k + 1)
  MaxEnv2 env;
  float mem_q_scale, mem_gain_scale;
  uint32_t mem_dirty; // membrane filter coefficients must be refreshed (update_membrane_params)
  float saved_freq; uint32_t has_saved;
  uint32_t k;
};
struct TomAud {
  // MorphOsc (gen/morph_osc.rs)
  float main_sine_phase, mtri_phase, fixed_sine_phase, rand_phase, rand_current, rand_target, gated_sine_phase;
  float tri_phase;
  uint32_t click_pos, click_playing;
  uint32_t past_attack, main_done, active, tri_enabled;
  float ring_level;
  uint32_t pad0;
  Biquad bp;
  Biquad mem[5];
};
struct TomState { TomCtl c; TomAud a; };
struct TomDer {
  float base_frequency, bend_scaled, tone, mix_control, rand_freq, fq, membrane, mm, vol;
  float w1, w2, w3;
  MaxEnvK ek;   // maxenv_k(c.env)
};
struct TomFront { float env, noise, rnd; };
enum { TOM_PLANES = 3 };
#ifdef __CUDACC__
__constant__ float c_tom_impulse[64] = {
#else
static const float c_tom_impulse[64] = {
#endif
    0.884058f, 0.942029f, 0.913043f, 0.869565f, 0.833333f, 0.797101f, 0.772947f, 0.748792f, 0.724638f,
    0.695652f, 0.666667f, 0.637681f, 0.619565f, 0.601449f, 0.583333f, 0.565217f, 0.536232f, 0.507246f,
    0.478261f, 0.449275f, 0.42029f,  0.391304f, 0.371981f, 0.352657f, 0.333333f, 0.304348f, 0.275362f,
    0.23913f,  0.202899f, 0.181159f, 0.15942f,  0.137681f, 0.115942f, 0.101449f, 0.086957f, 0.072464f,
    0.057971f, 0.043478f, 0.028986f, 0.014493f, 0.009662f, 0.004831f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f,
    0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.014493f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};

// MembraneResonator::update_filters (membrane_resonator.rs:87-93)
G_HD void tom_membrane_update(Biquad* mem, float q_scale, float gain_scale, float sr) {
  const float P[5][3] = {{275.0f, 165.0f, 376.0f}, {220.0f, 228.0f, 205.0f}, {79.0f, 294.0f, 143.0f}, {65.0f, 320.0f, 129.0f}, {57.0f, 326.0f, 141.0f}};
  for (int i = 0; i < 5; i++) {
    float sq = clampf(P[i][2] * q_scale, 0.1f, 100.0f);
    float sg = P[i][0] * gain_scale;
    bp_set(mem[i], sr, P[i][1], sq, sg);
  }
}
// Tom2::update_membrane_params (tom2.rs:405-411): set_q_scale then set_gain_scale, each followed by update_filters.
// The intermediate update uses the OLD gain scale with the new q scale; bp_set's change thresholds make that
// observable in principle, so both steps are replayed on the audio side (tom_span_begin).
G_HD void tom_update_membrane_params(TomCtl& c) {
  float qs = 0.005f + (c.p[T_MEMBRANE_Q] / 100.0f) * 0.015f;
  c.mem_q_scale = clampf(qs, 0.001f, 1.0f);
  c.mem_gain_scale = clampf(0.003f, 0.0001f, 0.1f);
  c.mem_dirty = 1;
}
// Tom2::new (tom2.rs:199-235), then optional set_config (:413-423) with cfg (0-100 units) if cfg != nullptr
G_HD void tom_init(TomState& s, const float* cfg, float sr) {
  TomCtl& c = s.c; TomAud& a = s.a;
  c.p[T_TUNE] = 50.0f; c.p[T_BEND] = 30.0f; c.p[T_TONE] = 50.0f; c.p[T_COLOR] = 50.0f; c.p[T_DECAY] = 50.0f;
  c.p[T_MEMBRANE] = 0.0f; c.p[T_MEMBRANE_Q] = 50.0f; c.p[T_VOLUME] = 100.0f; c.p[T_TUNING] = 0.5f;
  c.trig_k = 0;
  maxenv_init(c.env, 1.0f, 1.0f, 0.8f, 0.0f, 2000.0f, -0.83f);
  c.saved_freq = 0.0f; c.has_saved = 0; c.k = 0;
  a.main_sine_phase = a.mtri_phase = a.fixed_sine_phase = a.rand_phase = a.rand_current = a.rand_target = a.gated_sine_phase = 0.0f;
  a.tri_phase = 0.0f; a.click_pos = 0; a.click_playing = 0;
  a.past_attack = 0; a.main_done = 0; a.active = 0; a.tri_enabled = 1; a.ring_level = 0.0f; a.pad0 = 0;
  bp_init(a.bp, sr);
  for (int i = 0; i < 5; i++) bp_init(a.mem[i], sr);
  // MembraneResonator::with_params(q 0.01, gain 0.0031) then Tom2::new's update_membrane_params
  tom_membrane_update(a.mem, 0.01f, 0.0031f, sr);
  tom_update_membrane_params(c);
  tom_membrane_update(a.mem, c.mem_q_scale, 0.0031f, sr);
  tom_membrane_update(a.mem, c.mem_q_scale, c.mem_gain_scale, sr);
  c.mem_dirty = 0;
  if (cfg) {
    for (int i = 0; i < 8; i++) c.p[i] = cfg[i];
    tom_update_membrane_params(c);
    tom_membrane_update(a.mem, c.mem_q_scale, c.mem_gain_scale, sr);  // gain scale already 0.003: the two updates coincide
    c.mem_dirty = 0;
  }
}
G_HD void tom_trigger(TomCtl& c, double time) {  // :428-448 (velocity ignored)
  c.trig_k = c.k;
  float decay_ms = 0.5f + (c.p[T_DECAY] / 100.0f) * (4000.0f - 0.5f);
  maxenv_init(c.env, 1.0f, 1.0f, 0.8f, 0.0f, decay_ms, -0.83f);
  maxenv_trigger(c.env, time);
}
G_HD void tom_event(TomCtl& c, const VoiceEvent& e, const double* tt, uint32_t& resets) {
  switch (e.kind) {
    case EV_TRIGGER: tom_trigger(c, tt[c.k]); resets |= RST_TRIGGER; break;
    case EV_SET_TARGET:  // value already in the voice's internal units (0-100; tuning 0-1)
      if (e.param < T_NP) {
        {
          const float nv = e.param == T_TUNING ? clampf(e.value, 0.0f, 1.0f) : clampf(e.value, 0.0f, 100.0f);
#pragma unroll
          for (int i = 0; i < T_NP; i++) if ((uint32_t)i == e.param) c.p[i] = nv;
        }
        if (e.param == T_MEMBRANE_Q) tom_update_membrane_params(c);
      }
      break;
    case EV_SET_TIME: c.trig_k = e.aux - (c.k - c.trig_k); c.k = e.aux; break;   // keeps the MorphOsc counter running
    case EV_NOTE_FREQ:   // get_freq_param() = tune (0-100); set_param(0, v) = clamp01(v)*100 (ffi.rs:131-137, 213-217)
      if (!c.has_saved) { c.saved_freq = c.p[T_TUNE]; c.has_saved = 1; }
      c.p[T_TUNE] = clampf(clampf(e.value, 0.0f, 1.0f) * 100.0f, 0.0f, 100.0f);
      break;
    case EV_RESTORE_FREQ:
      if (c.has_saved) { c.has_saved = 0; c.p[T_TUNE] = clampf(clampf(c.saved_freq, 0.0f, 1.0f) * 100.0f, 0.0f, 100.0f); }
      break;
    case EV_SET_AUX:
      if (e.param >= AUX_TOM_RAW_PARAM0 && e.param < AUX_TOM_RAW_PARAM0 + 8) {  // set_config: unclamped
#pragma unroll
        for (int i = 0; i < 8; i++) if ((uint32_t)i == e.param - AUX_TOM_RAW_PARAM0) c.p[i] = e.value;
      }
      else if (e.param == AUX_TOM_CONFIG_DONE) tom_update_membrane_params(c);
      break;
    default: break;
  }
}
G_HD void tom_span_begin(TomAud& a, float mem_q_scale, float mem_gain_scale, uint32_t mem_dirty, uint32_t resets, float sr) {
  if (mem_dirty) tom_membrane_update(a.mem, mem_q_scale, mem_gain_scale, sr);
  if (resets & RST_TRIGGER) {
    a.active = 1; a.past_attack = 0;
    a.main_sine_phase = a.mtri_phase = a.fixed_sine_phase = a.rand_phase = a.rand_current = a.rand_target = a.gated_sine_phase = 0.0f;
    a.click_pos = 0; a.click_playing = 1;
    a.tri_phase = 0.0f;
    biquad_reset(a.bp);
    for (int i = 0; i < 5; i++) biquad_reset(a.mem[i]);
    a.ring_level = 0.0f;
    a.main_done = 0;
  }
}
G_HD TomDer tom_derive(const TomCtl& c) {
  TomDer d;
  float tn = c.p[T_TUNE] / 100.0f;
  d.base_frequency = (40.0f + (tn * tn) * (600.0f - 40.0f)) * tuning_to_multiplier(c.p[T_TUNING]);
  d.bend_scaled = (c.p[T_BEND] / 100.0f) * 2.0f;
  float tone = c.p[T_TONE], color = c.p[T_COLOR];
  d.tone = tone;
  d.mix_control = (tone / 100.0f) * 2.0f - 1.0f;
  float color_midi = 30.0f + (color / 100.0f) * 20.0f;
  float cf1 = 440.0f * gm::g_powf(2.0f, (color_midi - 69.0f) / 12.0f);
  d.rand_freq = 440.0f * gm::g_powf(2.0f, (cf1 - 69.0f) / 12.0f);
  float cn = color / 100.0f;
  d.fq = 1.0f + cn * cn;
  d.membrane = c.p[T_MEMBRANE];
  d.mm = d.membrane / 100.0f;
  d.vol = c.p[T_VOLUME] / 100.0f;
  d.w1 = clampf(-d.mix_control, 0.0f, 1.0f); d.w2 = clampf(1.0f - fabsf(d.mix_control), 0.0f, 1.0f); d.w3 = clampf(d.mix_control, 0.0f, 1.0f);
  d.ek = maxenv_k(c.env);
  return d;
}
// pure part: envelope value and the two SipHash draws keyed by the MorphOsc counter (= frames since the trigger + 1)
G_HD TomFront tom_front(const TomCtl& c, const TomDer& d, double now, uint32_t k) {
  TomFront f;
  f.env = maxenv_value_pure(c.env, d.ek, now);
  uint64_t counter = (uint64_t)(k - c.trig_k) + 1ull;
  f.noise = hash_noise(counter);
  f.rnd = hash_noise(counter + 0x12345678ull);
  return f;
}
G_D void phase_advance(float& ph, float f, float sr) { ph += f / sr; if (ph >= 1.0f) ph -= 1.0f; }
G_D float tri_wave(float ph) { float t = fract(ph); return t < 0.5f ? 4.0f * t - 1.0f : 3.0f - 4.0f * t; }
G_D float unit_sine(float ph) { return gm::g_sinf(ph * 2.0f * PI_F); }

// Tom2::tick (tom2.rs:450-585) with MorphOsc::tick (morph_osc.rs:137-202) inlined; env_complete = maxenv_complete after this tick
G_D float tom_back(TomAud& a, const TomDer& d, const TomFront& f, bool env_complete, const RateCtx& rc) {
  const float sr = rc.sr;
  float env = f.env;
  if (env > 0.9f) a.past_attack = 1;
  float eb = env * d.bend_scaled;
  float raw_freq = d.base_frequency * (1.0f + eb * eb);
  if (env_complete || (a.past_attack && raw_freq < 20.0f)) a.main_done = 1;
  if (a.main_done && !(a.ring_level > 0.0001f)) { a.active = 0; return 0.0f; }
  float fade = (a.past_attack && raw_freq < 40.0f) ? (raw_freq - 20.0f) / (40.0f - 20.0f) : 1.0f;
  float mf = fmaxf(raw_freq, 40.0f);
  float click = 0.0f;
  if (a.click_playing) {
    if (a.click_pos >= 64) a.click_playing = 0;
    else { click = c_tom_impulse[a.click_pos]; a.click_pos += 1; if (a.click_pos >= 64) a.click_playing = 0; }
  }
  float click_out = click * 1.1f;
  float tri_out = a.tri_enabled ? tri_wave(a.tri_phase) * 0.5f : 0.0f;
  phase_advance(a.tri_phase, mf, sr);
  // MorphOsc::tick
  float main_sine = unit_sine(a.main_sine_phase) * 0.5f;
  phase_advance(a.main_sine_phase, mf, sr);
  float mtri = tri_wave(a.mtri_phase) * 0.5f;
  phase_advance(a.mtri_phase, mf, sr);
  float fixed_sine = unit_sine(a.fixed_sine_phase) * 0.5f;
  phase_advance(a.fixed_sine_phase, 190.0f, sr);
  float noise = f.noise * 0.2f;
  float prev = a.rand_phase;
  phase_advance(a.rand_phase, d.rand_freq, sr);
  if (a.rand_phase < prev) { a.rand_current = a.rand_target; a.rand_target = f.rnd; }
  float rand_value = a.rand_current + (a.rand_target - a.rand_current) * a.rand_phase;
  float noise_combined = (noise + rand_value) * 0.4f;
  float gated = d.tone < 99.0f ? unit_sine(a.gated_sine_phase) * 0.2f : 0.0f;
  phase_advance(a.gated_sine_phase, mf, sr);
  float ch1 = main_sine * fixed_sine, ch2 = mtri + noise_combined, ch3 = noise_combined + gated;
  float morph_out = ch1 * d.w1 + ch2 * d.w2 + ch3 * d.w3;
  float mixed = click_out + tri_out + morph_out;
  float ff = fmaxf(mf, 20.0f);
  bp_set(a.bp, sr, ff, d.fq, 1.1f);
  float filtered = biquad_process(a.bp, mixed);
  float mem_out = 0.0f;
  if (d.membrane > 0.0f) {  // MembraneResonator::process (membrane_resonator.rs:189-200)
    float mi = a.main_done ? 0.0f : filtered * env;
    float acc = 0.0f;
#pragma unroll
    for (int i = 0; i < 5; i++) acc += biquad_process(a.mem[i], mi);
    float clipped = gm::g_tanhf(acc);
    a.ring_level = a.ring_level * 0.999f + fabsf(clipped) * 0.001f;
    mem_out = clipped;
  }
  if (a.main_done) {
    float fd = a.ring_level >= 0.005f ? 1.0f : (a.ring_level <= 0.0001f ? 0.0f : (a.ring_level - 0.0001f) / (0.005f - 0.0001f));
    return mem_out * d.mm * fd * 0.7f * d.vol;
  }
  float dry_gain = 1.0f - d.mm;
  float dry = filtered * env;
  float fs = dry * dry_gain + mem_out * d.mm;
  return fs * fade * 0.7f * d.vol;
}
G_D float tom_tick(TomState& s, const double* tt, const RateCtx& rc) {
  TomCtl& c = s.c;
  const uint32_t k = c.k;
  const double now = tt[k];
  c.k += 1;
  if (!s.a.active) return 0.0f;
  const TomDer d = tom_derive(c);
  TomFront f;
  f.env = maxenv_value(c.env, now);
  uint64_t counter = (uint64_t)(k - c.trig_k) + 1ull;
  f.noise = hash_noise(counter);
  f.rnd = hash_noise(counter + 0x12345678ull);
  return tom_back(s.a, d, f, maxenv_complete(c.env), rc);
}
struct TomSpan {
  int j0, j1, j_env;
  uint32_t kbase;
  uint32_t resets; float env_final;
  float mem_q_scale, mem_gain_scale; uint32_t mem_dirty, pad;
  TomDer d;
  TomCtl c;
};
G_HD void tom_plan(TomCtl& c, uint32_t resets, const double* tt, int ja, int jb, TomSpan& sp) {
  sp.j0 = ja; sp.j1 = jb; sp.kbase = c.k - (uint32_t)ja; sp.resets = resets;
  sp.mem_q_scale = c.mem_q_scale; sp.mem_gain_scale = c.mem_gain_scale; sp.mem_dirty = c.mem_dirty; sp.pad = 0;
  c.mem_dirty = 0;
  sp.d = tom_derive(c);
  sp.c = c;
  int jc = maxenv_complete_frame(c.env, tt, sp.kbase, ja, jb);
  sp.j_env = jc;
  sp.env_final = jc < jb ? maxenv_value_pure(sp.c.env, tt[sp.kbase + (uint32_t)jc]) : 0.0f;
  if (jb > ja) maxenv_value(c.env, tt[sp.kbase + (uint32_t)(jb - 1)]);
  c.k += (uint32_t)(jb - ja);
}

}  // namespace gd
