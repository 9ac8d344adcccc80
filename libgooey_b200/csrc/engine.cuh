// engine.cuh — host side of the engine-level path: the reference's GooeyEngine (src/ffi.rs:670-1541) restated as a
// thin host object whose audio state lives in device pools, plus the batch renderer that drives thousands of them in
// one pass: host-resolved sequencer schedule -> per-voice event tables -> voice kernels (kernels.cuh / wave.cuh) ->
// mix kernel (mix.cuh: strips, pan, MixerGraph, master gain, global effect chain, limiter, stereo / mono write-out).
#pragma once
#include <chrono>
#include <cmath>
#include <memory>
#include <functional>
#include "pool.cuh"
#include "patch.h"
#include "mix.cuh"
#include "chain.cuh"
#include "loops.cuh"

namespace gh {

// ---- engine/sequencer.rs: the 16th-note step sequencer, host side, event driven ------------------------------------
// Identical arithmetic to Sequencer::tick_with_settings (:883-952): u64 counters, f32 step math, f32::round, the swing
// SmoothedParam ticking once per sample while running.  Instead of ticking every sample it jumps from firing to firing;
// the swing smoother is stepped sample by sample only while it is unsettled.
struct SeqStep { bool enabled = false; float velocity = 1.0f; bool has_note = false; uint8_t note = 0; bool has_blend = false; float bx = 0, by = 0; };
struct SeqFire { uint32_t frame; float velocity; bool has_note; uint8_t note; bool has_blend; float bx, by; };
struct HostSeq {
  float bpm = 120.0f, sr = 44100.0f, sps = 0.0f;
  uint64_t sample_count = 0, next_trigger = 0;
  std::vector<SeqStep> pattern;
  size_t current_step = 0;
  bool running = false;
  float sw_cur = 0.5f, sw_tgt = 0.5f, sw_coeff = 1.0f;
  static float calc_sps(float bpm, float sr) { float s16 = (60.0f / bpm) / 4.0f; return s16 * sr; }   // :583-588
  void init(float bpm_, float sr_) { bpm = bpm_; sr = sr_; sps = calc_sps(bpm, sr); pattern.assign(16, SeqStep()); sw_coeff = gd::smooth_coeff(sr, 15.0f); }
  void set_bpm(float b) { bpm = b; sps = calc_sps(b, sr); }
  void set_swing(float s) { float c = gd::clampf(s, 0.0f, 1.0f); if (fabsf(sw_tgt - c) > 1e-8f) sw_tgt = c; }
  void start() { running = true; next_trigger = sample_count; }
  void stop() { running = false; }
  void reset() { sample_count = 0; next_trigger = 0; current_step = 0; }
  void set_beat_position(double beat) {   // :658-682 (a step is a 16th note = 1/4 beat); `start()` afterwards fires the landing step
    const size_t n = pattern.size();
    if (n == 0) return;
    const double step_f = beat * 4.0, fl = floor(step_f), frac = step_f - fl;
    current_step = (size_t)fl % n;
    const double off = frac * (double)sps;
    sample_count = off <= 0.0 ? 0 : (uint64_t)off;
    const double nt = round((double)sps - frac * (double)sps);
    next_trigger = nt <= 0.0 ? 0 : (uint64_t)nt;
  }
  void swing_ticks(uint64_t n) { while (n > 0 && sw_cur != sw_tgt) { gd::smooth_tick(sw_cur, sw_tgt, sw_coeff); n--; } }
  void run(uint32_t frames, std::vector<SeqFire>& out) {
    uint32_t f = 0;
    while (f < frames) {
      if (!running || pattern.empty()) { sample_count += frames - f; return; }
      const uint64_t wait = next_trigger > sample_count ? next_trigger - sample_count : 0;
      if (wait >= (uint64_t)(frames - f)) { swing_ticks(frames - f); sample_count += frames - f; return; }
      swing_ticks(wait);
      sample_count += wait; f += (uint32_t)wait;
      swing_ticks(1);
      const SeqStep& st = pattern[current_step];
      if (st.enabled) out.push_back({f, st.velocity, st.has_note, st.note, st.has_blend, st.bx, st.by});
      current_step = (current_step + 1) % pattern.size();
      const float swing_offset = (sw_cur - 0.5f) * 2.0f * sps;
      const float signed_off = (current_step % 2 == 1) ? swing_offset : -swing_offset;
      const float nx = roundf((float)next_trigger + sps + signed_off);
      next_trigger = gd::f32_to_u64_sat(nx);
      sample_count += 1; f += 1;
    }
  }
};

// ---- sampler-rack patterns on the mixer's transport (host side; needs no device) -----------------------------------------------------
// The clip-grid transport as far as the racks need it (clip_grid.rs:144-195, 526-579, 656-660): a beat clock that advances by
// bpm / (60 sr) per rendered frame while running — accumulated add by add like the reference, but only when somebody looks (`lazy` =
// frames rendered since the last look), so batches that never query it pay nothing.
struct Transport {
  bool running = false; double beat = 0.0; float bpm = 120.0f, sr = 44100.0f; uint64_t lazy = 0;
  double beats_per_sample() const { return (double)fmaxf(bpm, 0.0f) / (60.0 * (double)fmaxf(sr, 1.0f)); }
  double now() { const double bps = beats_per_sample(); for (; lazy; lazy--) beat += bps; return beat; }
  void set_bpm(float b) { if (std::isfinite(b) && b > 0.0f) { now(); bpm = b; } }    // ClipGrid::set_bpm (:520-524): beats so far at the old tempo
  double quantized_target(double interval) {                                         // :174-191: strictly the NEXT boundary once running
    if (!running) return 0.0;
    const double scaled = now() / interval, nearest = round(scaled);
    const double base = fabs(scaled - nearest) <= 1.0e-9 ? nearest : floor(scaled);
    return (base + 1.0) * interval;
  }
};
// A rack's 16-step pattern (step note = pad) and its transport-armed start (sampler.rs:160-175, 232-310)
struct RackPattern {
  HostSeq seq;
  bool pattern_running = false, has_pending = false; double pending_beat = 0.0;
};
struct RackHit { uint32_t frame, slot; float velocity; };
// One render call of `frames` frames for the (registered) racks of an engine: `bounce` resets and starts their sequencers first
// (sequencers_iter_mut covers the racks, ffi.rs:3777-3788, 7840-7843); a pending start fires at the first frame whose transport beat has
// reached it (:1139-1147, SamplerRack::activate_start_if_due); from there the rack's sequencer ticks with the others and its fires are
// pad hits (:1199-1210).  The transport advances by the call's frames.
inline void resolve_rack_patterns(Transport& T, RackPattern* const* racks, int n_racks, uint32_t frames, bool bounce, bool triggers_enabled,
                                  std::vector<RackHit>* hits) {
  bool any_pending = false;
  for (int r = 0; r < n_racks; r++) if (racks[r]) { if (bounce) { racks[r]->seq.reset(); racks[r]->seq.start(); } any_pending = any_pending || racks[r]->has_pending; }
  std::vector<uint32_t> act(n_racks, 0xffffffffu);
  if (T.running && any_pending) {
    double beat = T.now();
    const double bps = T.beats_per_sample();
    int left = 0;
    for (int r = 0; r < n_racks; r++) left += (racks[r] && racks[r]->has_pending) ? 1 : 0;
    uint32_t f = 0;
    for (; f < frames && left; f++) {
      for (int r = 0; r < n_racks; r++)
        if (racks[r] && racks[r]->has_pending && act[r] == 0xffffffffu && beat + 1.0e-8 >= racks[r]->pending_beat) { act[r] = f; left--; }
      beat += bps;
    }
    T.beat = beat; T.lazy = frames - f;
  } else if (T.running) T.lazy += frames;
  std::vector<SeqFire> fires;
  for (int r = 0; r < n_racks; r++) {
    if (!racks[r]) continue;
    RackPattern& R = *racks[r];
    uint32_t from = 0;
    if (act[r] != 0xffffffffu) {                       // activate_start_if_due (sampler.rs:266-275)
      R.has_pending = false;
      R.seq.set_beat_position(R.pending_beat); R.seq.start(); R.pattern_running = true;
      from = act[r];
    }
    if (!R.pattern_running) continue;                  // tick_sequencer: the rack's sequencer only ticks while its pattern runs
    fires.clear();
    R.seq.run(frames - from, fires);
    if (triggers_enabled)
      for (const SeqFire& f : fires) hits[r].push_back(RackHit{f.frame + from, f.has_note ? (uint32_t)f.note : 0u, f.velocity});
  }
}

// ---- utils/blendable.rs PresetBlender over the channel's config (ffi.rs ChannelBlender :405-560) ----------------------
// Presets as flat values in the order of the config's fields; preset ids ffi.rs:1882-1998.  Returns the field count (0 = unknown).
inline int preset_flat(uint32_t type, uint32_t id, float* v) {
  static const float KICK[4][18] = {   // KickConfig::{tight,punch,loose,dirt} (kick.rs:257-350)
      {0.22f, 0.00f, 1.00f, 0.00f, 0.12f, 0.70f, 0.01f, 0.85f, 0.64f, 1.00f, 0.07f, 0.01f, 0.02f, 0.20f, 0.00f, 0.47f, 0.12f, 0.02f},
      {0.50f, 0.20f, 1.00f, 0.20f, 0.12f, 0.60f, 0.10f, 0.85f, 0.24f, 1.00f, 0.07f, 0.11f, 0.42f, 0.20f, 0.00f, 0.47f, 0.12f, 0.02f},
      {0.32f, 0.40f, 1.00f, 0.00f, 0.62f, 0.20f, 0.12f, 0.85f, 0.84f, 1.00f, 0.07f, 0.01f, 0.02f, 0.25f, 0.00f, 0.47f, 0.12f, 0.12f},
      {0.62f, 0.10f, 1.00f, 0.10f, 0.10f, 0.60f, 0.10f, 0.85f, 0.44f, 1.00f, 0.20f, 0.10f, 0.82f, 0.20f, 0.00f, 0.47f, 0.10f, 0.10f}};
  const float d = 0.029f;   // SnareConfig::tight() = new(0.2, 0.4, 0.7, 0.5, 0.029, 0.3, 0.8): derived decays in f32 (snare.rs:99-132)
  const float SNARE[4][19] = {   // SnareConfig::{tight,loose,hiss,smack} (snare.rs:270-351), new_full order
      {0.2f, 0.4f, 0.7f, 0.5f, d, 0.3f, 0.8f, d * 0.8f, 0.091f, d * 0.6f, d, 0.495f, 0.053f, 1.0f, 0.5f, 0.0f, 0.0f, 0.125f, 0.02f},
      {0.16f, 0.80f, 0.60f, 0.30f, 0.79f, 0.10f, 0.90f, 0.33f, 0.20f, 0.23f, 0.34f, 0.55f, 0.05f, 1.0f, 0.50f, 0.00f, 0.10f, 0.12f, 0.02f},
      {0.16f, 0.00f, 0.60f, 0.30f, 0.04f, 0.40f, 0.90f, 0.53f, 0.09f, 0.38f, 0.29f, 0.29f, 0.45f, 1.0f, 0.50f, 1.00f, 0.20f, 0.18f, 0.02f},
      {0.2f, 0.3f, 0.8f, 0.0f, 0.029f, 0.3f, 0.85f, 0.014f, 0.091f, 0.034f, 0.086f, 0.293f, 0.158f, 1.0f, 0.4f, 0.5f, 0.0f, 0.125f, 0.02f}};
  static const float HAT[4][7] = {     // HiHat2Config::{short,loose,dark,soft} (hihat2.rs:79-96): pitch, decay, attack, pink, db24, tone, volume
      {0.76f, 0.05f, 0.00f, 0.0f, 1.0f, 1.00f, 1.0f}, {0.76f, 0.30f, 0.00f, 0.0f, 1.0f, 1.00f, 1.0f},
      {0.41f, 0.05f, 0.00f, 0.0f, 1.0f, 0.15f, 1.0f}, {0.41f, 0.05f, 0.15f, 0.0f, 1.0f, 0.60f, 1.0f}};
  static const float TOM[4][8] = {     // Tom2Config::{derp,ring,brush,void_preset} (tom2.rs:119-172)
      {60.0f, 70.0f, 50.0f, 0.0f, 20.0f, 0.0f, 50.0f, 100.0f}, {80.0f, 20.0f, 10.0f, 0.0f, 100.0f, 60.0f, 70.0f, 100.0f},
      {40.0f, 20.0f, 10.0f, 90.0f, 30.0f, 0.0f, 50.0f, 100.0f}, {60.0f, 30.0f, 100.0f, 50.0f, 90.0f, 40.0f, 80.0f, 100.0f}};
  static const float BASS[4][15] = {   // BassConfig::{acid,sub,reese,stab} (bass.rs:188-269)
      {0.24f, 0.40f, 0.80f, 0.00f, 0.00f, 0.10f, 0.15f, 0.70f, 0.85f, 0.15f, 0.08f, 0.35f, 0.10f, 0.30f, 0.80f},
      {0.18f, 1.00f, 0.15f, 0.00f, 0.00f, 0.00f, 0.70f, 0.05f, 0.10f, 0.30f, 0.20f, 0.60f, 0.15f, 0.00f, 0.85f},
      {0.18f, 0.30f, 0.80f, 0.80f, 0.50f, 0.05f, 0.35f, 0.30f, 0.50f, 0.40f, 0.15f, 0.55f, 0.12f, 0.60f, 0.80f},
      {0.30f, 0.20f, 0.90f, 0.00f, 0.00f, 0.90f, 0.20f, 0.40f, 0.90f, 0.08f, 0.05f, 0.20f, 0.08f, 0.20f, 0.80f}};
  if (id > 3) return 0;
  const float* src; int n;
  switch (type) {
    case GOOEY_INSTRUMENT_KICK: src = KICK[id]; n = 18; break;
    case GOOEY_INSTRUMENT_SNARE: src = SNARE[id]; n = 19; break;
    case GOOEY_INSTRUMENT_HIHAT: src = HAT[id]; n = 7; break;
    case GOOEY_INSTRUMENT_TOM: src = TOM[id]; n = 8; break;
    case GOOEY_INSTRUMENT_BASS: src = BASS[id]; n = 15; break;
    default: return 0;
  }
  for (int i = 0; i < n; i++) v[i] = src[i];
  return n;
}
struct ChannelBlender {
  uint32_t type = 0; int n = 0;
  float corner[4][24];                       // bottom_left, bottom_right, top_left, top_right
  uint32_t corner_ids[4] = {0, 1, 2, 3};
  void default_for_type(uint32_t t) { type = t; for (uint32_t c = 0; c < 4; c++) { n = preset_flat(t, c, corner[c]); corner_ids[c] = c; } }
  bool discrete(int i) const { return (type == GOOEY_INSTRUMENT_SNARE && i == 13) || (type == GOOEY_INSTRUMENT_HIHAT && (i == 3 || i == 4)); }
  void lerp(const float* a, const float* b, float t, float* o) const {   // impl Blendable: self * inv_t + other * t, enums switch at t = 0.5
    t = gd::clampf(t, 0.0f, 1.0f);
    volatile float inv_t = 1.0f - t;           // (volatile: keep the two roundings of `a * inv_t + b * t`, no host FMA contraction)
    for (int i = 0; i < n; i++) {
      if (discrete(i)) { o[i] = t < 0.5f ? a[i] : b[i]; continue; }
      volatile float p = a[i] * inv_t, q = b[i] * t;
      o[i] = p + q;
    }
  }
  void blend(float x, float y, float* o) const {   // blendable.rs:73-86
    x = gd::clampf(x, 0.0f, 1.0f); y = gd::clampf(y, 0.0f, 1.0f);
    float bottom[24], top[24];
    lerp(corner[0], corner[1], x, bottom);
    lerp(corner[2], corner[3], x, top);
    lerp(bottom, top, y, o);
  }
  void set_corner_preset(uint32_t c, uint32_t id) { float v[24]; if (c < 4 && preset_flat(type, id, v) > 0) for (int i = 0; i < n; i++) corner[c][i] = v[i]; }
  // `<Voice>::set_config(blend(x, y))` as voice events at `frame` (kick.rs:905-941, snare.rs:818-855, hihat2.rs:382-390, tom2.rs:400-411, bass.rs:636-662)
  template <class Add> void apply(float x, float y, uint32_t frame, Add add) const {
    float v[24];
    blend(x, y, v);
    switch (type) {
      case GOOEY_INSTRUMENT_KICK: for (int i = 0; i < 18; i++) add(make_event(frame, gd::EV_SET_TARGET, i, v[i])); break;
      case GOOEY_INSTRUMENT_SNARE: {
        float cfg[18]; uint32_t ft;
        snare_cfg_from_patch(v, cfg, ft);
        volatile float psm = v[5] * 1.5f;
        add(make_event(frame, gd::EV_SET_AUX, gd::AUX_SNARE_PITCH_START, 1.0f + psm));
        for (int i = 0; i < 18; i++) add(make_event(frame, gd::EV_SET_TARGET, i, cfg[i]));
        add(make_event(frame, gd::EV_SET_AUX, gd::AUX_SNARE_FILTER_TYPE, (float)ft));
      } break;
      case GOOEY_INSTRUMENT_HIHAT:
        add(make_event(frame, gd::EV_SET_TARGET, gd::H_PITCH, v[0])); add(make_event(frame, gd::EV_SET_TARGET, gd::H_DECAY, v[1]));
        add(make_event(frame, gd::EV_SET_TARGET, gd::H_ATTACK, v[2])); add(make_event(frame, gd::EV_SET_TARGET, gd::H_TONE, v[5]));
        add(make_event(frame, gd::EV_SET_TARGET, gd::H_VOLUME, v[6]));
        add(make_event(frame, gd::EV_SET_AUX, gd::AUX_HAT_PINK, v[3])); add(make_event(frame, gd::EV_SET_AUX, gd::AUX_HAT_DB24, v[4]));
        break;
      case GOOEY_INSTRUMENT_TOM:
        for (int i = 0; i < 8; i++) add(make_event(frame, gd::EV_SET_AUX, gd::AUX_TOM_RAW_PARAM0 + i, v[i]));
        add(make_event(frame, gd::EV_SET_AUX, gd::AUX_TOM_CONFIG_DONE, 0.0f));
        break;
      case GOOEY_INSTRUMENT_BASS: for (int i = 0; i < 15; i++) add(make_event(frame, gd::EV_SET_TARGET, i, v[i])); break;
      default: break;
    }
  }
};

// ---- geometry of the delay lines at a sample rate (delay.rs:189, reverb.rs:84-96, plate_reverb.rs:236-262) ----------
inline gd::FxGeom make_fx_geom(float sr) {
  gd::FxGeom g;
  memset(&g, 0, sizeof g);
  g.delay_len = (uint32_t)gd::f32_to_u64_sat(sr * 5.0f) + 1u;
  const float DL[6] = {131, 251, 389, 521, 617, 787}, DR[6] = {127, 263, 397, 541, 631, 797};
  const float scale = sr / 44100.0f;
  uint32_t off = 0;
  for (int i = 0; i < 12; i++) {
    const float base = i < 6 ? DL[i] : DR[i - 6];
    g.spring_len[i] = (uint32_t)gd::f32_to_u64_sat(fmaxf(base * scale, 1.0f));
    g.spring_off[i] = off; off += g.spring_len[i];
  }
  const uint32_t spring_words = off;
  const float sr_scale = sr / 29761.0f;
  g.plate_sr_scale = sr_scale;
  g.plate_excursion = 16.0f * sr_scale;
  auto fixed = [&](float base) { return (uint32_t)gd::f32_to_u64_sat(ceilf(base * sr_scale)) + 4u; };
  auto sized = [&](float base, float head) { return (uint32_t)gd::f32_to_u64_sat(ceilf(base * 2.0f * sr_scale + head)) + 4u; };
  auto cap4 = [](uint32_t c) { return c < 4u ? 4u : c; };
  const float IAD[4] = {142.0f, 107.0f, 379.0f, 277.0f};
  uint32_t caps[13];
  caps[0] = cap4((uint32_t)gd::f32_to_u64_sat(ceilf(200.0f * 0.001f * sr)) + 8u);
  for (int i = 0; i < 4; i++) { caps[1 + i] = cap4(fixed(IAD[i])); g.plate_in_delay[i] = fmaxf(IAD[i] * sr_scale, 1.0f); }
  const float TL[8] = {672.0f, 4453.0f, 1800.0f, 3720.0f, 908.0f, 4217.0f, 2656.0f, 3163.0f};
  for (int i = 0; i < 8; i++) { caps[5 + i] = cap4(sized(TL[i], (i == 0 || i == 4) ? g.plate_excursion : 0.0f)); g.plate_len[i] = TL[i] * sr_scale; }
  off = 0;
  for (int i = 0; i < 13; i++) { g.plate_cap[i] = caps[i]; g.plate_off[i] = off; off += caps[i]; }
  g.plate_lfo_ia = 0.50f / sr; g.plate_lfo_ib = 0.71f / sr;
  g.ring_words[0] = 0; g.ring_words[1] = 2u * g.delay_len; g.ring_words[2] = spring_words; g.ring_words[3] = off;
  return g;
}
inline uint32_t ring_words_of(const gd::FxGeom& g, uint32_t kind) {
  switch (kind) { case gd::FXK_DELAY: return g.ring_words[1]; case gd::FXK_SPRING: return g.ring_words[2]; case gd::FXK_PLATE: return g.ring_words[3];
    case gd::FXK_SATURATION: case gd::FXK_COMPRESSOR: case gd::FXK_WAVESHAPER: case gd::FXK_FBWS: return 2u * gd::OS_WORDS;   // oversampler history, one per channel
    default: return 0; }
}

// ---- everything resident on one device for one sample rate ---------------------------------------------------------
struct EngineBank {
  int device; float sr;
  gd::RateCtx rc; gd::FxGeom geo;
  VoiceBank voices;
  ClockWindow clock;
  Pool<gd::MixState> mix_pool;
  std::vector<gd::MixCfg> cfgs;           // by mix slot (host authoritative)
  DevBuf<gd::MixCfg> d_cfg;
  DevBuf<float> ring[gd::MAX_FX]; uint32_t ring_words[gd::MAX_FX] = {0};
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_piece = nullptr;
  // The mix of piece p runs on its own stream while the voices of piece p + 1 render into the other voice buffer.
  cudaStream_t mix_stream = nullptr;
  cudaEvent_t ev_voices[2] = {nullptr, nullptr}, ev_mixed[2] = {nullptr, nullptr};
  DevBuf<float> d_voice_bufs[2], d_out;
  DevBuf<int16_t> d_pcm;                  // 16-bit PCM of d_out (bounce_to_wav's quantisation done on the device)
  cudaStream_t copy_stream = nullptr;     // drains finished pieces to the host while later pieces render
  DevBuf<float> d_silent;                 // the granulator's 1-sample silent placeholder buffer (ffi.rs:929-933)
  DevBuf<uint32_t> d_mix_slots, d_mix_ev_begins[2];
  DevBuf<uint8_t> d_mix_fast;
  DevBuf<gd::MixConst> d_mix_consts;
  DevBuf<float> d_premix;                 // [2][n_lpad][vstride]: pre-chain stereo mix of the engines whose strips are time-parallel
  DevBuf<gd::LfoStream> d_lfo_streams;    // LFO pool of the current render call
  DevBuf<float> d_lfo_planes;             // [routed streams][frames] LFO values
  std::vector<gd::LfoStream> h_lfo_streams;
  // sample-playback sources (loops.cuh): per-call descriptors (state read back when the call ends) and the pieces' stereo rows
  std::vector<gd::LoopMixer> h_loop_descs; DevBuf<gd::LoopMixer> d_loop_descs;
  std::vector<gd::SamplerRack> h_rack_descs; DevBuf<gd::SamplerRack> d_rack_descs;
  DevBuf<gd::SamplerHit> d_rack_hits;
  DevBuf<float> d_ext[2];
  DevBuf<float> d_hann; uint32_t wsola_hop = 0;    // WSOLA window table of this sample rate (wsola.rs:80-82), built at first use
  // PreservePitch channel: the window table and the channel's own stretcher buffers (9 hops of floats, content irrelevant until the
  // device builds the stretcher) behind the descriptor
  template <class LoopHostT> void attach_stretcher(LoopHostT& l, gd::LoopChan& d) {
    d.hop = 0; d.hann = nullptr; d.st_buf = nullptr;
    if (!d.preserve) return;
    if (!d_hann.p) {
      wsola_hop = gd::wsola_hop_len(sr);
      std::vector<float> h((size_t)2 * wsola_hop);
      for (uint32_t i = 0; i < 2 * wsola_hop; i++) h[i] = gd::wsola_window_coeff(i, 2 * wsola_hop);
      d_hann.alloc(h.size());
      GH_CUDA(cudaMemcpy(d_hann.p, h.data(), h.size() * 4, cudaMemcpyHostToDevice));
    }
    if (!l.stretch) { l.stretch = std::make_shared<DevBuf<float>>(); l.stretch->alloc((size_t)9 * wsola_hop); l.st_valid = false; d.st_valid = 0; }
    d.hop = wsola_hop; d.hann = d_hann.p; d.st_buf = l.stretch->p;
  }
  DevBuf<float> d_peaks;                  // [n][N_PEAKS] maxima of the current render call
  DevBuf<unsigned long long> d_chain_units; unsigned long long h_chain_units = 0;   // engine-frames the settled-chain kernel took in the last render
  std::vector<float> h_peaks;
  DevBuf<gd::VoiceEvent> d_mix_eventss[2];
  std::recursive_mutex mu;   // every use of the bank's shared buffers / streams, held for a whole render call
  KernelTimer mix_timer;                  // the effect mixer of each piece of the last render (on mix_stream)
  void collect_stats() {                  // after the streams have been synchronised
    mix_timer.collect();
    voices.collect_stats();
    if (!h_chain_units) return;
    std::lock_guard<std::mutex> lk(kernel_stats_mutex());
    KernelStat& c = kernel_stats()["chain_fast_kernel"];
    c.launches++; c.voice_frames += (double)h_chain_units; h_chain_units = 0;
  }
  EngineBank(int dev, float sr_) : device(dev), sr(sr_) {
    rc = gd::make_rate_ctx(sr); geo = make_fx_geom(sr);
    GH_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    GH_CUDA(cudaEventCreate(&ev0)); GH_CUDA(cudaEventCreate(&ev1)); GH_CUDA(cudaEventCreateWithFlags(&ev_piece, cudaEventDisableTiming));
    GH_CUDA(cudaStreamCreateWithFlags(&mix_stream, cudaStreamNonBlocking));
    GH_CUDA(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
    for (int b = 0; b < 2; b++) { GH_CUDA(cudaEventCreateWithFlags(&ev_voices[b], cudaEventDisableTiming)); GH_CUDA(cudaEventCreateWithFlags(&ev_mixed[b], cudaEventDisableTiming)); }
    d_silent.alloc(4); d_silent.zero(stream);
  }
  // makes sure arena `slot` holds `words` ring words for `cap` engine slots (content preserving)
  void ensure_ring(int slot, uint32_t words, long long cap) {
    if (words == 0) return;
    if (ring[slot].p && ring_words[slot] >= words && ring_cap_of[slot] >= cap) return;
    const uint32_t nw = std::max(words, ring_words[slot]);
    const long long nc = std::max(cap, ring_cap_of[slot]);
    DevBuf<float> nb;
    nb.alloc((size_t)nw * (size_t)nc);
    GH_CUDA(cudaMemsetAsync(nb.p, 0, (size_t)nw * (size_t)nc * 4, stream));
    if (ring[slot].p && ring_words[slot] > 0)
      GH_CUDA(cudaMemcpy2DAsync(nb.p, (size_t)nc * 4, ring[slot].p, (size_t)ring_cap_of[slot] * 4, (size_t)ring_cap_of[slot] * 4, ring_words[slot], cudaMemcpyDeviceToDevice, stream));
    GH_CUDA(cudaStreamSynchronize(stream));
    std::swap(ring[slot].p, nb.p); std::swap(ring[slot].n, nb.n);
    ring_words[slot] = nw; ring_cap_of[slot] = nc;
  }
  long long ring_cap_of[gd::MAX_FX] = {0};
  std::vector<uint32_t> ring_dirty;       // engine slots re-used since the last render: their ring columns must read as silence
  DevBuf<uint32_t> d_ring_dirty;
  void clear_dirty_rings(cudaStream_t st);
};
EngineBank& engine_bank(int device, float sr);

__global__ void ring_clear_kernel(float* __restrict__ ring, long long cap, uint32_t words, const uint32_t* __restrict__ slots, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t slot = slots[i];
  if ((long long)slot >= cap) return;
  for (uint32_t w = blockIdx.y; w < words; w += gridDim.y) ring[(long long)w * cap + slot] = 0.0f;
}
inline void EngineBank::clear_dirty_rings(cudaStream_t st) {
  if (ring_dirty.empty()) return;
  std::sort(ring_dirty.begin(), ring_dirty.end());          // neighbouring slots -> neighbouring threads -> coalesced rows
  ring_dirty.erase(std::unique(ring_dirty.begin(), ring_dirty.end()), ring_dirty.end());
  d_ring_dirty.upload(ring_dirty.data(), ring_dirty.size(), st);
  const int n = (int)ring_dirty.size();
  for (int s = 0; s < gd::MAX_FX; s++)
    if (ring[s].p && ring_words[s]) {
      ring_clear_kernel<<<dim3((n + 127) / 128, std::min<uint32_t>(ring_words[s], 4096u)), 128, 0, st>>>(ring[s].p, ring_cap_of[s], ring_words[s], d_ring_dirty.p, n);
      g_launches.fetch_add(1, std::memory_order_relaxed);
    }
  GH_CUDA(cudaGetLastError());
  GH_CUDA(cudaStreamSynchronize(st));                       // ring_dirty (host) is reused
  ring_dirty.clear();
}

// An engine's voice channels: the five strips, the poly synth, the granulator.  Channel c renders into row c * n_lpad + engine
// of a render's voice buffer, and its default instrument is the one with id c.
constexpr int N_STRIPS = 5, CH_POLY = 5, CH_GRAN = 6, N_CH = 7;

}  // namespace gh

extern const float GOOEY_POLY_PRESETS[5][14];   // PolySynthConfig presets by ffi preset id (engine_api.cuh)

// ---- the engine handle (opaque to C callers) --------------------------------------------------------------------------
struct GooeyEngine {
  gh::EngineBank* bank = nullptr;
  float sr = 44100.0f, bpm = 120.0f, swing = 0.5f;
  uint32_t k = 0;                       // engine clock index (current_time = tt[k])
  // Every voice channel: its instrument, pool slot and the events queued for the next render.  The strips are always launched.
  // The poly synth's and granulator's FFI calls act immediately in the reference (ffi.rs:5571-5648, 7702-7827); here they
  // queue events that are applied before frame 0 of the next render — the same instant, since nothing ticks in between.
  // These two are only launched once the host has touched them (until then they contribute exactly +0.0).
  struct Voice {
    uint32_t type = 0; int slot = -1;
    bool launched = false;
    std::vector<gd::VoiceEvent> pending;
  } voice[gh::N_CH];
  struct Strip {                        // what only the strips have
    gh::HostSeq seq;
    bool muted = false, soloed = false, trig_pending = false;
    float trig_vel = 1.0f;
    gh::ChannelBlender blender; bool blend_enabled = false; float blend_x = 0.5f, blend_y = 0.5f;   // ffi.rs:598-600
  } strip[gh::N_STRIPS];
  std::shared_ptr<gh::DevBuf<float>> gran_buf;    // may be shared by many engines (gooey_b200_granulator_share_buffer)
  uint32_t gran_len = 1; float gran_sr = 44100.0f;
  int mix_slot = -1;
  gd::MixCfg cfg;
  std::vector<gd::VoiceEvent> mix_pending;
  bool track_muted[gd::MAX_TRACKS] = {false}, track_soloed[gd::MAX_TRACKS] = {false};
  float track_gain_t[gd::MAX_TRACKS], track_pan_t[gd::MAX_TRACKS];     // the strips' targets, for the getters (graph.rs:196-215)
  GooeyEngine() { for (int t = 0; t < gd::MAX_TRACKS; t++) { track_gain_t[t] = 1.0f; track_pan_t[t] = 0.5f; } }
  // LFO pool (ffi.rs:33-54, 716-719, 876-884): eight tempo-synced sine LFOs, disabled, Quarter division, amount 1, offset 0
  struct LfoHost { uint32_t division = 4; float phase = 0.0f, amount = 1.0f, offset = 0.0f; } lfos[8];
  bool lfo_enabled[8] = {false};
  struct LfoRoute { uint32_t id, instrument, param; float depth; };
  std::vector<LfoRoute> lfo_routes[8];
  uint32_t lfo_next_route_id[8] = {0};
  bool seq_triggers_enabled = true;
  // ---- sample-playback sources (loops.cuh; SURVEY.md §8f-4) ----
  // mixer/loop_channel.rs LoopChannel: the buffer lives on the device as two planes (left[len], right[len]); the rest is the
  // reference's struct, edited directly by the gooey_engine_loop_* setters and advanced by the device during a render.
  struct LoopHost {
    std::shared_ptr<gh::DevBuf<float>> buf;
    uint32_t len = 0; float buf_sr = 0.0f;
    bool has_source_bpm = false; float source_bpm = 0.0f;
    double cursor = 0.0;
    float loop_start = 0.0f, loop_end = 1.0f, speed = 1.0f;
    bool playing = false, muted = false, soloed = false;
    uint32_t pitch_mode = 0;
    gd::LSm gain = {1.0f, 1.0f}, active = {1.0f, 1.0f};
    // WsolaStretcher of PitchMode::PreservePitch (loop_channel.rs:141-146): its buffers on the device, its scalars here; dropped
    // (st_valid = false) whenever the cursor is moved from outside so that it re-seeds at the new position
    std::shared_ptr<gh::DevBuf<float>> stretch;
    bool st_valid = false; uint32_t st_have_prev = 0, st_drain = 0; double st_cursor = 0.0;
    // queue_swap (loop_channel.rs:147-156, 413-423): a take staged to replace the buffer at the next grid boundary of the loop
    std::shared_ptr<gh::DevBuf<float>> pend_buf;
    uint32_t pend_len = 0; float pend_sr = 0.0f; bool pend_has_bpm = false; float pend_bpm = 0.0f;
    uint32_t pend_div = 1; bool has_pending = false; uint32_t swaps_completed = 0;
    // fills the playback half of a device descriptor (shared by engines_render and the offline channel render)
    void describe(gd::LoopChan& d, float engine_bpm) const {
      const bool loaded = buf && len > 0;
      d.left = loaded ? buf->p : nullptr; d.right = loaded ? buf->p + len : nullptr;
      d.cursor = cursor; d.len = loaded ? len : 0u; d.buf_sr = buf_sr;
      const bool tagged = has_source_bpm && source_bpm > 0.0f && engine_bpm > 0.0f;               // warp_ratio (loop_channel.rs:282-291)
      const double ratio = tagged ? (double)engine_bpm / (double)source_bpm : 1.0;
      d.warp = pitch_mode == 1 ? ratio : 1.0;                                                      // advance(): Resample mode only (:239-243)
      d.warp_pp = pitch_mode != 0 ? ratio : 1.0;
      d.loop_start = loop_start; d.loop_end = loop_end; d.speed = speed; d.playing = playing ? 1u : 0u;
      d.gain = gain; d.active = active;
      d.preserve = pitch_mode == 2 ? 1u : 0u;
      d.st_valid = st_valid ? 1u : 0u; d.st_have_prev = st_have_prev; d.st_drain = st_drain; d.st_cursor = st_cursor;
      const bool queued = has_pending && pend_buf && pend_len > 0;
      d.has_pending = queued ? 1u : 0u; d.swaps = 0; d.pend_div = pend_div;
      d.pend_left = queued ? pend_buf->p : nullptr; d.pend_right = queued ? pend_buf->p + pend_len : nullptr;
      d.pend_len = queued ? pend_len : 0u; d.pend_buf_sr = pend_sr;
      const double pratio = (pend_has_bpm && pend_bpm > 0.0f && engine_bpm > 0.0f) ? (double)engine_bpm / (double)pend_bpm : 1.0;
      d.pend_warp = pitch_mode == 1 ? pratio : 1.0; d.pend_warp_pp = pitch_mode != 0 ? pratio : 1.0;
    }
    void absorb(const gd::LoopChan& d) {   // the state a render moved
      cursor = d.cursor; gain = d.gain; active = d.active;
      st_valid = d.st_valid != 0; st_have_prev = d.st_have_prev; st_drain = d.st_drain; st_cursor = d.st_cursor;
      if (has_pending && d.swaps) {          // the queued take landed: it is the channel's buffer now
        buf = pend_buf; len = pend_len; buf_sr = pend_sr; has_source_bpm = pend_has_bpm; source_bpm = pend_bpm;
        pend_buf.reset(); pend_len = 0; has_pending = false;
        swaps_completed += d.swaps;
      }
    }
    gd::LoopWindow window() const { return gd::loop_window(loop_start, loop_end, (double)len); }
  } loops[gd::LOOP_CHANNELS];
  float loop_engine_bpm = 120.0f;          // LoopChannel::engine_bpm: written by Mixer::set_bpm only (loop_channel.rs:28, 365-367)
  // instruments/sampler.rs SamplerRack: 16 slots of interleaved PCM on the device, 32 voices (a voice keeps its buffer alive)
  struct SamplerHost {
    bool registered = false;
    struct Slot { std::shared_ptr<gh::DevBuf<float>> buf; uint32_t frames = 0, channels = 0; float sr = 0.0f; } slots[gd::SAMPLER_SLOTS];
    gd::SampleVoice voices[gd::SAMPLER_VOICES];
    std::shared_ptr<gh::DevBuf<float>> voice_buf[gd::SAMPLER_VOICES];
    void voices_release(int v) { voices[v].samples = nullptr; voice_buf[v].reset(); }
    void stop_all() { for (int v = 0; v < gd::SAMPLER_VOICES; v++) voices_release(v); }
    // the rack's 16-step pattern (step note = pad) and its transport-armed start (sampler.rs:160-175, 232-310)
    gh::RackPattern pat;
    unsigned long long next_age = 0;
    SamplerHost() { memset(voices, 0, sizeof voices); for (auto& v : voices) v.increment = 1.0; }
  } samplers[gd::SAMPLER_RACKS];
  // the mixer's transport (the beat clock sampler-rack pattern starts are armed on)
  gh::Transport transport;
  float peaks[gd::N_PEAKS] = {0};          // read-and-reset meters (ffi.rs:2572-2584, graph.rs:233-237), merged after every render
  struct MidiEvent { uint32_t instrument_index; float velocity; uint32_t sample_offset; };   // GooeyMidiEvent (ffi.rs:78-83)
  std::vector<MidiEvent> midi_events;      // of the most recent render call, at most 64 (ffi.rs:71, 994-1004, 1045)
  bool has_error = false;
  std::string error;
  void (*error_cb)(void*, const char*) = nullptr; void* error_ctx = nullptr;
  bool error_cb_fired = false;
};

namespace gh {

struct BadBatch : std::runtime_error { using std::runtime_error::runtime_error; };   // caller error, not a device failure

inline void engine_fail(GooeyEngine* e, const std::string& msg) {   // sticky error + one-shot callback (ffi.rs:2236-2284)
  if (!e) return;
  if (!e->has_error) { e->has_error = true; e->error = msg; }
  if (e->error_cb && !e->error_cb_fired) { e->error_cb_fired = true; e->error_cb(e->error_ctx, e->error.c_str()); }
}

// `<Voice>::new(sample_rate)` of each channel instrument: kick(tight) / snare(tight) / hihat(short) / Tom2::new / bass(acid) /
// PolySynth (default config) / Granulator (ffi.rs:809-850 and :2320-2326; kick.rs:772, snare.rs:764, hihat2.rs:350, tom2.rs:199,
// bass.rs:608)
inline GooeyVoicePatch default_patch(uint32_t type) {
  GooeyVoicePatch p;
  memset(&p, 0, sizeof p);
  p.instrument = type;
  switch (type) {
    case GOOEY_INSTRUMENT_KICK: case GOOEY_INSTRUMENT_SNARE: case GOOEY_INSTRUMENT_BASS: preset_flat(type, 0, p.params); break;
    case GOOEY_INSTRUMENT_HIHAT: { const float h[5] = {0.76f, 0.05f, 0.00f, 1.00f, 1.0f}; memcpy(p.params, h, sizeof h); } break;
    case GOOEY_B200_VOICE_POLY: memcpy(p.params, GOOEY_POLY_PRESETS[0], sizeof GOOEY_POLY_PRESETS[0]); break;
    default: break;   // tom: Tom2::new; the granulator takes no patch
  }
  return p;
}

inline GooeyEngine* engine_create(int device, float sr) {
  EngineBank& B = engine_bank(device, sr);
  std::lock_guard<std::recursive_mutex> lk(B.mu);
  std::unique_ptr<GooeyEngine> e(new GooeyEngine);
  e->bank = &B; e->sr = sr; e->transport.sr = sr;
  for (int c = 0; c < N_CH; c++) {
    const GooeyVoicePatch p = default_patch((uint32_t)c);
    e->voice[c] = {p.instrument, B.voices.create(p, sr), c < N_STRIPS, {}};
  }
  for (int c = 0; c < N_STRIPS; c++) { e->strip[c].seq.init(120.0f, sr); e->strip[c].blender.default_for_type(e->voice[c].type); }
  gd::MixState ms;
  memset(&ms, 0, sizeof ms);
  for (int c = 0; c < gd::N_VOICE_CH; c++) { ms.ch_gain[c] = {1.0f, 1.0f}; ms.ch_mute[c] = {1.0f, 1.0f}; ms.ch_pan[c] = {0.5f, 0.5f}; }
  for (int t = 0; t < gd::MAX_TRACKS; t++) { ms.tr_gain[t] = {1.0f, 1.0f}; ms.tr_pan[t] = {0.5f, 0.5f}; ms.tr_mute[t] = {1.0f, 1.0f}; }
  ms.master = {0.25f, 0.25f};
  const uint32_t kinds[4] = {gd::FXK_TILT, gd::FXK_DELAY, gd::FXK_SPRING, gd::FXK_PLATE};
  for (int s = 0; s < 4; s++) gd::fx_construct(ms.fx[s], kinds[s], false, sr, 120.0f);
  e->mix_slot = B.mix_pool.alloc(ms);
  // a recycled slot inherits its predecessor's delay-line columns: a fresh engine starts from silence.  The columns are
  // cleared in bulk at the next render (one coalesced kernel per arena over every dirty slot) instead of one strided
  // memset per engine and arena (thousands of engines re-created between two batches: ~14 MB of 4-byte writes each).
  GH_CUDA(cudaSetDevice(B.device));
  for (int s = 0; s < gd::MAX_FX; s++)
    if (B.ring[s].p && e->mix_slot < B.ring_cap_of[s]) { B.ring_dirty.push_back((uint32_t)e->mix_slot); break; }
  gd::MixCfg& c = e->cfg;
  memset(&c, 0, sizeof c);
  c.n_tracks = 4;
  const int32_t routes[9] = {0, 1, 2, 3, 3, -1, -1, -1, -1};   // graph.rs:131-143; sampler racks start unrouted
  for (int i = 0; i < 9; i++) c.route[i] = routes[i];
  const uint32_t order[9] = {7, 2, 0, 4, 1, 3, 8, 6, 9};   // DEFAULT_EFFECT_ORDER (ffi.rs:1583-1593)
  for (int i = 0; i < 9; i++) c.order[i] = order[i];
  for (int s = 0; s < gd::MAX_FX; s++) { c.fx_kind[s] = s < 4 ? kinds[s] : (uint32_t)gd::FXK_NONE; c.fx_enabled[s] = 0; }
  for (int i = 0; i < 12; i++) c.gslot[i] = 0xff;
  for (int s = 0; s < 4; s++) c.gslot[kinds[s]] = (uint8_t)s;
  c.comp_sidechain = 0xFFFFFFFFu; c.fx_rack = 0;
  c.limiter_on = 0; c.lim_th = 1.0f; c.lim_inv = 1.0f;
  if ((int)B.cfgs.size() <= e->mix_slot) B.cfgs.resize(e->mix_slot + 1);
  B.cfgs[e->mix_slot] = c;
  return e.release();
}

inline void engine_destroy(GooeyEngine* e) {
  if (!e) return;
  EngineBank& B = *e->bank;
  std::lock_guard<std::recursive_mutex> lk(B.mu);
  for (const auto& v : e->voice) B.voices.release(v.type, v.slot);
  bool holds_pcm = (bool)e->gran_buf;
  for (auto& l : e->loops) holds_pcm = holds_pcm || l.buf;
  for (auto& r : e->samplers) holds_pcm = holds_pcm || r.registered;
  if (holds_pcm) { cudaSetDevice(B.device); cudaStreamSynchronize(B.stream); }   // no launch may still read the buffers
  B.mix_pool.release(e->mix_slot);
  delete e;
}

// note -> normalized frequency parameter of the voice (ffi.rs:1505-1518)
inline bool note_freq_range(uint32_t type, float& mn, float& mx) {
  if (type == GOOEY_INSTRUMENT_BASS) { mn = 30.0f; mx = 200.0f; return true; }
  if (type == GOOEY_INSTRUMENT_KICK) { mn = 30.0f; mx = 120.0f; return true; }
  if (type == GOOEY_INSTRUMENT_TOM) { mn = 40.0f; mx = 600.0f; return true; }
  return false;
}
inline float midi_to_norm(uint8_t note, float mn, float mx) {
  float hz = 440.0f * gm::g_powf(2.0f, ((float)note - 69.0f) / 12.0f);
  return gd::clampf((hz - mn) / (mx - mn), 0.0f, 1.0f);
}

enum { OUT_MONO = 0, OUT_STEREO = 1 };

// ChannelInstrument::apply_modulation (ffi.rs:322-405): FFI parameter id of the channel's instrument type -> internal
// parameter index + how the bipolar value lands on it.  false: the id is not modulatable (ignored, like the reference).
inline bool lfo_route_target(uint32_t type, uint32_t ffi_param, uint32_t& param, uint32_t& mode) {
  mode = 0;
  switch (type) {
    case GOOEY_INSTRUMENT_KICK: if (ffi_param >= 8 || ffi_param == 5) return false; param = (uint32_t)kKickFfi[ffi_param]; return true;   // not the pitch envelope (:330-332)
    case GOOEY_INSTRUMENT_SNARE: if (ffi_param >= 20 || ffi_param == 12) return false; param = (uint32_t)kSnareFfi[ffi_param]; return true;
    case GOOEY_INSTRUMENT_HIHAT: if (ffi_param >= 6) return false; param = (uint32_t)kHatFfi[ffi_param]; return true;
    case GOOEY_INSTRUMENT_TOM: if (ffi_param >= 9) return false; param = ffi_param; mode = ffi_param == 8 ? 2u : 1u; return true;
    case GOOEY_INSTRUMENT_BASS: if (ffi_param >= 16) return false; param = ffi_param; return true;
    default: return false;
  }
}
inline float lfo_beats(uint32_t d) { const float B[8] = {16.0f, 8.0f, 4.0f, 2.0f, 1.0f, 0.5f, 0.25f, 0.125f}; return B[d < 8 ? d : 4]; }   // lfo.rs:14-25

// First FFI touch of the poly synth / granulator of an engine: from now on the voice is launched with the engine.  It was
// not ticked so far (an untouched poly synth / granulator is bit-exactly silent and its state does not move), so its
// clock is set to the engine's and, for the granulator, the placeholder buffer is attached.  Returns the channel's pending events.
inline std::vector<gd::VoiceEvent>& aux_touch(GooeyEngine* e, int ch) {
  GooeyEngine::Voice& v = e->voice[ch];
  if (v.launched) return v.pending;
  v.launched = true;
  v.pending.push_back(make_event(0, gd::EV_SET_TIME, 1, 0.0f, e->k));
  if (ch == CH_GRAN) { gran_buffer_events(v.pending, 0, e->bank->d_silent.p, 44100.0f, 1); e->cfg.src_gran = 1; }
  else e->cfg.src_poly = 1;
  std::lock_guard<std::recursive_mutex> lk(e->bank->mu);
  e->bank->cfgs[e->mix_slot] = e->cfg;
  return v.pending;
}

using PieceHook = std::function<void(uint32_t f0, uint32_t nf, cudaEvent_t mixed)>;   // see engines_render

// Appends the events of `ev` from `pos` on that lie before frame `end` to `out`, rebased to frame f0, and advances `pos` past them.
inline void take_piece(const std::vector<gd::VoiceEvent>& ev, size_t& pos, uint32_t f0, uint32_t end, std::vector<gd::VoiceEvent>& out) {
  for (; pos < ev.size() && ev[pos].frame < end; pos++) { gd::VoiceEvent x = ev[pos]; x.frame -= f0; out.push_back(x); }
}

// GOOEY_B200_TRACE=1: per piece, the host time of its launch phases and the device times of its voice and mix stages, on
// stderr (diagnostic)
struct PieceTrace {
  using Clock = std::chrono::steady_clock;
  const bool on = getenv("GOOEY_B200_TRACE") != nullptr;
  std::vector<cudaEvent_t> tv0, tv1, tm0, tm1;   // per piece: voice stage start / end (voice stream), mix stage start / end (mix stream)
  Clock::time_point host[3];                     // the current piece: start, event lists built, voices launched
  void host_mark(int k) { if (on) host[k] = Clock::now(); }
  void mark(std::vector<cudaEvent_t>& v, cudaStream_t s) { if (!on) return; cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, s); v.push_back(e); }
  void host_line(size_t pc) const {
    if (!on) return;
    auto msf = [](Clock::time_point a, Clock::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
    fprintf(stderr, "[gooey trace] host, piece %zu: wait + event lists %.1f ms, voice launches %.1f ms, mixer launches %.1f ms\n", pc, msf(host[0], host[1]), msf(host[1], host[2]), msf(host[2], Clock::now()));
  }
  void device_lines(cudaStream_t st, const std::vector<uint32_t>& cuts) {   // once every piece has been enqueued on `st`
    if (!on) return;
    GH_CUDA(cudaStreamSynchronize(st));
    for (size_t pc = 0; pc < tv0.size(); pc++) {
      float a = 0, b = 0, c = 0, d = 0;
      cudaEventElapsedTime(&a, tv0[0], tv0[pc]); cudaEventElapsedTime(&b, tv0[pc], tv1[pc]); cudaEventElapsedTime(&c, tv0[0], tm0[pc]); cudaEventElapsedTime(&d, tm0[pc], tm1[pc]);
      fprintf(stderr, "[gooey trace] piece %zu frames %u: voices start %.1f ms, take %.1f ms; mix start %.1f ms, takes %.1f ms\n", pc, cuts[pc] - (pc ? cuts[pc - 1] : 0), a, b, c, d);
    }
    for (auto* v : {&tv0, &tv1, &tm0, &tm1}) for (auto e : *v) cudaEventDestroy(e);
  }
};

// One engines_render call.  Its stages run in the order they are declared; each fills the members listed above it.
struct EngineRender {
  EngineBank& B;
  const std::vector<GooeyEngine*>& E;
  const uint32_t frames;
  const bool bounce;
  const int n, n_lpad;
  const cudaStream_t st;
  // schedule: the call's events of every voice channel ([engine * N_CH + channel]) and of every engine's mixer
  std::vector<std::vector<gd::VoiceEvent>> vev, mev;
  uint32_t chan_mask = 0;                 // bit c: some engine launches channel c
  uint64_t kmin = ~0ull, kmax = 0;        // the engines' clock range
  // external sources: one stereo row pair per loop mixer / sounding rack
  struct ExtRef { int engine, rack; };
  std::vector<int> loop_refs; std::vector<ExtRef> rack_refs;
  uint32_t ext_pairs = 0;
  // device state
  const double* tt = nullptr;
  size_t vstride = 0;                     // row pitch of the voice buffers
  bool two_bufs = false;                  // more than one piece: the mix of piece p overlaps the voices of piece p + 1
  std::vector<uint32_t> cuts;             // the end frame of every piece
  // LFO pool
  std::vector<std::vector<gd::ModRoute>> vroutes;   // [engine * N_CH + channel]; only strips are routed
  struct LfoRef { int engine, lfo; };
  std::vector<LfoRef> lfo_refs;
  const float* lfo_planes = nullptr;
  // pieces
  gd::MixLaunch M;                        // filled once; every piece sets events, ev_begin, voice_buf, frames, out and ext
  float* out = nullptr;
  std::vector<size_t> vpos, mpos;         // the next event of every voice / mix event list
  std::vector<gd::VoiceEvent> cur, mflat;
  std::vector<uint32_t> mbegin;
  PieceTrace trace;

  EngineRender(EngineBank& B_, const std::vector<GooeyEngine*>& E_, uint32_t frames_, bool bounce_)
      : B(B_), E(E_), frames(frames_), bounce(bounce_), n((int)E_.size()), n_lpad(pad32(n)), st(B_.stream),
        vev((size_t)n * N_CH), mev(n), vpos((size_t)n * N_CH, 0), mpos(n, 0) {}

  // argument errors are found before any engine is touched (BadBatch -> GOOEY_E_INVALID, no sticky error)
  void check_batch() const {
    std::set<const GooeyEngine*> seen;
    for (const GooeyEngine* e : E) {
      if (e->bank != &B) throw BadBatch("engines of one batch must share device and sample rate");
      if (!seen.insert(e).second) throw BadBatch("the same engine appears twice in one batch");
      if (!bounce && (uint64_t)e->k + frames >= 0xffffffffull) throw BadBatch("engine clock index would pass 2^32 frames (27 h at 44.1 kHz); bounce or recreate the engine");
    }
  }

  // ---- per-engine schedule (host): event lists over the whole call ----
  struct MidiKey { uint32_t frame, seq, ch; float vel; };
  void schedule() {
    std::vector<SeqFire> fires;
    std::vector<MidiKey> midi;
    for (int i = 0; i < n; i++) {
      GooeyEngine* e = E[i];
      if (bounce) {
        e->k = 0;
        for (auto& s : e->strip) { s.seq.reset(); s.seq.start(); }
      }
      kmin = std::min<uint64_t>(kmin, e->k);
      kmax = std::max<uint64_t>(kmax, (uint64_t)e->k + frames);
      mix_events(e, mev[i]);
      midi.clear();
      channel_events(e, &vev[(size_t)i * N_CH], midi, fires);
      midi_export(e, midi);
    }
  }
  // pending mixer edits, the bounce preamble's snaps and the per-buffer mute / solo targets (ffi.rs:1099-1109, graph.rs
  // update_mute_solo_targets)
  void mix_events(GooeyEngine* e, std::vector<gd::VoiceEvent>& mx) const {
    mx = e->mix_pending; e->mix_pending.clear();
    if (bounce) mx.push_back(make_event(0, gd::MX_SNAP, 0, 0.0f));       // voice strips snap to their current targets
    bool any_solo = false, any_tsolo = false;
    for (auto& s : e->strip) any_solo |= s.soloed;
    for (uint32_t t = 0; t < e->cfg.n_tracks; t++) any_tsolo |= e->track_soloed[t];
    auto strip_mutes = [&] {
      for (int ch = 0; ch < N_STRIPS; ch++) {
        const auto& s = e->strip[ch];
        mx.push_back(make_event(0, gd::MX_SET, gd::MP_CH_MUTE + ch, s.soloed ? 1.0f : (any_solo ? 0.0f : (s.muted ? 0.0f : 1.0f))));
      }
    };
    auto track_mutes = [&] {
      for (uint32_t t = 0; t < e->cfg.n_tracks; t++)
        mx.push_back(make_event(0, gd::MX_SET, gd::MP_TR_MUTE + t, e->track_soloed[t] ? 1.0f : ((any_tsolo || e->track_muted[t]) ? 0.0f : 1.0f)));
    };
    if (!bounce) { strip_mutes(); track_mutes(); return; }
    // graph.snap_strip_params() refreshes the track mute targets and snaps; master_gain.snap(); the voice-strip
    // mute targets are only written by render() afterwards, so they glide (ffi.rs:7846-7854, 1099-1109)
    track_mutes();
    mx.push_back(make_event(0, gd::MX_SNAP, 1, 0.0f));
    mx.push_back(make_event(0, gd::MX_SNAP, 2, 0.0f));
    strip_mutes();
  }
  // every launched channel: its pending events, then the bounce's clock reset; a strip then adds its manual trigger and its
  // sequencer's fires (ffi.rs:1162-1198), and both go to the MIDI export
  void channel_events(GooeyEngine* e, std::vector<gd::VoiceEvent>* out_ev, std::vector<MidiKey>& midi, std::vector<SeqFire>& fires) {
    for (int ch = 0; ch < N_CH; ch++) {
      GooeyEngine::Voice& v = e->voice[ch];
      if (!v.launched) continue;
      chan_mask |= 1u << ch;
      auto& ev = out_ev[ch];
      ev.insert(ev.end(), v.pending.begin(), v.pending.end());
      v.pending.clear();
      // the bounce's clock reset comes after the pending edits: a voice swapped in since the last render carries a
      // "join the engine clock at k" event that must not outlive the reset (the clock window of a bounce is [0, frames])
      if (bounce) ev.push_back(make_event(0, gd::EV_SET_TIME, 0, 0.0f, 0));
      if (ch >= N_STRIPS) continue;
      auto& s = e->strip[ch];
      if (s.trig_pending) { s.trig_pending = false; ev.push_back(make_event(0, gd::EV_TRIGGER, 0, s.trig_vel)); midi.push_back({0u, 0u, (uint32_t)ch, s.trig_vel}); }
      fires.clear();
      s.seq.run(frames, fires);
      if (!e->seq_triggers_enabled) continue;
      for (const SeqFire& f : fires) midi.push_back({f.frame, 1u, (uint32_t)ch, f.velocity});
      for (const SeqFire& f : fires) {
        // apply_sequencer_blend_setting (:1384-1402): the step's own blend, else the channel's pad position when blending is
        // on; a blend that was applied is followed by snap_params (:1168-1171)
        auto add = [&](const gd::VoiceEvent& x) { ev.push_back(x); };
        if (f.has_blend) s.blender.apply(f.bx, f.by, f.frame, add);
        else if (s.blend_enabled) s.blender.apply(s.blend_x, s.blend_y, f.frame, add);
        if (f.has_blend || s.blend_enabled) ev.push_back(make_event(f.frame, gd::EV_SNAP, 0, 0.0f));
        float mn, mxf;
        if (f.has_note) { if (note_freq_range(v.type, mn, mxf)) ev.push_back(make_event(f.frame, gd::EV_NOTE_FREQ, 0, midi_to_norm(f.note, mn, mxf))); }
        else ev.push_back(make_event(f.frame, gd::EV_RESTORE_FREQ, 0, 0.0f));
        ev.push_back(make_event(f.frame, gd::EV_TRIGGER, 0, f.velocity));
      }
    }
  }
  // MIDI note-on export (ffi.rs:994-1004, 1079-1094, 1196): manual triggers first (offset 0, channel order), then the sequencer's
  // in frame / channel order; the list is cleared by every render() call and capped at 64, and a bounce IS a run of 512-frame
  // render() calls (ffi.rs:7855-7870), so after a bounce only the last chunk's events are pending, offsets relative to it.
  void midi_export(GooeyEngine* e, std::vector<MidiKey>& midi) const {
    std::stable_sort(midi.begin(), midi.end(), [](const MidiKey& a, const MidiKey& b) {
      return a.frame != b.frame ? a.frame < b.frame : (a.seq != b.seq ? a.seq < b.seq : a.ch < b.ch); });
    const uint32_t base = bounce ? ((frames - 1) / 512u) * 512u : 0u;
    e->midi_events.clear();
    for (const MidiKey& m : midi) {
      if (m.frame < base) continue;
      if (e->midi_events.size() >= 64) break;
      e->midi_events.push_back({m.ch, m.vel, m.frame - base});
    }
  }

  // ---- sample-playback sources: one descriptor per engine with a loaded loop / per rack with a sounding voice ----
  void ext_sources() {
    B.h_loop_descs.clear(); B.h_rack_descs.clear();
    std::vector<gd::SamplerHit> rack_hits; std::vector<size_t> rack_hit_off;
    for (int i = 0; i < n; i++) {
      GooeyEngine* e = E[i];
      e->cfg.src_ext = 0;
      for (int s = 0; s < gd::EXT_SOURCES; s++) e->cfg.ext_row[s] = 0;
      // Mixer::tick writes the gate targets every sample from the mute / solo flags, which only change between calls (mod.rs:63-72)
      bool any_lsolo = false, any_loaded = false;
      for (auto& l : e->loops) { any_lsolo = any_lsolo || l.soloed; any_loaded = any_loaded || (l.buf && l.len > 0); }
      for (auto& l : e->loops) gd::lsm_set(l.active, (any_lsolo ? l.soloed : !l.muted) ? 1.0f : 0.0f, 0.0f, 1.0f);
      if (any_loaded) {
        gd::LoopMixer m;
        memset(&m, 0, sizeof m);
        for (int c = 0; c < gd::LOOP_CHANNELS; c++) {
          auto& l = e->loops[c];
          l.describe(m.ch[c], e->loop_engine_bpm);
          B.attach_stretcher(l, m.ch[c]);
        }
        m.row = ext_pairs;
        e->cfg.src_ext |= 1u; e->cfg.ext_row[0] = ext_pairs++;
        B.h_loop_descs.push_back(m); loop_refs.push_back(i);
      } else {
        // nothing to read: the channels output exactly 0 and only their smoothers move (they tick every sample, :202-207)
        for (auto& l : e->loops)
          for (uint32_t f = 0; f < frames && (l.gain.c != l.gain.t || l.active.c != l.active.t); f++) { gd::lsm_tick(l.gain, B.rc.smooth15); gd::lsm_tick(l.active, B.rc.smooth15); }
      }
      // rack patterns: resolved on the host into pad hits (resolve_rack_patterns above)
      gh::RackPattern* pats[gd::SAMPLER_RACKS];
      std::vector<gh::RackHit> rhits[gd::SAMPLER_RACKS];
      bool any_rack = false;
      for (int r = 0; r < gd::SAMPLER_RACKS; r++) { pats[r] = e->samplers[r].registered ? &e->samplers[r].pat : nullptr; any_rack = any_rack || pats[r]; }
      if (any_rack) gh::resolve_rack_patterns(e->transport, pats, gd::SAMPLER_RACKS, frames, bounce, e->seq_triggers_enabled, rhits);
      else if (e->transport.running) e->transport.lazy += frames;       // nothing listens to the transport: it just advances
      for (int r = 0; any_rack && r < gd::SAMPLER_RACKS; r++) {
        auto& R = e->samplers[r];
        if (!R.registered) continue;
        std::vector<gd::SamplerHit> hits;
        for (const gh::RackHit& h : rhits[r]) hits.push_back(gd::SamplerHit{h.frame, h.slot, h.velocity, 0u});
        bool sounding = false;
        for (const auto& v : R.voices) sounding = sounding || v.samples != nullptr;
        if (!sounding && hits.empty()) continue;         // no active voice and no hit: the rack ticks to exactly 0 and its state does not move
        gd::SamplerRack d;
        memset(&d, 0, sizeof d);
        memcpy(d.v, R.voices, sizeof d.v);
        d.row = ext_pairs; d.rack = (uint32_t)r;
        for (int k = 0; k < gd::SAMPLER_SLOTS; k++) {
          const auto& S = R.slots[k];
          if (S.buf) d.slots[k] = gd::SamplerSlotRef{S.buf->p, S.frames, S.channels, (double)S.sr / (double)e->sr};
        }
        d.next_age = R.next_age;
        d.n_hits = (uint32_t)hits.size(); d.next_hit = 0; d.cur_frame = 0;
        rack_hit_off.push_back(rack_hits.size());
        rack_hits.insert(rack_hits.end(), hits.begin(), hits.end());
        e->cfg.src_ext |= 2u << r; e->cfg.ext_row[1 + r] = ext_pairs++;
        B.h_rack_descs.push_back(d); rack_refs.push_back({i, r});
      }
      B.cfgs[e->mix_slot] = e->cfg;
    }
    if (!rack_hits.empty()) {                             // one flat hit table for the call; the descriptors point into it
      B.d_rack_hits.upload(rack_hits.data(), rack_hits.size(), st);
      for (size_t q = 0; q < B.h_rack_descs.size(); q++) if (B.h_rack_descs[q].n_hits) B.h_rack_descs[q].hits = B.d_rack_hits.p + rack_hit_off[q];
    }
  }

  // ---- device state: clock window, pools, configs, rings, piece geometry, buffers ----
  void device_state() {
    tt = B.clock.view(clock_table(B.sr), kmin, kmax, st);
    B.mix_pool.flush(st);
    B.d_cfg.upload(B.cfgs.data(), B.cfgs.size(), st);
    uint32_t need_words[gd::MAX_FX] = {0};
    for (int i = 0; i < n; i++) {
      const gd::MixCfg& c = E[i]->cfg;
      for (int s = 0; s < gd::MAX_FX; s++) {
        const bool used = c.fx_kind[s] != gd::FXK_NONE && (s >= 4 || c.fx_enabled[s] != 0);
        if (used) need_words[s] = std::max(need_words[s], ring_words_of(B.geo, c.fx_kind[s]));
      }
    }
    B.clear_dirty_rings(st);
    // every arena shares one row pitch (the mix pool's capacity); arenas that already exist are re-laid when it grows
    for (int s = 0; s < gd::MAX_FX; s++) {
      const uint32_t words = std::max(need_words[s], B.ring_words[s]);
      if (words) B.ensure_ring(s, words, B.mix_pool.cap);
    }
    std::vector<uint32_t> mix_slots(n);
    for (int i = 0; i < n; i++) mix_slots[i] = (uint32_t)E[i]->mix_slot;
    B.d_mix_slots.upload(mix_slots.data(), n, st);
    // pieces: bound the voice buffer (a row per engine and launched channel) to ~2 GiB
    int n_ch = 0;
    for (int c = 0; c < N_CH; c++) if (chan_mask >> c & 1u) n_ch = c + 1;
    const size_t rows = (size_t)n_ch * n_lpad;
    size_t piece = ((size_t)2 << 30) / (rows * 4);
    piece = std::min<size_t>(std::max<size_t>(piece & ~(size_t)31, 2048), 65536);
    piece = std::min<size_t>(piece, (frames + 31) & ~31u);
    two_bufs = frames > piece || frames > 4096;
    // row pitch of the voice buffers: an odd multiple of 32 frames (the mixer reads 32 rows x 7 channels per tile; rows a power of
    // two apart would all fall into the same cache sets)
    vstride = ((piece / 32) & 1) ? piece : piece + 32;
    B.d_voice_bufs[0].alloc(rows * vstride);
    if (two_bufs) B.d_voice_bufs[1].alloc(rows * vstride);
    if (ext_pairs) {
      B.d_ext[0].alloc((size_t)2 * ext_pairs * vstride);
      if (two_bufs) B.d_ext[1].alloc((size_t)2 * ext_pairs * vstride);
      if (!B.h_loop_descs.empty()) B.d_loop_descs.upload(B.h_loop_descs.data(), B.h_loop_descs.size(), st);
      if (!B.h_rack_descs.empty()) B.d_rack_descs.upload(B.h_rack_descs.data(), B.h_rack_descs.size(), st);
    }
    bool any_chain = false;
    for (int i = 0; i < n && !any_chain; i++) for (int q = 0; q < gd::MAX_FX; q++) any_chain = any_chain || (E[i]->cfg.fx_kind[q] != gd::FXK_NONE && E[i]->cfg.fx_enabled[q]);
    if (any_chain) B.d_premix.alloc((size_t)2 * n_lpad * vstride);
    // Piece schedule.  Parameters edited through the FFI glide for ~10 smoother time constants (kick.rs: 15 ms -> ~6000
    // samples) and the planner keeps a voice on the per-sample general path for a whole piece while anything glides, so the
    // first pieces are short: a gliding voice re-enters the time-parallel path within a few thousand frames.
    const uint32_t lead[10] = {2048, 2048, 2048, 2048, 2048, 2048, 4096, 4096, 8192, 16384};
    uint32_t f = 0;
    for (int k = 0; k < 10 && f + lead[k] < frames && lead[k] < piece; k++) { f += lead[k]; cuts.push_back(f); }
    while (f + piece < frames) { f += (uint32_t)piece; cuts.push_back(f); }
    cuts.push_back(frames);
  }

  // ---- LFO pool: one stream per enabled LFO; routed ones get a plane of per-frame values (computed on the device) ----
  void lfo_pool() {
    vroutes.resize((size_t)n * N_CH);
    B.h_lfo_streams.clear();
    int n_planes = 0;
    for (int i = 0; i < n; i++) {
      GooeyEngine* e = E[i];
      for (int li = 0; li < 8; li++) {
        if (!e->lfo_enabled[li]) continue;
        gd::LfoStream sdesc;
        volatile float bps = e->bpm / 60.0f;                                   // MusicalDivision::to_frequency (lfo.rs:27-33)
        volatile float freq = bps / lfo_beats(e->lfos[li].division);
        sdesc.phase = e->lfos[li].phase; sdesc.inc = freq / e->sr; sdesc.amount = e->lfos[li].amount; sdesc.offset = e->lfos[li].offset;
        sdesc.plane = -1;
        for (const auto& r : e->lfo_routes[li]) {
          if (r.instrument >= (uint32_t)N_STRIPS) continue;                    // voice_mut(channel) is None
          uint32_t param, mode;
          if (!lfo_route_target(e->voice[r.instrument].type, r.param, param, mode)) continue;
          if (sdesc.plane < 0) sdesc.plane = n_planes++;
          vroutes[(size_t)i * N_CH + r.instrument].push_back(gd::ModRoute{param, mode, r.depth, (uint32_t)sdesc.plane});
        }
        B.h_lfo_streams.push_back(sdesc);
        lfo_refs.push_back({i, li});
      }
    }
    if (B.h_lfo_streams.empty()) return;
    B.d_lfo_streams.upload(B.h_lfo_streams.data(), B.h_lfo_streams.size(), st);
    if (n_planes) B.d_lfo_planes.alloc((size_t)n_planes * frames);
    gd::lfo_kernel<<<((int)B.h_lfo_streams.size() + 63) / 64, 64, 0, st>>>(B.d_lfo_streams.p, (int)B.h_lfo_streams.size(), B.d_lfo_planes.p, (long long)frames, (int)frames);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    GH_CUDA(cudaGetLastError());
    if (n_planes) lfo_planes = B.d_lfo_planes.p;
  }

  // ---- the mixer's launch record and the call's meters; the mix stream starts after everything queued so far ----
  void mixer_setup(int out_mode, float* out_dev, size_t stride) {
    B.d_peaks.alloc((size_t)n * gd::N_PEAKS);
    GH_CUDA(cudaMemsetAsync(B.d_peaks.p, 0, (size_t)n * gd::N_PEAKS * 4, st));
    B.d_chain_units.alloc(1);
    GH_CUDA(cudaMemsetAsync(B.d_chain_units.p, 0, sizeof(unsigned long long), st));
    B.d_mix_fast.alloc(n); B.d_mix_consts.alloc(n);
    out = out_dev;
    memset(&M, 0, sizeof M);
    M.state = B.mix_pool.d.p; M.n = n; M.state_cap = B.mix_pool.cap; M.slots = B.d_mix_slots.p; M.n_lpad = n_lpad;
    M.cfg = B.d_cfg.p; M.voice_stride = (long long)vstride; M.chan_mask = chan_mask;
    for (int s = 0; s < gd::MAX_FX; s++) M.ring[s] = B.ring[s].p;
    M.ring_cap = B.mix_pool.cap;
    M.out_stride = (long long)stride; M.out_mode = out_mode; M.out_rows = nullptr;
    M.rc = B.rc; M.geo = B.geo;
    M.center_l = gm::g_cosf(0.5f * 1.57079632679489661923f); M.center_r = gm::g_sinf(0.5f * 1.57079632679489661923f);
    M.fast = B.d_mix_fast.p; M.consts = B.d_mix_consts.p;
    M.peaks = B.d_peaks.p;
    M.premix = B.d_premix.p; M.premix_stride = (long long)vstride;
    M.ext_stride = (long long)vstride;
    M.chain_units = B.d_chain_units.p;
    // dynamic shared memory beyond 48 KB (with the static tiles)
    func_attr_once((const void*)gd::mix_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gd::MIX_DYN_SMEM);
    func_attr_once((const void*)gd::chain_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gd::CHAIN_SMEM);
    GH_CUDA(cudaEventRecord(B.ev_piece, st));
    GH_CUDA(cudaStreamWaitEvent(B.mix_stream, B.ev_piece, 0));   // after the uploads and the ring set-up
    GH_CUDA(cudaEventRecord(B.ev0, st));
    B.mix_timer.clear();
  }

  // ---- one piece, frames [f0, f0 + nf): voices and external sources on the voice stream, then the mixer on its own ----
  void piece(size_t pc, const PieceHook* on_piece) {
    const uint32_t f0 = pc ? cuts[pc - 1] : 0, nf = cuts[pc] - f0;
    const int vb = two_bufs ? (int)(pc & 1) : 0;
    trace.host_mark(0);
    if (pc >= (two_bufs ? 2u : 1u)) GH_CUDA(cudaStreamWaitEvent(st, B.ev_mixed[vb], 0));   // voice buffer vb is free again
    B.voices.reset();
    for (int i = 0; i < n; i++)
      for (int ch = 0; ch < N_CH; ch++) {
        const GooeyEngine::Voice& v = E[i]->voice[ch];
        const size_t q = (size_t)i * N_CH + ch;
        if (!v.launched) continue;
        cur.clear();
        take_piece(vev[q], vpos[q], f0, f0 + nf, cur);
        B.voices.add(v.type, (uint32_t)v.slot, (uint32_t)(ch * n_lpad + i), cur, lfo_planes && !vroutes[q].empty() ? &vroutes[q] : nullptr);
      }
    trace.host_mark(1);
    GH_CUDA(cudaEventRecord(B.ev_piece, st));
    // the clock index differs per engine only through e->k; voices carry their own k, the launch passes the table
    trace.mark(trace.tv0, st);
    B.voices.set_mod(lfo_planes, (long long)frames, (int)f0);
    B.voices.launch(st, B.ev_piece, B.rc, tt, (int)nf, B.d_voice_bufs[vb].p, (long long)vstride);
    if (ext_pairs) {   // loop mixers and sampler racks of this piece, on the voice stream (the mixer waits for ev_voices)
      const gd::ExtTickCtx xc{B.sr, B.rc.smooth15};
      if (!B.h_loop_descs.empty()) {
        const int nd = (int)B.h_loop_descs.size();
        gd::ext_source_kernel<gd::LoopMixer><<<(nd + 63) / 64, 64, 0, st>>>(B.d_loop_descs.p, nd, B.d_ext[vb].p, (long long)vstride, (int)nf, xc);
        g_launches.fetch_add(1, std::memory_order_relaxed);
      }
      if (!B.h_rack_descs.empty()) {
        const int nd = (int)B.h_rack_descs.size();
        gd::ext_source_kernel<gd::SamplerRack><<<(nd + 63) / 64, 64, 0, st>>>(B.d_rack_descs.p, nd, B.d_ext[vb].p, (long long)vstride, (int)nf, xc);
        g_launches.fetch_add(1, std::memory_order_relaxed);
      }
      GH_CUDA(cudaGetLastError());
    }
    trace.mark(trace.tv1, st);
    trace.host_mark(2);
    GH_CUDA(cudaEventRecord(B.ev_voices[vb], st));
    GH_CUDA(cudaStreamWaitEvent(B.mix_stream, B.ev_voices[vb], 0));
    mix_piece(f0, nf, vb);
    if (on_piece) (*on_piece)(f0, nf, B.ev_mixed[vb]);
    trace.mark(trace.tm1, B.mix_stream);
    trace.host_line(pc);
  }
  void mix_piece(uint32_t f0, uint32_t nf, int vb) {
    cudaStream_t ms = B.mix_stream;
    mflat.clear(); mbegin.assign(1, 0);
    for (int i = 0; i < n; i++) { take_piece(mev[i], mpos[i], f0, f0 + nf, mflat); mbegin.push_back((uint32_t)mflat.size()); }
    if (mflat.empty()) mflat.push_back(make_event(0xffffffffu, 0xffff, 0, 0.0f));
    B.d_mix_eventss[vb].upload(mflat.data(), mflat.size(), ms);      // pageable source: staged before the call returns
    B.d_mix_ev_begins[vb].upload(mbegin.data(), mbegin.size(), ms);
    M.events = B.d_mix_eventss[vb].p; M.ev_begin = B.d_mix_ev_begins[vb].p; M.voice_buf = B.d_voice_bufs[vb].p; M.frames = (int)nf;
    M.out = out + (M.out_mode == OUT_MONO ? (size_t)f0 : (size_t)2 * f0);
    M.ext = ext_pairs ? B.d_ext[vb].p : nullptr;
    trace.mark(trace.tm0, ms);
    gd::mix_prepare_kernel<<<(n + 127) / 128, 128, 0, ms>>>(M);
    gd::mix_fast_kernel<<<dim3((nf + 1023) / 1024, n), 256, 0, ms>>>(M);
    B.mix_timer.begin(ms);
    // settled tilt / delay / spring chains: whole warps of engines go to the pipelined chain kernel, mix_kernel takes the rest
    const bool chain_fast = getenv("GOOEY_B200_NO_CHAIN_FAST") == nullptr;     // (tests compare the two paths bit for bit)
    if (chain_fast && M.premix) { gd::chain_fast_kernel<<<(n + 31) / 32, 32, gd::CHAIN_SMEM, ms>>>(M); g_launches.fetch_add(1, std::memory_order_relaxed); }
    gd::mix_kernel<<<(n + 31) / 32, 32, gd::MIX_DYN_SMEM, ms>>>(M);
    B.mix_timer.end(ms, "mix_kernel", (double)n * nf);
    g_launches.fetch_add(3, std::memory_order_relaxed);
    GH_CUDA(cudaGetLastError());
    GH_CUDA(cudaEventRecord(B.ev_mixed[vb], ms));
  }

  // ---- read-back, once the voice stream has joined the last mixes: meters, LFO phases, loop and rack state, clocks ----
  void read_back() {
    GH_CUDA(cudaStreamWaitEvent(st, B.ev_mixed[0], 0));
    if (two_bufs && cuts.size() > 1) GH_CUDA(cudaStreamWaitEvent(st, B.ev_mixed[1], 0));
    GH_CUDA(cudaEventRecord(B.ev1, st));
    trace.device_lines(st, cuts);
    // the call's maxima join the engines' read-and-reset peaks (one small copy; the caller synchronises the stream anyway)
    B.h_peaks.resize((size_t)n * gd::N_PEAKS);
    GH_CUDA(cudaMemcpyAsync(B.h_peaks.data(), B.d_peaks.p, B.h_peaks.size() * 4, cudaMemcpyDeviceToHost, st));
    GH_CUDA(cudaMemcpyAsync(&B.h_chain_units, B.d_chain_units.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    if (!B.h_lfo_streams.empty()) GH_CUDA(cudaMemcpyAsync(B.h_lfo_streams.data(), B.d_lfo_streams.p, B.h_lfo_streams.size() * sizeof(gd::LfoStream), cudaMemcpyDeviceToHost, st));
    if (!B.h_loop_descs.empty()) GH_CUDA(cudaMemcpyAsync(B.h_loop_descs.data(), B.d_loop_descs.p, B.h_loop_descs.size() * sizeof(gd::LoopMixer), cudaMemcpyDeviceToHost, st));
    if (!B.h_rack_descs.empty()) GH_CUDA(cudaMemcpyAsync(B.h_rack_descs.data(), B.d_rack_descs.p, B.h_rack_descs.size() * sizeof(gd::SamplerRack), cudaMemcpyDeviceToHost, st));
    GH_CUDA(cudaStreamSynchronize(st));
    for (size_t q = 0; q < loop_refs.size(); q++)      // playback state back into the engines' loop channels / sampler voices
      for (int c = 0; c < gd::LOOP_CHANNELS; c++) E[loop_refs[q]]->loops[c].absorb(B.h_loop_descs[q].ch[c]);
    for (size_t q = 0; q < rack_refs.size(); q++) {
      auto& R = E[rack_refs[q].engine]->samplers[rack_refs[q].rack];
      memcpy(R.voices, B.h_rack_descs[q].v, sizeof R.voices);
      R.next_age = B.h_rack_descs[q].next_age;
      for (int v = 0; v < gd::SAMPLER_VOICES; v++) {    // a voice the device started plays its pad's buffer (a pad cannot change during a call)
        if (!R.voices[v].samples) R.voices_release(v);
        else R.voice_buf[v] = R.slots[R.voices[v].slot].buf;
      }
    }
    for (size_t q = 0; q < lfo_refs.size(); q++) E[lfo_refs[q].engine]->lfos[lfo_refs[q].lfo].phase = B.h_lfo_streams[q].phase;
    for (int i = 0; i < n; i++) {
      for (int q = 0; q < gd::N_PEAKS; q++) { const float v = B.h_peaks[(size_t)i * gd::N_PEAKS + q]; if (v > E[i]->peaks[q]) E[i]->peaks[q] = v; }
      E[i]->k += frames;
      if (bounce) { for (auto& s : E[i]->strip) s.seq.stop(); for (auto& R : E[i]->samplers) if (R.registered) R.pat.seq.stop(); }
    }
  }
};

// Renders `frames` frames of every engine of `E` (all on one bank) into out_dev: mono rows [n][stride] (the bounce
// downmix 0.5 (l + r)) or interleaved stereo rows [n][stride >= 2 frames].  `bounce`: apply the reference's bounce
// preamble first (ffi.rs:7840-7854): clock to 0, sequencers reset + start, strips / graph / master snapped.
// on_piece (optional): called after the mix of frames [f0, f0 + nf) has been enqueued, with the event that marks it done.
inline void engines_render(const std::vector<GooeyEngine*>& E, uint32_t frames, int out_mode, bool bounce, float* out_dev, size_t stride,
                           const PieceHook* on_piece = nullptr) {
  if (E.empty() || frames == 0) return;
  EngineBank& B = *E[0]->bank;
  std::lock_guard<std::recursive_mutex> lk(B.mu);
  GH_CUDA(cudaSetDevice(B.device));
  EngineRender R(B, E, frames, bounce);
  R.check_batch();
  R.schedule();
  R.ext_sources();
  R.device_state();
  R.lfo_pool();
  R.mixer_setup(out_mode, out_dev, stride);
  for (size_t pc = 0; pc < R.cuts.size(); pc++) R.piece(pc, on_piece);
  R.read_back();
}

}  // namespace gh
