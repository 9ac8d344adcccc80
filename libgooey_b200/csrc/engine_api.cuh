// engine_api.cuh — extern "C" surface of include/gooey.h over engine.cuh (reference: src/ffi.rs, cited per function in
// the header).  Conventions follow the reference: null / out-of-range arguments are ignored, nothing throws across the
// boundary; a device failure latches the engine's sticky error and zero-fills the output (ffi.rs:2079-2121).
#pragma once
#include <thread>
#include "engine.cuh"
#include "music.h"
#include "../../include/gooey.h"

namespace gh {
static thread_local int g_cur_device = 0;
EngineBank& engine_bank(int device, float sr) {
  static std::mutex mu;
  static std::map<std::pair<int, uint32_t>, EngineBank*> banks;
  std::lock_guard<std::mutex> lk(mu);
  uint32_t key; memcpy(&key, &sr, 4);
  auto it = banks.find({device, key});
  if (it == banks.end()) it = banks.emplace(std::make_pair(device, key), new EngineBank(device, sr)).first;
  return *it->second;
}
static GooeyEngine::Voice* strip_by_type(GooeyEngine* e, uint32_t type) {
  for (int c = 0; c < N_STRIPS; c++) if (e->voice[c].type == type) return &e->voice[c];
  return nullptr;
}
static void strip_set_param(GooeyEngine::Voice* s, uint32_t param, float value) {
  if (!s) return;
  ffi_param_to_events(s->type, param, value, [&](uint32_t kind, uint32_t p, float v) { s->pending.push_back(make_event(0, kind, p, v)); });
}
// Slot of a global effect.  Tilt / delay / spring / plate own slots 0-3 from construction; the other five reorderable
// effects are built in a free slot the first time the host touches them (until then they sit, disabled, in their constructor
// state, which nothing can observe).  -1: not a slot effect (limiter, unknown id) or no slot left (sticky error).
static int gslot_ensure(GooeyEngine* e, uint32_t effect) {
  if (effect > 9 || effect == gd::FXK_LIMITER) return -1;
  if (e->cfg.gslot[effect] != 0xff) return e->cfg.gslot[effect];
  for (int s = gd::FXS_RACK0; s < gd::MAX_FX; s++)
    if (e->cfg.fx_kind[s] == gd::FXK_NONE) {
      e->cfg.fx_kind[s] = effect; e->cfg.fx_enabled[s] = 0; e->cfg.gslot[effect] = (uint8_t)s;
      e->mix_pending.push_back(make_event(0, gd::MX_FX_INIT, s, e->bpm, effect));
      return s;
    }
  engine_fail(e, "libgooey_b200: more than 8 track-rack + saturation/compressor/lowpass/waveshaper effect instances on one engine");
  return -1;
}
static void sync_cfg(GooeyEngine* e) {
  EngineBank& B = *e->bank;
  std::lock_guard<std::recursive_mutex> lk(B.mu);
  B.cfgs[e->mix_slot] = e->cfg;
}
static uint32_t bounce_frames(const GooeyEngine* e, uint32_t bars) {   // ffi.rs:7836-7838 / bounce.rs:20-32
  double spb = 4.0 * (60.0 / (double)e->bpm) * (double)e->sr;
  double tot = round((double)bars * spb);
  if (!(tot > 0.0)) return 0;
  return tot >= 4294967295.0 ? 0xffffffffu : (uint32_t)tot;
}
}  // namespace gh

const float GOOEY_POLY_PRESETS[5][14] = {   // PolySynthConfig::{default,pad,pluck,keys,strings} (poly_synth.rs:49-142), ffi preset ids 0-4
    {0.0f, 0.2f, 0.6f, 0.15f, 0.3f, 0.55f, 0.7f, 0.7f, 0.8f, 0.5f, 0.65f, 0.4f, 0.75f, 0.7f},
    {0.0f, 0.4f, 0.45f, 0.2f, 0.2f, 0.8f, 0.75f, 0.8f, 0.85f, 0.75f, 0.7f, 0.5f, 0.8f, 0.6f},
    {0.3f, 0.1f, 0.7f, 0.25f, 0.6f, 0.0f, 0.75f, 0.0f, 0.65f, 0.0f, 0.7f, 0.1f, 0.65f, 0.7f},
    {0.5f, 0.15f, 0.55f, 0.1f, 0.4f, 0.35f, 0.7f, 0.5f, 0.75f, 0.3f, 0.65f, 0.3f, 0.7f, 0.7f},
    {0.0f, 0.5f, 0.5f, 0.1f, 0.15f, 0.85f, 0.7f, 0.9f, 0.85f, 0.8f, 0.7f, 0.6f, 0.8f, 0.5f}};

extern "C" {

int gooey_b200_set_device(int device) {
  if (device < 0 || device >= gh::device_count()) { gh::set_error("device index out of range"); return GOOEY_E_INVALID; }
  gh::g_cur_device = device;
  return GOOEY_E_OK;
}

GooeyEngine* gooey_engine_new(float sample_rate) {
  try {
    if (!(sample_rate > 0.0f)) { gh::set_error("sample_rate must be > 0"); return nullptr; }
    gh::use_device(gh::g_cur_device);
    return gh::engine_create(gh::g_cur_device, sample_rate);
  } catch (const std::exception& ex) { gh::set_error(ex.what()); return nullptr; }
}
void gooey_engine_free(GooeyEngine* e) { try { gh::engine_destroy(e); } catch (...) {} }

bool gooey_engine_has_error(const GooeyEngine* e) { return e ? e->has_error : false; }
const char* gooey_engine_get_error_message(const GooeyEngine* e) { return (e && e->has_error) ? e->error.c_str() : nullptr; }
void gooey_engine_set_error_callback(GooeyEngine* e, void* ctx, void (*cb)(void*, const char*)) { if (e) { e->error_cb = cb; e->error_ctx = ctx; } }

void gooey_engine_set_kick_param(GooeyEngine* e, uint32_t p, float v) { if (e) gh::strip_set_param(gh::strip_by_type(e, GOOEY_INSTRUMENT_KICK), p, v); }
void gooey_engine_set_snare_param(GooeyEngine* e, uint32_t p, float v) { if (e) gh::strip_set_param(gh::strip_by_type(e, GOOEY_INSTRUMENT_SNARE), p, v); }
void gooey_engine_set_hihat_param(GooeyEngine* e, uint32_t p, float v) { if (e) gh::strip_set_param(gh::strip_by_type(e, GOOEY_INSTRUMENT_HIHAT), p, v); }
void gooey_engine_set_tom_param(GooeyEngine* e, uint32_t p, float v) { if (e) gh::strip_set_param(gh::strip_by_type(e, GOOEY_INSTRUMENT_TOM), p, v); }
void gooey_engine_set_bass_param(GooeyEngine* e, uint32_t p, float v) { if (e) gh::strip_set_param(gh::strip_by_type(e, GOOEY_INSTRUMENT_BASS), p, v); }
void gooey_engine_set_channel_param(GooeyEngine* e, uint32_t ch, uint32_t p, float v) { if (e && ch < 5) gh::strip_set_param(&e->voice[ch], p, v); }
// ffi.rs:2304-2343: a different synthesizer type on `channel`; the new instrument is `<Voice>::new(sample_rate)` and
// starts fresh, the strip (gain, pan, mute / solo, sequencer pattern) is kept.  Parameter edits still queued for the old
// instrument were applied to it (and die with it).
void gooey_engine_set_channel_instrument_type(GooeyEngine* e, uint32_t ch, uint32_t type) {
  if (!e || ch >= 5 || type > GOOEY_INSTRUMENT_BASS) return;
  GooeyEngine::Voice& v = e->voice[ch];
  GooeyEngine::Strip& s = e->strip[ch];
  if (v.type == type) return;
  try {
    gh::EngineBank& B = *e->bank;
    std::lock_guard<std::recursive_mutex> lk(B.mu);
    const GooeyVoicePatch p = gh::default_patch(type);
    const int slot = B.voices.create(p, e->sr);
    if (slot < 0) return;
    B.voices.release(v.type, v.slot);
    v.type = type; v.slot = slot;
    v.pending.clear();
    v.pending.push_back(gh::make_event(0, gd::EV_SET_TIME, 0, 0.0f, e->k));   // the fresh voice joins the engine's clock
    s.blender.default_for_type(type);                                          // ffi.rs:2334-2342
    if (s.blend_enabled) s.blender.apply(s.blend_x, s.blend_y, 0, [&](const gd::VoiceEvent& x) { v.pending.push_back(x); });
  } catch (const std::exception& ex) { gh::set_error(ex.what()); gh::engine_fail(e, ex.what()); }
}
uint32_t gooey_engine_get_channel_instrument_type(const GooeyEngine* e, uint32_t ch) { return (e && ch < 5) ? e->voice[ch].type : 0xFFFFFFFFu; }   /* :2354-2371 */

// ---- LFO pool (ffi.rs:4616-4993): eight tempo-synced sine LFOs, each routed to up to 16 (channel, parameter, depth) targets ----
uint32_t gooey_engine_lfo_count(void) { return 8; }
uint32_t gooey_engine_lfo_timing_count(void) { return 8; }
void gooey_engine_set_lfo_enabled(GooeyEngine* e, uint32_t i, bool on) { if (e && i < 8) e->lfo_enabled[i] = on; }
bool gooey_engine_get_lfo_enabled(const GooeyEngine* e, uint32_t i) { return e && i < 8 && e->lfo_enabled[i]; }
void gooey_engine_set_lfo_timing(GooeyEngine* e, uint32_t i, uint32_t timing) { if (e && i < 8 && timing < 8) e->lfos[i].division = timing; }
uint32_t gooey_engine_get_lfo_timing(const GooeyEngine* e, uint32_t i) { return (e && i < 8) ? e->lfos[i].division : 0xFFFFFFFFu; }
void gooey_engine_set_lfo_amount(GooeyEngine* e, uint32_t i, float a) { if (e && i < 8) e->lfos[i].amount = a; }
float gooey_engine_get_lfo_amount(const GooeyEngine* e, uint32_t i) { return (e && i < 8) ? e->lfos[i].amount : 0.0f; }
void gooey_engine_set_lfo_offset(GooeyEngine* e, uint32_t i, float o) { if (e && i < 8) e->lfos[i].offset = o; }
float gooey_engine_get_lfo_offset(const GooeyEngine* e, uint32_t i) { return (e && i < 8) ? e->lfos[i].offset : 0.0f; }
uint32_t gooey_engine_add_lfo_route(GooeyEngine* e, uint32_t i, uint32_t instrument, uint32_t param, float depth) {
  if (!e || i >= 8 || e->lfo_routes[i].size() >= 16) return 0xFFFFFFFFu;
  const uint32_t id = e->lfo_next_route_id[i]++;
  e->lfo_routes[i].push_back({id, instrument, param, depth});
  return id;
}
bool gooey_engine_remove_lfo_route(GooeyEngine* e, uint32_t i, uint32_t route_id) {
  if (!e || i >= 8) return false;
  auto& r = e->lfo_routes[i];
  for (size_t k = 0; k < r.size(); k++) if (r[k].id == route_id) { r.erase(r.begin() + k); return true; }
  return false;
}
void gooey_engine_clear_lfo_routes(GooeyEngine* e, uint32_t i) { if (e && i < 8) e->lfo_routes[i].clear(); }
uint32_t gooey_engine_get_lfo_route_count(const GooeyEngine* e, uint32_t i) { return (e && i < 8) ? (uint32_t)e->lfo_routes[i].size() : 0u; }
void gooey_engine_reset_lfo_phase(GooeyEngine* e, uint32_t i) { if (e && i < 8) e->lfos[i].phase = 0.0f; }
float gooey_engine_get_lfo_phase(const GooeyEngine* e, uint32_t i) { return (e && i < 8) ? e->lfos[i].phase : -1.0f; }

// ---- preset blend: 2-D pad over four corner presets (ffi.rs:5245-5490) and per-step blends (:4009-4075, 4314-4380) ----
void gooey_engine_blend_enable(GooeyEngine* e, uint32_t inst) { if (e && inst < 5) e->strip[inst].blend_enabled = true; }
void gooey_engine_blend_disable(GooeyEngine* e, uint32_t inst) { if (e && inst < 5) e->strip[inst].blend_enabled = false; }
bool gooey_engine_blend_is_enabled(const GooeyEngine* e, uint32_t inst) { return e && inst < 5 && e->strip[inst].blend_enabled; }
void gooey_engine_blend_set_position(GooeyEngine* e, uint32_t inst, float x, float y) {
  if (!e || inst >= 5) return;
  GooeyEngine::Strip& s = e->strip[inst];
  if (!s.blend_enabled) return;
  s.blend_x = gd::clampf(x, 0.0f, 1.0f); s.blend_y = gd::clampf(y, 0.0f, 1.0f);
  s.blender.apply(s.blend_x, s.blend_y, 0, [&](const gd::VoiceEvent& ev) { e->voice[inst].pending.push_back(ev); });
}
float gooey_engine_blend_get_position_x(const GooeyEngine* e, uint32_t inst) { return (e && inst < 5) ? e->strip[inst].blend_x : -1.0f; }
float gooey_engine_blend_get_position_y(const GooeyEngine* e, uint32_t inst) { return (e && inst < 5) ? e->strip[inst].blend_y : -1.0f; }
void gooey_engine_blend_set_corner_preset(GooeyEngine* e, uint32_t inst, uint32_t corner, uint32_t preset_id) {
  if (!e || inst >= 5 || corner >= 4) return;
  e->strip[inst].blender.corner_ids[corner] = preset_id;
  e->strip[inst].blender.set_corner_preset(corner, preset_id);
}
uint32_t gooey_engine_blend_get_corner_preset(const GooeyEngine* e, uint32_t inst, uint32_t corner) {
  return (e && inst < 5 && corner < 4) ? e->strip[inst].blender.corner_ids[corner] : 0xFFFFFFFFu;
}
void gooey_engine_blend_reset_corners(GooeyEngine* e, uint32_t inst) { if (e && inst < 5) e->strip[inst].blender.default_for_type(e->voice[inst].type); }
void gooey_engine_sequencer_set_instrument_step_blend(GooeyEngine* e, uint32_t inst, uint32_t step, float x, float y) {
  if (!e || inst >= 5 || step >= e->strip[inst].seq.pattern.size()) return;
  gh::SeqStep& st = e->strip[inst].seq.pattern[step];
  st.has_blend = true; st.bx = gd::clampf(x, 0.0f, 1.0f); st.by = gd::clampf(y, 0.0f, 1.0f);
}
void gooey_engine_sequencer_set_instrument_step_blend_override(GooeyEngine* e, uint32_t inst, uint32_t step, float x, float y) { gooey_engine_sequencer_set_instrument_step_blend(e, inst, step, x, y); }
void gooey_engine_sequencer_clear_instrument_step_blend(GooeyEngine* e, uint32_t inst, uint32_t step) {
  if (!e || inst >= 5 || step >= e->strip[inst].seq.pattern.size()) return;
  e->strip[inst].seq.pattern[step].has_blend = false;
}
void gooey_engine_sequencer_clear_instrument_step_blend_override(GooeyEngine* e, uint32_t inst, uint32_t step) { gooey_engine_sequencer_clear_instrument_step_blend(e, inst, step); }
float gooey_engine_sequencer_get_instrument_step_blend_x(const GooeyEngine* e, uint32_t inst, uint32_t step) {
  if (!e || inst >= 5 || step >= e->strip[inst].seq.pattern.size() || !e->strip[inst].seq.pattern[step].has_blend) return -1.0f;
  return e->strip[inst].seq.pattern[step].bx;
}
float gooey_engine_sequencer_get_instrument_step_blend_y(const GooeyEngine* e, uint32_t inst, uint32_t step) {
  if (!e || inst >= 5 || step >= e->strip[inst].seq.pattern.size() || !e->strip[inst].seq.pattern[step].has_blend) return -1.0f;
  return e->strip[inst].seq.pattern[step].by;
}

void gooey_engine_load_bass_preset(GooeyEngine* e, uint32_t id) {   // BassConfig::{acid,sub,reese,stab} (gh::preset_flat); set_config = 15 set_targets
  GooeyEngine::Voice* bass = e ? gh::strip_by_type(e, GOOEY_INSTRUMENT_BASS) : nullptr;
  float v[24];
  if (!bass || gh::preset_flat(GOOEY_INSTRUMENT_BASS, id, v) == 0) return;
  for (uint32_t i = 0; i < 15; i++) bass->pending.push_back(gh::make_event(0, gd::EV_SET_TARGET, i, gh::clamp01(v[i])));
}

void gooey_engine_set_bpm(GooeyEngine* e, float bpm) {
  if (!e) return;
  e->bpm = bpm;
  e->loop_engine_bpm = bpm;                                    // Mixer::set_bpm (ffi.rs:3360, mixer/mod.rs:80-87)
  e->transport.set_bpm(bpm);
  for (auto& s : e->strip) s.seq.set_bpm(bpm);
  for (auto& R : e->samplers) if (R.registered) R.pat.seq.set_bpm(bpm);
  for (int slot = 0; slot < gd::MAX_FX; slot++)
    if (e->cfg.fx_kind[slot] == gd::FXK_DELAY) e->mix_pending.push_back(gh::make_event(0, gd::MX_FX_BPM, slot, bpm));
}
float gooey_engine_get_bpm(const GooeyEngine* e) { return e ? e->bpm : 120.0f; }
void gooey_engine_set_swing(GooeyEngine* e, float swing) {
  if (!e) return;
  float c = gd::clampf(swing, 0.0f, 1.0f);
  e->swing = c;
  for (auto& s : e->strip) s.seq.set_swing(c);
  for (auto& R : e->samplers) if (R.registered) R.pat.seq.set_swing(c);
}
void gooey_engine_set_master_gain(GooeyEngine* e, float g) { if (e && std::isfinite(g)) e->mix_pending.push_back(gh::make_event(0, gd::MX_SET, gd::MP_MASTER, g)); }

void gooey_engine_sequencer_set_instrument_step_settings(GooeyEngine* e, uint32_t inst, uint32_t step, bool enabled, bool set_vel, float vel,
                                                         bool set_blend, float bx, float by, bool set_note, uint8_t note) {
  if (!e || inst >= 5) return;
  auto& pat = e->strip[inst].seq.pattern;
  if (step >= pat.size()) return;
  gh::SeqStep& st = pat[step];
  st.enabled = enabled;
  if (set_vel) st.velocity = gd::clampf(vel, 0.0f, 1.0f);
  if (set_blend) { st.has_blend = true; st.bx = gd::clampf(bx, 0.0f, 1.0f); st.by = gd::clampf(by, 0.0f, 1.0f); }
  if (set_note) { if (note == 255) st.has_note = false; else { st.has_note = true; st.note = note; } }
}
void gooey_engine_sequencer_set_instrument_step(GooeyEngine* e, uint32_t inst, uint32_t step, bool enabled) {
  if (!e || inst >= 5) return;
  auto& pat = e->strip[inst].seq.pattern;
  if (step < pat.size()) pat[step].enabled = enabled;
}
void gooey_engine_sequencer_set_step(GooeyEngine* e, uint32_t step, bool enabled) { gooey_engine_sequencer_set_instrument_step(e, 0, step, enabled); }
void gooey_engine_sequencer_set_instrument_step_with_velocity(GooeyEngine* e, uint32_t inst, uint32_t step, bool enabled, float vel) {
  if (!e || inst >= 5) return;
  auto& pat = e->strip[inst].seq.pattern;
  if (step < pat.size()) { pat[step].enabled = enabled; pat[step].velocity = gd::clampf(vel, 0.0f, 1.0f); }
}
void gooey_engine_sequencer_set_instrument_step_note(GooeyEngine* e, uint32_t inst, uint32_t step, uint8_t note) {
  if (!e || inst >= 5) return;
  auto& pat = e->strip[inst].seq.pattern;
  if (step < pat.size()) { if (note == 255) pat[step].has_note = false; else { pat[step].has_note = true; pat[step].note = note; } }
}
void gooey_engine_sequencer_set_instrument_pattern(GooeyEngine* e, uint32_t inst, const bool* pattern) {
  if (!e || !pattern || inst >= 5) return;
  gh::HostSeq& q = e->strip[inst].seq;
  q.pattern.assign(16, gh::SeqStep());            // SequencerStep::from(bool): velocity 1, no blend, no note
  for (int i = 0; i < 16; i++) q.pattern[i].enabled = pattern[i];
  if (q.current_step >= q.pattern.size()) q.current_step = 0;
}
// ffi.rs:3501-3561: every sequencer — the strips' and the registered sampler racks' — plus the mixer's transport (the beat clock the
// racks' pattern starts are armed on); stop / reset also drop the racks' pending starts, patterns and sounding voices
void gooey_engine_sequencer_start(GooeyEngine* e) {
  if (!e) return;
  for (auto& s : e->strip) s.seq.start();
  for (auto& R : e->samplers) if (R.registered) R.pat.seq.start();
  e->transport.running = true;
}
void gooey_engine_sequencer_stop(GooeyEngine* e) {
  if (!e) return;
  for (auto& s : e->strip) s.seq.stop();
  for (auto& R : e->samplers) if (R.registered) { R.pat.has_pending = false; R.pat.pattern_running = false; R.pat.seq.stop(); R.stop_all(); }
  e->transport.now();
  e->transport.running = false;
}
void gooey_engine_sequencer_reset(GooeyEngine* e) {
  if (!e) return;
  for (auto& s : e->strip) s.seq.reset();
  for (auto& R : e->samplers) if (R.registered) { R.pat.has_pending = false; R.pat.pattern_running = false; R.pat.seq.reset(); R.stop_all(); }
  e->transport.beat = 0.0; e->transport.lazy = 0;
}
// ffi.rs:2188-2215: with the triggers disabled the sequencers keep ticking (clock, step position) but fire nothing and export no
// MIDI event; host triggers (trigger_instrument*) still sound.  The render path reads the flag per call (engine.cuh).
void gooey_engine_set_sequencer_triggers_enabled(GooeyEngine* e, bool enabled) { if (e) e->seq_triggers_enabled = enabled; }
bool gooey_engine_get_sequencer_triggers_enabled(const GooeyEngine* e) { return e ? e->seq_triggers_enabled : true; }     // null: the safe default of ffi.rs:2209-2211

void gooey_engine_set_instrument_gain(GooeyEngine* e, uint32_t i, float g) { if (e && i < 5) e->mix_pending.push_back(gh::make_event(0, gd::MX_SET, gd::MP_CH_GAIN + i, gd::clampf(g, 0.0f, 1.0f))); }
void gooey_engine_set_instrument_pan(GooeyEngine* e, uint32_t i, float p) { if (e && i < 5) e->mix_pending.push_back(gh::make_event(0, gd::MX_SET, gd::MP_CH_PAN + i, gd::clampf(p, 0.0f, 1.0f))); }
void gooey_engine_set_instrument_mute(GooeyEngine* e, uint32_t i, bool m) { if (e && i < 5) e->strip[i].muted = m; }
void gooey_engine_set_instrument_solo(GooeyEngine* e, uint32_t i, bool s) { if (e && i < 5) e->strip[i].soloed = s; }
void gooey_engine_trigger_instrument_with_velocity(GooeyEngine* e, uint32_t i, float v) {
  if (e && i < 5) { e->strip[i].trig_vel = gd::clampf(v, 0.0f, 1.0f); e->strip[i].trig_pending = true; }
}
void gooey_engine_trigger_instrument(GooeyEngine* e, uint32_t i) { gooey_engine_trigger_instrument_with_velocity(e, i, 1.0f); }

void gooey_engine_set_global_effect_param(GooeyEngine* e, uint32_t fx, uint32_t p, float v) {
  if (!e) return;
  if (fx == gd::FXK_LIMITER) {
    if (p == 0 && std::isfinite(v)) { float t = gd::clampf(v, 0.001f, 1.0f); e->cfg.lim_th = t; e->cfg.lim_inv = 1.0f / t; gh::sync_cfg(e); }
    return;
  }
  const int slot = gh::gslot_ensure(e, fx);
  if (slot >= 0 && p < 256) e->mix_pending.push_back(gh::make_event(0, gd::MX_FX_SET, ((uint32_t)slot << 8) | p, v));
  if (slot >= 0) gh::sync_cfg(e);
}
void gooey_engine_set_global_effect_enabled(GooeyEngine* e, uint32_t fx, bool on) {
  if (!e) return;
  if (fx == gd::FXK_LIMITER) e->cfg.limiter_on = on;
  else { const int slot = gh::gslot_ensure(e, fx); if (slot < 0) return; e->cfg.fx_enabled[slot] = on; }
  gh::sync_cfg(e);
}
bool gooey_engine_get_global_effect_enabled(const GooeyEngine* e, uint32_t fx) {   /* :3214-3237 */
  if (!e || fx > 9) return false;
  if (fx == gd::FXK_LIMITER) return e->cfg.limiter_on != 0;
  const uint32_t slot = e->cfg.gslot[fx];
  return slot < (uint32_t)gd::MAX_FX && e->cfg.fx_enabled[slot] != 0;
}
void gooey_engine_set_compressor_sidechain(GooeyEngine* e, uint32_t instrument) { if (e) { e->cfg.comp_sidechain = instrument; gh::sync_cfg(e); } }   /* :3252-3265 */
uint32_t gooey_engine_get_compressor_sidechain(const GooeyEngine* e) { return e ? e->cfg.comp_sidechain : 0xFFFFFFFFu; }
static bool gooey_reorderable(uint32_t id) { return id <= 9 && id != gd::FXK_LIMITER; }
bool gooey_engine_set_effect_order(GooeyEngine* e, const uint32_t* ids, uint32_t len) {   // a permutation of the 9 reorderable ids (:4498-4528)
  if (!e || !ids || len != 9) return false;
  for (uint32_t i = 0; i < 9; i++) { if (!gooey_reorderable(ids[i])) return false; for (uint32_t j = 0; j < i; j++) if (ids[j] == ids[i]) return false; }
  for (uint32_t i = 0; i < 9; i++) e->cfg.order[i] = ids[i];
  e->mix_pending.push_back(gh::make_event(0, gd::MX_FX_RESET, 0, 0.0f));   // reset_effect_states
  gh::sync_cfg(e);
  return true;
}
bool gooey_engine_move_effect(GooeyEngine* e, uint32_t effect_id, uint32_t new_position) {   /* :4544-4581 */
  if (!e || !gooey_reorderable(effect_id) || new_position >= 9) return false;
  int cur = -1;
  for (int i = 0; i < 9; i++) if (e->cfg.order[i] == effect_id) cur = i;
  if (cur < 0) return false;
  const int np = (int)new_position;
  if (cur == np) return true;
  if (np > cur) for (int i = cur; i < np; i++) e->cfg.order[i] = e->cfg.order[i + 1];
  else for (int i = cur - 1; i >= np; i--) e->cfg.order[i + 1] = e->cfg.order[i];
  e->cfg.order[np] = effect_id;
  e->mix_pending.push_back(gh::make_event(0, gd::MX_FX_RESET, 0, 0.0f));
  gh::sync_cfg(e);
  return true;
}
uint32_t gooey_engine_get_effect_order(const GooeyEngine* e, uint32_t* out_ids, uint32_t max_len) {   /* :4596-4615 */
  if (!e || !out_ids || max_len == 0) return 0;
  const uint32_t n = max_len < 9 ? max_len : 9;
  for (uint32_t i = 0; i < n; i++) out_ids[i] = e->cfg.order[i];
  return n;
}

int32_t gooey_engine_mixer_add_track(GooeyEngine* e, const char*) {
  if (!e || e->cfg.n_tracks >= gd::MAX_TRACKS) return -1;
  const uint32_t t = e->cfg.n_tracks++;
  e->cfg.rack_n[t] = 0;
  e->track_muted[t] = e->track_soloed[t] = false;
  e->track_gain_t[t] = 1.0f; e->track_pan_t[t] = 0.5f;
  e->mix_pending.push_back(gh::make_event(0, gd::MX_TRACK_INIT, t, 0.0f));
  gh::sync_cfg(e);
  return (int32_t)t;
}
uint32_t gooey_engine_mixer_get_track_count(const GooeyEngine* e) { return e ? e->cfg.n_tracks : 0; }
bool gooey_engine_mixer_route_source(GooeyEngine* e, uint32_t src, uint32_t track) {
  // MixerGraph::route (graph.rs:243-250): the five fixed sources, and sampler racks once registered (source 5 + rack)
  if (!e || src >= 9 || track >= e->cfg.n_tracks) return false;
  if (src >= 5 && !e->samplers[src - 5].registered) return false;
  e->cfg.route[src] = (int32_t)track;
  gh::sync_cfg(e);
  return true;
}
void gooey_engine_mixer_set_track_gain(GooeyEngine* e, uint32_t t, float g) {
  if (!e || t >= e->cfg.n_tracks) return;
  const float c = gd::clampf(g, 0.0f, 2.0f);
  if (fabsf(e->track_gain_t[t] - c) > 1e-8f) e->track_gain_t[t] = c;            // SmoothedParam::set_target keeps the old target within 1e-8
  e->mix_pending.push_back(gh::make_event(0, gd::MX_SET, gd::MP_TR_GAIN + t, c));
}
void gooey_engine_mixer_set_track_pan(GooeyEngine* e, uint32_t t, float p) {
  if (!e || t >= e->cfg.n_tracks) return;
  const float c = gd::clampf(p, 0.0f, 1.0f);
  if (fabsf(e->track_pan_t[t] - c) > 1e-8f) e->track_pan_t[t] = c;
  e->mix_pending.push_back(gh::make_event(0, gd::MX_SET, gd::MP_TR_PAN + t, c));
}
// strip getters (ffi.rs:6472-6566): the targets, with the reference's defaults for a bad index
float gooey_engine_mixer_get_track_gain(const GooeyEngine* e, uint32_t t) { return (e && t < e->cfg.n_tracks) ? e->track_gain_t[t] : 1.0f; }
float gooey_engine_mixer_get_track_pan(const GooeyEngine* e, uint32_t t) { return (e && t < e->cfg.n_tracks) ? e->track_pan_t[t] : 0.5f; }
bool gooey_engine_mixer_get_track_mute(const GooeyEngine* e, uint32_t t) { return e && t < e->cfg.n_tracks && e->track_muted[t]; }
bool gooey_engine_mixer_get_track_solo(const GooeyEngine* e, uint32_t t) { return e && t < e->cfg.n_tracks && e->track_soloed[t]; }
// graph routes and layout (ffi.rs:6291-6320, 6427-6455; graph.rs:131-149, 253-266)
static bool source_is_active(const GooeyEngine* e, uint32_t src) { return src < 5 || (src < 9 && e->samplers[src - 5].registered); }
bool gooey_engine_mixer_unroute_source(GooeyEngine* e, uint32_t src) {
  if (!e || !source_is_active(e, src)) return false;
  const bool had = e->cfg.route[src] >= 0;
  e->cfg.route[src] = -1;
  gh::sync_cfg(e);
  return had;
}
int32_t gooey_engine_mixer_get_source_route(const GooeyEngine* e, uint32_t src) { return (e && source_is_active(e, src)) ? e->cfg.route[src] : -1; }
bool gooey_engine_track_effect_remove(GooeyEngine* e, uint32_t t, uint32_t pos);
void gooey_engine_mixer_clear_layout(GooeyEngine* e) {   // MixerGraph::reset: no tracks (their racks go with them), no routes; registered sources stay registered
  if (!e) return;
  for (uint32_t t = 0; t < e->cfg.n_tracks; t++) while (e->cfg.rack_n[t]) gooey_engine_track_effect_remove(e, t, 0);
  e->cfg.n_tracks = 0;
  for (int s = 0; s < 9; s++) e->cfg.route[s] = -1;
  for (int t = 0; t < gd::MAX_TRACKS; t++) e->track_muted[t] = e->track_soloed[t] = false;
  gh::sync_cfg(e);
}
int32_t gooey_engine_mixer_add_track(GooeyEngine* e, const char*);
void gooey_engine_mixer_reset_default_layout(GooeyEngine* e) {   // MixerGraph::with_default_layout: Drums / Bass / Synth / Loops, fresh strips, the five fixed routes
  if (!e) return;
  gooey_engine_mixer_clear_layout(e);
  for (int t = 0; t < 4; t++) gooey_engine_mixer_add_track(e, "");
  const int32_t routes[5] = {0, 1, 2, 3, 3};
  for (int s = 0; s < 5; s++) e->cfg.route[s] = routes[s];
  gh::sync_cfg(e);
}
void gooey_engine_mixer_set_track_mute(GooeyEngine* e, uint32_t t, bool m) { if (e && t < e->cfg.n_tracks) e->track_muted[t] = m; }
void gooey_engine_mixer_set_track_solo(GooeyEngine* e, uint32_t t, bool s) { if (e && t < e->cfg.n_tracks) e->track_soloed[t] = s; }
int32_t gooey_engine_track_effect_add(GooeyEngine* e, uint32_t t, uint32_t fx) {   // ChannelEffect::from_id (effect_chain.rs:57-109): every effect but the limiter
  if (!e || t >= e->cfg.n_tracks) return -1;
  if (!gooey_reorderable(fx)) return -1;
  if (e->cfg.rack_n[t] >= 4) { gh::engine_fail(e, "libgooey_b200: a track rack holds at most 4 effects"); return -1; }
  int slot = -1;
  for (int s = gd::FXS_RACK0; s < gd::MAX_FX; s++) if (e->cfg.fx_kind[s] == gd::FXK_NONE) { slot = s; break; }
  if (slot < 0) { gh::engine_fail(e, "libgooey_b200: more than 8 track-rack + saturation/compressor/lowpass/waveshaper effect instances on one engine"); return -1; }
  e->cfg.fx_kind[slot] = fx; e->cfg.fx_enabled[slot] = 1; e->cfg.fx_rack |= 1u << slot;
  const uint32_t pos = e->cfg.rack_n[t]++;
  e->cfg.rack_slot[t][pos] = (uint8_t)slot;
  e->mix_pending.push_back(gh::make_event(0, gd::MX_FX_INIT, slot, e->bpm, fx | 0x100u));
  gh::sync_cfg(e);
  return (int32_t)pos;
}
// A removed effect frees its slot; queued edits that were addressed to it are dropped with it (they were applied to an effect
// that no longer exists).  Ring memory of the slot is cleared when the slot is constructed again (MX_FX_INIT).
bool gooey_engine_track_effect_remove(GooeyEngine* e, uint32_t t, uint32_t pos) {   /* :6607-6616, effect_chain.rs:310-317 */
  if (!e || t >= e->cfg.n_tracks || pos >= e->cfg.rack_n[t]) return false;
  const uint32_t slot = e->cfg.rack_slot[t][pos];
  for (uint32_t k = pos; k + 1 < e->cfg.rack_n[t]; k++) e->cfg.rack_slot[t][k] = e->cfg.rack_slot[t][k + 1];
  e->cfg.rack_n[t]--;
  e->cfg.fx_kind[slot] = gd::FXK_NONE; e->cfg.fx_enabled[slot] = 0; e->cfg.fx_rack &= ~(1u << slot);
  auto& mp = e->mix_pending;
  mp.erase(std::remove_if(mp.begin(), mp.end(), [&](const gd::VoiceEvent& v) {
    return ((v.kind == gd::MX_FX_SET && (uint32_t)(v.param >> 8) == slot) || ((v.kind == gd::MX_FX_INIT || v.kind == gd::MX_FX_BPM) && v.param == slot)); }), mp.end());
  gh::sync_cfg(e);
  return true;
}
bool gooey_engine_track_effect_move(GooeyEngine* e, uint32_t t, uint32_t pos, uint32_t new_position) {   /* :6623-6640, effect_chain.rs:322-330 */
  if (!e || t >= e->cfg.n_tracks || pos >= e->cfg.rack_n[t]) return false;
  const uint32_t n = e->cfg.rack_n[t];
  uint8_t tmp[4]; uint32_t m = 0;
  const uint8_t moved = e->cfg.rack_slot[t][pos];
  for (uint32_t k = 0; k < n; k++) if (k != pos) tmp[m++] = e->cfg.rack_slot[t][k];
  const uint32_t dest = new_position < m ? new_position : m;
  for (uint32_t k = 0, j = 0; k < n; k++) e->cfg.rack_slot[t][k] = (k == dest) ? moved : tmp[j++];
  gh::sync_cfg(e);
  return true;
}
uint32_t gooey_engine_track_effect_count(const GooeyEngine* e, uint32_t t) { return (e && t < e->cfg.n_tracks) ? e->cfg.rack_n[t] : 0; }
void gooey_engine_track_effect_set_param(GooeyEngine* e, uint32_t t, uint32_t pos, uint32_t p, float v) {
  if (!e || t >= e->cfg.n_tracks || pos >= e->cfg.rack_n[t] || p >= 256) return;
  e->mix_pending.push_back(gh::make_event(0, gd::MX_FX_SET, ((uint32_t)e->cfg.rack_slot[t][pos] << 8) | p, v));
}

// ---- poly synth (ffi.rs:5571-5648, 5899-5935; poly_synth.rs) ----
void gooey_engine_poly_set_preset(GooeyEngine* e, uint32_t preset) {   // set_config: 14 smoothed targets, no snap
  if (!e) return;
  auto& pending = gh::aux_touch(e, gh::CH_POLY);
  const float* t = GOOEY_POLY_PRESETS[preset < 5 ? preset : 0];
  for (uint32_t i = 0; i < 14; i++) pending.push_back(gh::make_event(0, gd::EV_SET_TARGET, i, t[i]));
}
void gooey_engine_poly_set_param(GooeyEngine* e, uint32_t param, float value) {
  if (!e || param >= 14) return;
  gh::aux_touch(e, gh::CH_POLY).push_back(gh::make_event(0, gd::EV_SET_TARGET, param, gd::clampf(value, 0.0f, 1.0f)));
}
void gooey_engine_poly_release(GooeyEngine* e) {
  if (!e) return;
  gh::aux_touch(e, gh::CH_POLY).push_back(gh::make_event(0, gd::EV_POLY_RELEASE, 0, 0.0f));
}
// The tail of gooey_engine_poly_trigger_chord (ffi.rs:5594-5611) once `music::apply_voicing` has produced the MIDI notes:
// preset as smoothed targets, release_all, trigger every note.  (The chord -> notes tables of src/music are host-side
// integer logic outside this library's scope; SURVEY.md section 2 row 34.)
void gooey_engine_poly_trigger_notes(GooeyEngine* e, const uint8_t* notes, uint32_t n, uint32_t preset, float velocity) {
  if (!e || (!notes && n)) return;
  gooey_engine_poly_set_preset(e, preset);
  const float v = gd::clampf(velocity, 0.0f, 1.0f);
  e->voice[gh::CH_POLY].pending.push_back(gh::make_event(0, gd::EV_POLY_RELEASE, 0, 0.0f));
  for (uint32_t i = 0; i < n; i++) e->voice[gh::CH_POLY].pending.push_back(gh::make_event(0, gd::EV_POLY_NOTE, notes[i], v));
}

// ffi.rs:5571-5611: diatonic seventh chord of (root, scale) at `degree`, voiced, on the poly synth
void gooey_engine_poly_trigger_chord(GooeyEngine* e, uint32_t root, uint32_t scale_type, uint32_t degree, uint32_t voicing, uint32_t preset,
                                     int32_t octave, float velocity) {
  if (!e) return;
  const std::vector<uint8_t> notes = gh::chord_notes(root, scale_type, degree, voicing, octave);
  gooey_engine_poly_trigger_notes(e, notes.data(), (uint32_t)notes.size(), preset, velocity);
}
// host-only view of the table above (tests, hosts that want to display the notes)
uint32_t gooey_b200_chord_notes(uint32_t root, uint32_t scale_type, uint32_t degree, uint32_t voicing, int32_t octave, uint8_t* out_notes, uint32_t capacity) {
  const std::vector<uint8_t> notes = gh::chord_notes(root, scale_type, degree, voicing, octave);
  for (uint32_t i = 0; i < notes.size() && i < capacity; i++) if (out_notes) out_notes[i] = notes[i];
  return (uint32_t)notes.size();
}

// ---- granulator (ffi.rs:5969-5990, 7702-7827; granulator.rs) ----
static void gran_attach(GooeyEngine* e) { gh::gran_buffer_events(gh::aux_touch(e, gh::CH_GRAN), 0, e->gran_buf->p, e->gran_sr, e->gran_len); }
bool gooey_engine_granulator_set_buffer(GooeyEngine* e, const float* samples, uint32_t len, float sample_rate) {
  if (!e || !samples || len == 0) return false;
  if (!std::isfinite(sample_rate) || !(sample_rate > 0.0f)) return false;            // SampleBuffer::from_mono (granulator.rs:60-90)
  for (uint32_t i = 0; i < len; i++) if (!std::isfinite(samples[i])) return false;
  try {
    gh::use_device(e->bank->device);
    auto buf = std::make_shared<gh::DevBuf<float>>();
    buf->alloc(len);
    GH_CUDA(cudaMemcpy(buf->p, samples, (size_t)len * 4, cudaMemcpyHostToDevice));
    GH_CUDA(cudaStreamSynchronize(e->bank->stream));   // the previous buffer may still be read by an in-flight render
    e->gran_buf = buf; e->gran_len = len; e->gran_sr = sample_rate;
  } catch (const std::exception& ex) { gh::set_error(ex.what()); return false; }
  gran_attach(e);
  return true;
}
// libgooey_b200 addition: `dst` plays the buffer already loaded into `src` (same device) without another copy —
// thousands of granulators over one 60 s source keep one 10.6 MB buffer resident instead of one each.
bool gooey_b200_granulator_share_buffer(GooeyEngine* dst, const GooeyEngine* src) {
  if (!dst || !src || !src->gran_buf || dst->bank->device != src->bank->device) return false;
  try { gh::use_device(dst->bank->device); GH_CUDA(cudaStreamSynchronize(dst->bank->stream)); } catch (const std::exception& ex) { gh::set_error(ex.what()); return false; }
  dst->gran_buf = src->gran_buf; dst->gran_len = src->gran_len; dst->gran_sr = src->gran_sr;
  gran_attach(dst);
  return true;
}
void gooey_engine_granulator_trigger(GooeyEngine* e, float velocity) {
  if (!e) return;
  gh::aux_touch(e, gh::CH_GRAN).push_back(gh::make_event(0, gd::EV_TRIGGER, 0, gd::clampf(velocity, 0.0f, 1.0f)));
}
void gooey_engine_granulator_set_param(GooeyEngine* e, uint32_t param, float value) {
  if (!e || param >= 12) return;
  gh::aux_touch(e, gh::CH_GRAN).push_back(gh::make_event(0, gd::EV_SET_TARGET, param, gd::clampf(value, 0.0f, 1.0f)));
}
void gooey_engine_granulator_set_seed(GooeyEngine* e, uint32_t seed) {
  if (!e) return;
  gh::aux_touch(e, gh::CH_GRAN).push_back(gh::make_event(0, gd::EV_GRAN_SEED, 0, 0.0f, seed));
}
void gooey_engine_granulator_snap_params(GooeyEngine* e) {
  if (!e) return;
  gh::aux_touch(e, gh::CH_GRAN).push_back(gh::make_event(0, gd::EV_SNAP, 0, 0.0f));
}
uint32_t gooey_engine_granulator_buffer_len(const GooeyEngine* e) { return e ? e->gran_len : 0; }                        /* :7665 */
float gooey_engine_granulator_buffer_sample_rate(const GooeyEngine* e) { return e ? e->gran_sr : 0.0f; }               /* :7680 */

// Host-only: the trigger schedule the bounce of an engine with this tempo / swing / pattern resolves to (the frames at
// which kernel events are placed).  Needs no device; used by the CPU tests for the bit-exact trigger-index gate.
uint32_t gooey_b200_sequencer_schedule(float sample_rate, float bpm, float swing, const uint8_t* enabled, const float* velocity, uint32_t steps,
                                       uint32_t frames, uint32_t* out_frames, float* out_velocity, uint32_t capacity) {
  if (!enabled || steps == 0) return 0;
  gh::HostSeq q;
  q.init(120.0f, sample_rate);
  q.set_bpm(bpm);
  q.pattern.assign(steps, gh::SeqStep());
  for (uint32_t i = 0; i < steps; i++) { q.pattern[i].enabled = enabled[i] != 0; q.pattern[i].velocity = velocity ? gd::clampf(velocity[i], 0.0f, 1.0f) : 1.0f; }
  q.set_swing(swing);
  q.reset(); q.start();
  std::vector<gh::SeqFire> fires;
  q.run(frames, fires);
  uint32_t n = 0;
  for (const auto& f : fires) { if (n < capacity) { if (out_frames) out_frames[n] = f.frame; if (out_velocity) out_velocity[n] = f.velocity; } n++; }
  return n;
}

// Host-only: the pad hits one sampler rack's pattern resolves to over a sequence of render calls (gh::resolve_rack_patterns, the code
// engines_render runs).  steps: 16 x (enabled, pad, velocity).  The transport starts at `transport_beat` (running or not); the pattern start
// is armed at `pending_beat` (< 0: the pattern already runs from step 0 — a bounce); calls[i] frames are rendered one call after the other
// (`bounce`: every call is a bounce).  Hits come back with frames counted from the first call.  Returns their number (may exceed capacity);
// *out_transport_beat = the beat after the last call.  Needs no device; used by the CPU tests.
uint32_t gooey_b200_sampler_schedule(float sample_rate, float bpm, float swing, const uint8_t* enabled, const uint8_t* pads, const float* velocity,
                                     int transport_running, double transport_beat, double pending_beat, int bounce, const uint32_t* calls, uint32_t n_calls,
                                     uint32_t* out_frames, uint32_t* out_pads, float* out_velocity, uint32_t capacity, double* out_transport_beat) {
  if (!enabled || !pads || !calls) return 0;
  gh::Transport T;
  T.sr = sample_rate; T.bpm = 120.0f; T.set_bpm(bpm); T.running = transport_running != 0; T.beat = transport_beat;
  gh::RackPattern R;
  R.seq.init(bpm, sample_rate);
  for (int i = 0; i < 16; i++) { gh::SeqStep& s = R.seq.pattern[i]; s.enabled = enabled[i] != 0; s.velocity = velocity ? gd::clampf(velocity[i], 0.0f, 1.0f) : 1.0f; s.has_note = true; s.note = pads[i]; }
  R.seq.set_swing(swing);
  if (pending_beat >= 0.0) { R.has_pending = true; R.pending_beat = pending_beat; }
  else { R.pattern_running = true; if (!bounce) R.seq.start(); }
  gh::RackPattern* pats[1] = {&R};
  uint32_t n = 0, base = 0;
  for (uint32_t k = 0; k < n_calls; k++) {
    std::vector<gh::RackHit> hits[1];
    gh::resolve_rack_patterns(T, pats, 1, calls[k], bounce != 0, true, hits);
    if (bounce) R.seq.stop();
    for (const auto& h : hits[0]) { if (n < capacity) { if (out_frames) out_frames[n] = base + h.frame; if (out_pads) out_pads[n] = h.slot; if (out_velocity) out_velocity[n] = h.velocity; } n++; }
    base += calls[k];
  }
  if (out_transport_beat) *out_transport_beat = T.now();
  return n;
}

// ---- meters and MIDI export (ffi.rs:2572-2584, 6573-6580, 2145-2167) ----
void gooey_engine_get_channel_peaks(GooeyEngine* e, float* out_peaks, uint32_t count) {
  if (!e || !out_peaks) return;
  for (uint32_t i = 0; i < count && i < 5; i++) { out_peaks[i] = e->peaks[i]; e->peaks[i] = 0.0f; }
}
float gooey_engine_mixer_get_track_peak(GooeyEngine* e, uint32_t track) {
  if (!e || track >= e->cfg.n_tracks) return 0.0f;
  const float p = e->peaks[5 + track]; e->peaks[5 + track] = 0.0f; return p;
}
uint32_t gooey_engine_drain_midi_events(GooeyEngine* e, GooeyMidiEvent* out_events, uint32_t max_events) {
  if (!e || !out_events || max_events == 0) return 0;
  const size_t n = std::min<size_t>(e->midi_events.size(), max_events);
  for (size_t i = 0; i < n; i++) { out_events[i].instrument_index = e->midi_events[i].instrument_index; out_events[i].velocity = e->midi_events[i].velocity; out_events[i].sample_offset = e->midi_events[i].sample_offset; }
  e->midi_events.erase(e->midi_events.begin(), e->midi_events.begin() + n);
  return (uint32_t)n;
}

// ---- render / bounce ----
// Where the result of one device pass goes.  Exactly one of: dev (stays in HBM), host (pitched block of f32 rows), pcm (pitched
// block of 16-bit PCM rows, quantised on the device), rows (one host pointer per engine: the per-engine buffers of batch bounce).
struct RenderDst {
  float* dev = nullptr; size_t dev_stride = 0;
  float* host = nullptr; size_t host_pitch = 0;
  int16_t* pcm = nullptr; size_t pcm_pitch = 0;
  float* const* rows = nullptr;
};
static std::mutex g_ms_mutex;
static int batch_render_impl(GooeyEngine* const* engines, uint32_t n, uint32_t frames, int mode, bool bounce, const RenderDst& D, bool accumulate_ms = false) {
  std::vector<GooeyEngine*> E(engines, engines + n);
  try {
    gh::EngineBank& B = *E[0]->bank;
    gh::use_device(B.device);
    // The bank's output / voice buffers, streams and events are shared by every engine of (device, sample rate): the lock
    // is held from the allocation to the end of the drain, so concurrent renders of different engines serialise here.
    std::lock_guard<std::recursive_mutex> lk(B.mu);
    float* dst = D.dev;
    size_t stride = D.dev_stride;
    const size_t row = mode == gh::OUT_MONO ? (size_t)frames : (size_t)2 * frames;
    const size_t per_frame = mode == gh::OUT_MONO ? 1 : 2;
    if (!dst) {
      stride = (row + 3) & ~(size_t)3;
      B.d_out.alloc((size_t)n * stride);
      dst = B.d_out.p;
    }
    if (D.pcm) B.d_pcm.alloc((size_t)n * stride);
    // Pitched host destinations are drained piece by piece on the copy stream while later pieces render; the PCM path
    // quantises each finished piece on the device first and ships half the bytes.
    gh::PieceHook hook = [&](uint32_t f0, uint32_t nf, cudaEvent_t mixed) {
      GH_CUDA(cudaStreamWaitEvent(B.copy_stream, mixed, 0));
      const size_t c0 = per_frame * f0, nc = per_frame * nf;
      if (D.pcm) {
        gd::quantize_pcm16_kernel<<<dim3((unsigned)((nc + 1023) / 1024), n), 256, 0, B.copy_stream>>>(dst, (long long)stride, B.d_pcm.p, (long long)stride, (int)c0, (int)nc);
        gh::g_launches.fetch_add(1, std::memory_order_relaxed);
        GH_CUDA(cudaGetLastError());
        GH_CUDA(cudaMemcpy2DAsync(D.pcm + c0, D.pcm_pitch * 2, B.d_pcm.p + c0, stride * 2, nc * 2, n, cudaMemcpyDeviceToHost, B.copy_stream));
      } else {
        GH_CUDA(cudaMemcpy2DAsync(D.host + c0, D.host_pitch * 4, dst + c0, stride * 4, nc * 4, n, cudaMemcpyDeviceToHost, B.copy_stream));
      }
    };
    // ... when the destination is pinned.  An asynchronous copy into pageable memory is staged by the driver and blocks the
    // calling thread, which would stall the enqueueing of the next pieces: pageable destinations get one copy at the end.
    bool pinned = false;
    if (D.host || D.pcm) {
      cudaPointerAttributes at;
      if (cudaPointerGetAttributes(&at, D.host ? (const void*)D.host : (const void*)D.pcm) == cudaSuccess) pinned = at.type == cudaMemoryTypeHost;
      else cudaGetLastError();
    }
    const bool piecewise = pinned;
    gh::engines_render(E, frames, mode, bounce, dst, stride, piecewise ? &hook : nullptr);
    if ((D.host || D.pcm) && !piecewise) { GH_CUDA(cudaEventRecord(B.ev_piece, B.stream)); hook(0, frames, B.ev_piece); }
    if (D.rows) for (uint32_t i = 0; i < n; i++) GH_CUDA(cudaMemcpyAsync(D.rows[i], dst + (size_t)i * stride, row * 4, cudaMemcpyDeviceToHost, B.stream));
    if (D.host || D.pcm) GH_CUDA(cudaStreamSynchronize(B.copy_stream));
    GH_CUDA(cudaStreamSynchronize(B.stream));
    float ms = 0.0f;
    GH_CUDA(cudaEventElapsedTime(&ms, B.ev0, B.ev1));
    {
      std::lock_guard<std::mutex> g(g_ms_mutex);
      gh::g_last_kernel_ms = accumulate_ms ? std::max(gh::g_last_kernel_ms, ms) : ms;
    }
    B.collect_stats();
    return GOOEY_E_OK;
  } catch (const gh::BadBatch& ex) {
    gh::set_error(ex.what());
    return GOOEY_E_INVALID;
  } catch (const std::exception& ex) {
    gh::set_error(ex.what());
    for (auto* e : E) gh::engine_fail(e, ex.what());
    return GOOEY_E_CUDA;
  }
}
// A batch whose engines live on several devices (or sample rates): one group per bank, every group rendered by its own host
// thread (its own device, streams and pinned drain), no data-path collective (SURVEY.md section 8e).  Host destinations are
// sliced per group; a group whose engines are not a contiguous index range of the batch falls back to per-engine row copies.
static int batch_render_multi(GooeyEngine* const* engines, uint32_t n, uint32_t frames, int mode, bool bounce, const RenderDst& D) {
  std::map<gh::EngineBank*, std::vector<uint32_t>> groups;
  for (uint32_t i = 0; i < n; i++) groups[engines[i]->bank].push_back(i);
  if (groups.size() == 1) return batch_render_impl(engines, n, frames, mode, bounce, D);
  if (D.dev) { gh::set_error("engines of a device-resident batch must share device and sample rate"); return GOOEY_E_INVALID; }
  { std::lock_guard<std::mutex> g(g_ms_mutex); gh::g_last_kernel_ms = 0.0f; }
  const size_t row = mode == gh::OUT_MONO ? (size_t)frames : (size_t)2 * frames;
  std::vector<int> rcs(groups.size(), GOOEY_E_OK);
  std::vector<std::string> errs(groups.size());
  std::vector<std::thread> threads;
  size_t gi = 0;
  for (auto& g : groups) {
    const std::vector<uint32_t>& idx = g.second;
    threads.emplace_back([&, gi, idx]() {
      std::vector<GooeyEngine*> E;
      for (uint32_t i : idx) E.push_back(engines[i]);
      bool contiguous = true;
      for (size_t k = 1; k < idx.size(); k++) contiguous = contiguous && idx[k] == idx[k - 1] + 1;
      RenderDst G;
      std::vector<float*> rows;
      std::vector<int16_t> pcm_tmp;
      if (D.rows) { for (uint32_t i : idx) rows.push_back(D.rows[i]); G.rows = rows.data(); }
      else if (D.host && contiguous) { G.host = D.host + (size_t)idx[0] * D.host_pitch; G.host_pitch = D.host_pitch; }
      else if (D.pcm && contiguous) { G.pcm = D.pcm + (size_t)idx[0] * D.pcm_pitch; G.pcm_pitch = D.pcm_pitch; }
      else if (D.host) { for (uint32_t i : idx) rows.push_back(D.host + (size_t)i * D.host_pitch); G.rows = rows.data(); }
      else { pcm_tmp.resize(idx.size() * row); G.pcm = pcm_tmp.data(); G.pcm_pitch = row; }
      rcs[gi] = batch_render_impl(E.data(), (uint32_t)E.size(), frames, mode, bounce, G, true);
      if (rcs[gi] != GOOEY_E_OK) errs[gi] = gh::last_error();          // the error string is thread-local
      if (D.pcm && !contiguous && rcs[gi] == GOOEY_E_OK)
        for (size_t k = 0; k < idx.size(); k++) memcpy(D.pcm + (size_t)idx[k] * D.pcm_pitch, pcm_tmp.data() + k * row, row * 2);
    });
    gi++;
  }
  for (auto& t : threads) t.join();
  for (size_t k = 0; k < rcs.size(); k++) if (rcs[k] != GOOEY_E_OK) { gh::set_error(errs[k]); return rcs[k]; }
  return GOOEY_E_OK;
}

void gooey_engine_render(GooeyEngine* e, float* buffer, uint32_t frames) {
  if (!e || !buffer) return;
  if (frames == 0) return;
  RenderDst D; D.host = buffer; D.host_pitch = (size_t)2 * frames;
  if (e->has_error || batch_render_impl(&e, 1, frames, gh::OUT_STEREO, false, D) != GOOEY_E_OK)
    memset(buffer, 0, (size_t)frames * 2 * sizeof(float));
}
int gooey_batch_render(GooeyEngine* const* engines, uint32_t n, uint32_t frames, float* out_host) {
  if (!engines || !out_host) { gh::set_error("null argument"); return GOOEY_E_INVALID; }
  if (n == 0 || frames == 0) return GOOEY_E_OK;
  for (uint32_t i = 0; i < n; i++) if (!engines[i]) { gh::set_error("null engine in batch"); return GOOEY_E_INVALID; }
  RenderDst D; D.host = out_host; D.host_pitch = (size_t)2 * frames;
  return batch_render_multi(engines, n, frames, gh::OUT_STEREO, false, D);
}
float* gooey_engine_bounce_to_buffer(GooeyEngine* e, uint32_t bars, uint32_t* out_length) {
  if (!e || !out_length) return nullptr;
  float* buf = nullptr;
  if (gooey_batch_bounce(&e, 1, bars, &buf, out_length) != GOOEY_E_OK) return nullptr;
  return buf;
}
void gooey_engine_free_buffer(float* buffer, uint32_t) { free(buffer); }

int gooey_batch_bounce(GooeyEngine* const* engines, uint32_t n, uint32_t bars, float** out_buffers, uint32_t* out_lengths) {
  if (!engines || !out_buffers || !out_lengths) { gh::set_error("null argument"); return GOOEY_E_INVALID; }
  for (uint32_t i = 0; i < n; i++) { if (!engines[i]) { gh::set_error("null engine in batch"); return GOOEY_E_INVALID; } out_buffers[i] = nullptr; out_lengths[i] = 0; }
  // engines whose tempo gives a different length are bounced as separate groups
  std::map<uint32_t, std::vector<uint32_t>> groups;
  for (uint32_t i = 0; i < n; i++) groups[gh::bounce_frames(engines[i], bars)].push_back(i);
  for (auto& g : groups) {
    const uint32_t frames = g.first;
    std::vector<GooeyEngine*> E;
    for (uint32_t i : g.second) E.push_back(engines[i]);
    const size_t cnt = E.size();
    // each engine's result goes straight from the device into the buffer the caller will own (no staging copy)
    std::vector<float*> bufs(cnt, nullptr);
    for (size_t j = 0; j < cnt; j++) {
      bufs[j] = (float*)malloc(std::max<size_t>((size_t)frames, 1) * sizeof(float));
      if (!bufs[j]) {
        for (float* q : bufs) free(q);
        for (uint32_t i = 0; i < n; i++) { free(out_buffers[i]); out_buffers[i] = nullptr; out_lengths[i] = 0; }
        gh::set_error("out of host memory"); return GOOEY_E_INVALID;
      }
    }
    if (frames > 0) {
      RenderDst D; D.rows = bufs.data();
      int rc = batch_render_multi(E.data(), (uint32_t)cnt, frames, gh::OUT_MONO, true, D);
      if (rc != GOOEY_E_OK) {
        for (float* q : bufs) free(q);
        for (uint32_t i = 0; i < n; i++) { free(out_buffers[i]); out_buffers[i] = nullptr; out_lengths[i] = 0; }   // earlier groups
        return rc;
      }
    }
    for (size_t j = 0; j < cnt; j++) { out_buffers[g.second[j]] = bufs[j]; out_lengths[g.second[j]] = frames; }
  }
  return GOOEY_E_OK;
}
int gooey_batch_bounce_device(GooeyEngine* const* engines, uint32_t n, uint32_t bars, float* out_dev, size_t stride, uint32_t* out_frames) {
  if (!engines || !out_dev || n == 0) { gh::set_error("bad arguments"); return GOOEY_E_INVALID; }
  for (uint32_t i = 0; i < n; i++) if (!engines[i]) { gh::set_error("null engine in batch"); return GOOEY_E_INVALID; }
  const uint32_t frames = gh::bounce_frames(engines[0], bars);
  for (uint32_t i = 1; i < n; i++) if (gh::bounce_frames(engines[i], bars) != frames) { gh::set_error("engines of a device-resident batch must have equal length"); return GOOEY_E_INVALID; }
  if (stride < frames) { gh::set_error("stride < frames"); return GOOEY_E_INVALID; }
  if (out_frames) *out_frames = frames;
  if (frames == 0) return GOOEY_E_OK;
  RenderDst D; D.dev = out_dev; D.dev_stride = stride;
  return batch_render_multi(engines, n, frames, gh::OUT_MONO, true, D);
}
// Mono bounce of n engines of equal length into one pitched host block (f32) / 16-bit PCM block: the drain of finished pieces
// overlaps the rendering of later ones; engines may live on several devices (one host thread per device).
static int bounce_block_checks(GooeyEngine* const* engines, uint32_t n, uint32_t bars, const void* out, size_t pitch, uint32_t* out_frames, uint32_t& frames) {
  if (!engines || !out || n == 0) { gh::set_error("bad arguments"); return GOOEY_E_INVALID; }
  for (uint32_t i = 0; i < n; i++) if (!engines[i]) { gh::set_error("null engine in batch"); return GOOEY_E_INVALID; }
  frames = gh::bounce_frames(engines[0], bars);
  for (uint32_t i = 1; i < n; i++) if (gh::bounce_frames(engines[i], bars) != frames) { gh::set_error("engines of a block bounce must have equal length"); return GOOEY_E_INVALID; }
  if (pitch < frames) { gh::set_error("pitch < frames"); return GOOEY_E_INVALID; }
  if (out_frames) *out_frames = frames;
  return GOOEY_E_OK;
}
int gooey_batch_bounce_host(GooeyEngine* const* engines, uint32_t n, uint32_t bars, float* out_host, size_t pitch, uint32_t* out_frames) {
  uint32_t frames = 0;
  const int rc = bounce_block_checks(engines, n, bars, out_host, pitch, out_frames, frames);
  if (rc != GOOEY_E_OK || frames == 0) return rc;
  RenderDst D; D.host = out_host; D.host_pitch = pitch;
  return batch_render_multi(engines, n, frames, gh::OUT_MONO, true, D);
}
int gooey_batch_bounce_pcm16(GooeyEngine* const* engines, uint32_t n, uint32_t bars, int16_t* out_host, size_t pitch, uint32_t* out_frames) {
  uint32_t frames = 0;
  const int rc = bounce_block_checks(engines, n, bars, out_host, pitch, out_frames, frames);
  if (rc != GOOEY_E_OK || frames == 0) return rc;
  RenderDst D; D.pcm = out_host; D.pcm_pitch = pitch;
  return batch_render_multi(engines, n, frames, gh::OUT_MONO, true, D);
}

}  // extern "C"
