// patch.h — host-side translation of the reference's configuration surface into voice states and events:
// GooeyVoicePatch -> initial State (the `<Voice>::with_config` constructors), FFI parameter ids -> events.
// Plain C++ (no CUDA): shared by the product host code and by the host-emulation test harness (tests/emu).
#pragma once
#include <cstring>
#include "voices2.cuh"
#include "../../include/gooey_batch.h"

namespace gh {

// FFI parameter id -> smoother index (ffi.rs:168-250 with ids ffi.rs:1737-1836)
static const int kKickFfi[8] = {gd::K_FREQ, gd::K_PUNCH, gd::K_SUB, gd::K_CLICK, gd::K_OSC_DECAY, gd::K_PITCH_ENV_AMT, gd::K_VOLUME, gd::K_TUNING};
static const int kSnareFfi[20] = {gd::S_FREQ, gd::S_DECAY, gd::S_BRIGHTNESS, gd::S_VOLUME, gd::S_TONAL, gd::S_NOISE, gd::S_PITCH_DROP,
                                  gd::S_TONAL_DECAY, gd::S_NOISE_DECAY, gd::S_NOISE_TAIL_DECAY, gd::S_FILTER_CUTOFF, gd::S_FILTER_RES, -1,
                                  gd::S_XFADE, gd::S_PHASE_MOD, gd::S_OVERDRIVE, gd::S_AMP_DECAY, gd::S_AMP_DECAY_CURVE,
                                  gd::S_TONAL_DECAY_CURVE, gd::S_TUNING};
static const int kHatFfi[6] = {gd::H_PITCH, gd::H_DECAY, gd::H_ATTACK, gd::H_TONE, gd::H_VOLUME, gd::H_TUNING};

static inline float clamp01(float v) { return v < 0.0f ? 0.0f : (v > 1.0f ? 1.0f : v); }

// Translate `ChannelInstrument::set_param(param, value)` into voice events.  Returns false for unknown ids
// (the reference ignores them silently).
template <class AddFn> static bool ffi_param_to_events(uint32_t instrument, uint32_t param, float value, AddFn add) {
  switch (instrument) {
    case GOOEY_INSTRUMENT_KICK:
      if (param >= 8) return false;
      add(gd::EV_SET_TARGET, kKickFfi[param], clamp01(value));
      return true;
    case GOOEY_INSTRUMENT_SNARE:
      if (param >= 20) return false;
      if (param == 12) {  // `value as u8` (saturating) then .min(3)
        int t = !(value == value) ? 0 : (value <= 0.0f ? 0 : (value >= 255.0f ? 255 : (int)value));
        add(gd::EV_SET_AUX, gd::AUX_SNARE_FILTER_TYPE, (float)(t > 3 ? 3 : t));
      } else add(gd::EV_SET_TARGET, kSnareFfi[param], clamp01(value));
      return true;
    case GOOEY_INSTRUMENT_HIHAT:
      if (param >= 6) return false;
      add(gd::EV_SET_TARGET, kHatFfi[param], clamp01(value));
      return true;
    case GOOEY_INSTRUMENT_TOM:
      if (param >= 9) return false;
      add(gd::EV_SET_TARGET, param, param == 8 ? clamp01(value) : clamp01(value) * 100.0f);
      return true;
    case GOOEY_INSTRUMENT_BASS:
      if (param >= 16) return false;
      add(gd::EV_SET_TARGET, param, clamp01(value));   // BASS_PARAM_* ids follow the smoother order (ffi.rs:1904-1934)
      return true;
    case GOOEY_B200_VOICE_POLY:                          // PolySynth::set_param: ids 0-13 in PolyConfig order (poly_synth.rs)
      if (param >= gd::P_NP) return false;
      add(gd::EV_SET_TARGET, param, clamp01(value));
      return true;
    case GOOEY_B200_VOICE_GRANULATOR:                    // gooey_engine_granulator_set_param: ids 0-11 in GranulatorConfig order
      if (param >= gd::G_NP) return false;
      add(gd::EV_SET_TARGET, param, clamp01(value));
      return true;
    default: return false;
  }
}

static void snare_cfg_from_patch(const float* p, float* cfg, uint32_t& filter_type) {
  // new_full order -> S_* order (snare.rs:135-180 / SnareParams::from_config :420-545)
  // p: 0 freq,1 tonal,2 noise,3 crack,4 decay,5 pitch_drop,6 volume,7 tonal_decay,8 tonal_decay_curve,9 noise_decay,
  //    10 noise_tail_decay,11 filter_cutoff,12 filter_res,13 filter_type,14 xfade,15 phase_mod,16 overdrive,17 amp_decay,18 amp_decay_curve
  cfg[gd::S_FREQ] = p[0]; cfg[gd::S_TONAL] = p[1]; cfg[gd::S_NOISE] = p[2]; cfg[gd::S_BRIGHTNESS] = p[3]; cfg[gd::S_DECAY] = p[4];
  cfg[gd::S_PITCH_DROP] = p[5]; cfg[gd::S_VOLUME] = p[6]; cfg[gd::S_TONAL_DECAY] = p[7]; cfg[gd::S_TONAL_DECAY_CURVE] = p[8];
  cfg[gd::S_NOISE_DECAY] = p[9]; cfg[gd::S_NOISE_TAIL_DECAY] = p[10]; cfg[gd::S_FILTER_CUTOFF] = p[11]; cfg[gd::S_FILTER_RES] = p[12];
  float ft = p[13];
  int t = !(ft == ft) ? 0 : (ft <= 0.0f ? 0 : (ft >= 255.0f ? 255 : (int)ft));
  filter_type = (uint32_t)(t > 3 ? 3 : t);
  cfg[gd::S_XFADE] = p[14]; cfg[gd::S_PHASE_MOD] = p[15]; cfg[gd::S_OVERDRIVE] = p[16]; cfg[gd::S_AMP_DECAY] = p[17]; cfg[gd::S_AMP_DECAY_CURVE] = p[18];
}


inline void init_from_patch(gd::KickState& s, const GooeyVoicePatch& p, float sr) {
  memset(&s, 0, sizeof s);
  gd::kick_init(s, p.params, sr);
  if (p.aux & 0x100) s.c.cur[gd::K_TUNING] = s.c.tgt[gd::K_TUNING] = clamp01(p.params[23]);
}
inline void init_from_patch(gd::SnareState& s, const GooeyVoicePatch& p, float sr) {
  memset(&s, 0, sizeof s);
  float cfg[18]; uint32_t ft;
  snare_cfg_from_patch(p.params, cfg, ft);
  gd::snare_init(s, cfg, ft, sr);
  if (p.aux & 0x100) s.c.cur[gd::S_TUNING] = s.c.tgt[gd::S_TUNING] = clamp01(p.params[23]);
}
inline void init_from_patch(gd::HatState& s, const GooeyVoicePatch& p, float sr) {
  memset(&s, 0, sizeof s);
  gd::hat_init(s, p.params, p.aux & 1, (p.aux & 2) ? 0 : 1, sr);
  if (p.aux & 0x100) s.c.cur[gd::H_TUNING] = s.c.tgt[gd::H_TUNING] = clamp01(p.params[23]);
}
inline void init_from_patch(gd::TomState& s, const GooeyVoicePatch& p, float sr) {
  memset(&s, 0, sizeof s);
  gd::tom_init(s, (p.aux & 1) ? p.params : nullptr, sr);
  if (p.aux & 0x100) s.c.p[gd::T_TUNING] = clamp01(p.params[23]);
}
inline void init_from_patch(gd::BassState& s, const GooeyVoicePatch& p, float sr) {
  memset(&s, 0, sizeof s);
  gd::bass_init(s, p.params, sr);
  if (p.aux & 0x100) s.cur[gd::B_TUNING] = s.tgt[gd::B_TUNING] = clamp01(p.params[23]);
}
inline void init_from_patch(gd::PolyState& s, const GooeyVoicePatch& p, float sr) {   // params = PolyConfig (14 values)
  memset(&s, 0, sizeof s);
  gd::poly_init(s, p.params, sr);
}
inline void init_from_patch(gd::GranState& s, const GooeyVoicePatch&, float sr) {
  memset(&s, 0, sizeof s);
  gd::gran_init(s, sr);
}

}  // namespace gh
