// mix.cuh — the per-engine mix stage: voice strips (gain x mute, equal-power pan), MixerGraph
// (scatter -> per-track strip + effect rack -> sum), master gain, global effect chain
// (tilt / delay / spring reverb / plate reverb in the engine's effect order), optional soft limiter,
// and the stereo or mono-downmix write-out.  One engine per thread.
//
// Delay-line memory lives in "ring arenas": one per effect slot, laid out [ring word][engine slot]
// so that engines running in lock-step (same write index) touch adjacent addresses (coalesced).
// Reference: src/ffi.rs:1264-1377, src/frame.rs:31-53, src/mixer/graph.rs:47-58,344-399,
// src/effects/{tilt_filter,delay,reverb,plate_reverb,limiter}.rs.
#pragma once
#include "kernels.cuh"

namespace gd {

constexpr int MAX_TRACKS = 8;
constexpr int MAX_FX = 12;       // slots 0..3 = global tilt/delay/spring/plate, 4..11 = track-rack effects and the other global effects (on first use)
constexpr int N_VOICE_CH = 5;
constexpr int N_PEAKS = 5 + 8;   // voice strips + MAX_TRACKS
enum { FXK_NONE = 0xff, FXK_LOWPASS = 0, FXK_DELAY = 1, FXK_SATURATION = 2, FXK_COMPRESSOR = 3, FXK_TILT = 4, FXK_LIMITER = 5, FXK_SPRING = 6,
       FXK_WAVESHAPER = 7, FXK_FBWS = 8, FXK_PLATE = 9 };  // = FFI effect ids (ffi.rs:1548-1575)
enum { FXS_TILT = 0, FXS_DELAY = 1, FXS_SPRING = 2, FXS_PLATE = 3, FXS_RACK0 = 4 };
constexpr uint32_t OS_WORDS = 64;   // half-band history of one Oversampler (4 stages x 8 sections x {x, y}), kept in the slot's ring arena

struct Sm { float c, t; };
G_HD void sm_set(Sm& s, float v, float lo, float hi) { float c = clampf(v, lo, hi); if (fabsf(s.t - c) > 1e-8f) s.t = c; }
G_HD float sm_tick(Sm& s, float coeff) { smooth_tick(s.c, s.t, coeff); return s.c; }

struct TiltDyn { Sm cutoff[2], res[2]; Tpt svf[2]; float cutoff_target, res_target; float memo_t[2], memo_pow[2]; };   // memo: powf of the settled knob
struct DelayCh { uint32_t write_index; float z1, z2; uint32_t prev_timing; Sm time, fb, mix, cutoff; };
struct DelayDyn { DelayCh ch[2]; uint32_t timing_target; float bpm_target, fb_target, mix_target, cutoff_target; uint32_t pingpong; float memo_cut[2], memo_g[2]; };
struct SpringCh { uint32_t idx[6]; float fb, damp; Sm decay, mix, damping; };
struct SpringDyn { SpringCh ch[2]; float decay_target, mix_target, damping_target; float memo_decay[2], memo_fb[2]; };
struct PlateDyn {
  uint32_t idx[13];   // 0 predelay, 1..4 input APs, 5 mod_ap_a, 6 delay1_a, 7 ap2_a, 8 delay2_a, 9 mod_ap_b, 10 delay1_b, 11 ap2_b, 12 delay2_b
  float bandwidth, damp_a, damp_b, fb_a, fb_b, lfo_pa, lfo_pb;
  Sm decay, mix, damping, predelay, width, size;
  float t_decay, t_mix, t_damping, t_predelay, t_width, t_size;
  float memo_sz, memo_size;
};
// effects/lowpass_filter.rs, saturation.rs, compressor.rs; waveshaper.rs / feedback_waveshaper.rs as effect slots.  Index 0 = left / mono,
// 1 = right.  The global waveshapers are ONE instance fed L then R (ffi.rs:1344-1355): `shared` = 1 and only index 0 is used.
struct LpDyn { Sm cutoff[2], res[2]; float stage1[2], stage2[2]; float cutoff_target, res_target; float memo_c[2], memo_g[2]; };
struct SatDyn { Sm drive[2], warmth[2], mix[2]; float dc_x1[2], dc_y1[2]; float t_drive, t_warmth, t_mix; };
struct CompDyn { Sm th[2], ratio[2], att[2], rel[2], mix[2]; float env[2], gain[2], dc_x1[2], dc_y1[2]; float t_th, t_ratio, t_att, t_rel, t_mix; };
struct WsDyn { float drive[2], mix[2]; uint32_t shared; };
struct FbSmall { float drive, mix, feedback, cutoff, filter_coeff, env_att, env_rel, last_out, filter_state, dc_x1, dc_y1, env, memo_drive, memo_fb, memo_makeup; };
struct FbwsDyn { FbSmall s[2]; uint32_t shared; };
union FxDyn { TiltDyn tilt; DelayDyn delay; SpringDyn spring; PlateDyn plate; LpDyn lp; SatDyn sat; CompDyn comp; WsDyn ws; FbwsDyn fbws; uint32_t w[40]; };
static_assert(sizeof(FxDyn) == 160, "FxDyn must stay 40 words");

struct MixState {
  Sm ch_gain[N_VOICE_CH], ch_mute[N_VOICE_CH], ch_pan[N_VOICE_CH];
  Sm tr_gain[MAX_TRACKS], tr_pan[MAX_TRACKS], tr_mute[MAX_TRACKS];
  Sm master;
  FxDyn fx[MAX_FX];
};
// MixParam indices for MX_SET
enum { MP_CH_GAIN = 0, MP_CH_MUTE = 5, MP_CH_PAN = 10, MP_TR_GAIN = 15, MP_TR_PAN = 23, MP_TR_MUTE = 31, MP_MASTER = 39 };

// Host-authoritative structure of one engine's mixer (AoS; re-uploaded when edited).
struct MixCfg {
  uint32_t n_tracks;
  int32_t route[9];                 // source -> track (-1 none): drumkit, bass, poly, granulator, loop mixer, sampler racks 0-3 (graph.rs:31-42)
  uint32_t order[9];                // effect_order (ffi.rs:1583-1593)
  uint8_t gslot[12];                // global effect id -> slot (0xff = never touched: the effect is still in its constructor state and disabled)
  uint32_t comp_sidechain;          // compressor_sidechain (ffi.rs:3252-3265): instrument 0-4 or 0xFFFFFFFF
  uint32_t fx_kind[MAX_FX];         // FXK_* (FXK_NONE = slot unused)
  uint32_t fx_enabled[MAX_FX];      // global slots: *_enabled flags; rack slots: 1
  uint32_t fx_rack;                 // bit s: slot s belongs to a track rack (not touched by reset_effect_states)
  uint32_t rack_n[MAX_TRACKS];
  uint8_t rack_slot[MAX_TRACKS][4];
  uint32_t limiter_on;
  float lim_th, lim_inv;
  uint32_t src_poly, src_gran;      // 1 when the poly / granulator voice buffers carry this engine's output
  // sample-playback sources (loops.cuh), rewritten by every render call: bit 0 = the loop mixer, bit 1 + k = sampler rack k has a
  // stereo row pair in the launch's ext planes; ext_row[s] = that pair's index (left row 2 * r, right row 2 * r + 1)
  uint32_t src_ext;
  uint32_t ext_row[5];
};

// Geometry of the delay lines at the launch's sample rate (host-computed, reference formulas).
struct FxGeom {
  uint32_t delay_len;                 // (sr * 5) as usize + 1            (delay.rs:189)
  uint32_t spring_off[12], spring_len[12];   // L0..5, R0..5             (reverb.rs:84-96)
  uint32_t plate_off[13], plate_cap[13];     // DelayLine capacities       (plate_reverb.rs:236-262)
  float plate_in_delay[4], plate_len[8], plate_excursion, plate_sr_scale, plate_lfo_ia, plate_lfo_ib;
  uint32_t ring_words[4];             // words per engine for FXK_TILT(0)/DELAY/SPRING/PLATE arenas
};

struct MixLaunch {
  uint32_t* state; int n, state_cap;  // MixState pool (SoA words, row pitch state_cap)
  const uint32_t* slots;              // launch index -> engine slot in the pool / cfg array / ring arenas
  int n_lpad;                         // launch count padded to 32: voice row of channel ch, engine i = ch * n_lpad + i
  const MixCfg* cfg;
  const VoiceEvent* events; const uint32_t* ev_begin;
  const float* voice_buf;             // voice-major [row][voice_stride]; ch 0-4 = voice strips, 5 = poly, 6 = granulator
  long long voice_stride;
  uint32_t chan_mask;                 // bit ch set: some engine of the launch has a source on that channel
  float* ring[MAX_FX];                // per fx-slot arenas [word][ring_cap]
  long long ring_cap;
  int frames;
  float* out; long long out_stride; int out_mode;  // 0: mono downmix [engine][frame], 1: interleaved stereo [engine][2*frame]
  const uint32_t* out_rows;
  RateCtx rc; FxGeom geo;
  long long premix_stride;
  float center_l, center_r;           // cos/sin(0.5 * pi/2) for the center-panned poly / granulator (ffi.rs:1287-1288)
  // time-parallel path for engines whose mixer is memoryless over this launch (see mix_prepare_kernel)
  float* peaks;                       // [n][N_PEAKS] running maxima of the call (bit pattern of a non-negative float): 5 voice strips
                                      // (pre-pan |x|, ffi.rs:1281-1282), then MAX_TRACKS post-strip max(|l|, |r|) (graph.rs:395)
  uint8_t* fast;                      // [n] 1 = handled by mix_fast_kernel, the general kernel skips it; 2 = mix_fast_kernel writes the
                                      // engine's pre-chain stereo mix (strips -> graph -> master) and the general kernel runs only its global chain
  float* premix;                      // [2][n_lpad][premix_stride]: left plane, right plane
  const float* ext; long long ext_stride;   // sample-playback sources of this piece: [2 * pairs][ext_stride] (MixCfg::ext_row), or nullptr
  struct MixConst* consts;            // [n]
  unsigned long long* chain_units;    // engine-frames taken by chain_fast_kernel (chain.cuh) in this render call
};
// Everything mix_fast_kernel needs for one engine: the settled smoother values and the trig of the constant pans.
struct MixConst {
  float g[N_VOICE_CH], m[N_VOICE_CH], pc[N_VOICE_CH], ps[N_VOICE_CH];
  float tgain[MAX_TRACKS], tbl[MAX_TRACKS], tbr[MAX_TRACKS];
  float master, lim_th, lim_inv;
  uint32_t n_tracks, limiter_on, src_poly, src_gran;
  int32_t route[9];
  uint32_t src_ext, ext_row[5];
};

// ---------------------------------------------------------------- effect constructors (device + host) ----
G_HD void tilt_init(TiltDyn& d, float sr) {  // TiltFilterEffect::new
  for (int c = 0; c < 2; c++) { d.cutoff[c] = {0.5f, 0.5f}; d.res[c] = {0.0f, 0.0f}; tpt_init(d.svf[c], sr, 1000.0f, 0.5f); }
  d.cutoff_target = 0.5f; d.res_target = 0.0f;
  d.memo_t[0] = d.memo_t[1] = -1.0f; d.memo_pow[0] = d.memo_pow[1] = 0.0f;   // no valid input is negative
}
G_HD float delay_beats(uint32_t t) {
  switch (t) { case 0: return 4.0f; case 1: return 2.0f; case 2: return 1.0f; case 3: return 0.5f; case 4: return 0.25f;
    case 5: return 4.0f / 3.0f; case 6: return 2.0f / 3.0f; case 7: return 1.0f / 3.0f; case 8: return 1.0f / 6.0f; default: return 1.0f; }
}
G_HD float delay_seconds(uint32_t timing, float bpm) { return fminf((60.0f / bpm) * delay_beats(timing), 5.0f); }
G_HD void delay_init(DelayDyn& d, uint32_t timing, float bpm, float fb, float mix, float cutoff) {  // DelayEffect::new
  float time = delay_seconds(timing, bpm);
  float fbc = clampf(fb, 0.0f, 0.95f), mc = clampf(mix, 0.0f, 1.0f), cc = clampf(cutoff, 20.0f, 20000.0f);
  for (int c = 0; c < 2; c++) {
    DelayCh& s = d.ch[c];
    s.write_index = 0; s.z1 = s.z2 = 0.0f; s.prev_timing = timing;
    float tc = clampf(time, 0.0f, 5.0f);
    s.time = {tc, tc}; s.fb = {fbc, fbc}; s.mix = {mc, mc}; s.cutoff = {cc, cc};
  }
  d.timing_target = timing; d.bpm_target = bpm; d.fb_target = fbc; d.mix_target = mc; d.cutoff_target = cc; d.pingpong = 0;
  d.memo_cut[0] = d.memo_cut[1] = -1.0f; d.memo_g[0] = d.memo_g[1] = 0.0f;
}
G_HD void spring_init(SpringDyn& d, float decay, float mix, float damping) {  // SpringReverbEffect::new
  decay = clampf(decay, 0.0f, 1.0f); mix = clampf(mix, 0.0f, 1.0f); damping = clampf(damping, 0.0f, 1.0f);
  for (int c = 0; c < 2; c++) {
    SpringCh& s = d.ch[c];
    for (int i = 0; i < 6; i++) s.idx[i] = 0;
    s.fb = s.damp = 0.0f; s.decay = {decay, decay}; s.mix = {mix, mix}; s.damping = {damping, damping};
  }
  d.decay_target = decay; d.mix_target = mix; d.damping_target = damping;
  d.memo_decay[0] = d.memo_decay[1] = -1.0f; d.memo_fb[0] = d.memo_fb[1] = 0.0f;
}
G_HD void plate_init(PlateDyn& d, float decay, float mix, float damping) {  // PlateReverbEffect::new
  decay = clampf(decay, 0.0f, 1.0f); mix = clampf(mix, 0.0f, 1.0f); damping = clampf(damping, 0.0f, 1.0f);
  for (int i = 0; i < 13; i++) d.idx[i] = 0;
  d.bandwidth = d.damp_a = d.damp_b = d.fb_a = d.fb_b = d.lfo_pa = d.lfo_pb = 0.0f;
  d.decay = {decay, decay}; d.mix = {mix, mix}; d.damping = {damping, damping}; d.predelay = {0.0f, 0.0f}; d.width = {1.0f, 1.0f}; d.size = {0.5f, 0.5f};
  d.t_decay = decay; d.t_mix = mix; d.t_damping = damping; d.t_predelay = 0.0f; d.t_width = 1.0f; d.t_size = 0.5f;
  d.memo_sz = -1.0f; d.memo_size = 0.0f;
}
G_HD void lp_init(LpDyn& d, float cutoff, float res) {  // LowpassFilterEffect::new (lowpass_filter.rs:55-81)
  cutoff = clampf(cutoff, 20.0f, 20000.0f); res = clampf(res, 0.0f, 0.95f);
  for (int c = 0; c < 2; c++) { d.cutoff[c] = {cutoff, cutoff}; d.res[c] = {res, res}; d.stage1[c] = d.stage2[c] = 0.0f; d.memo_c[c] = -1.0f; d.memo_g[c] = 0.0f; }
  d.cutoff_target = cutoff; d.res_target = res;
}
G_HD void sat_init(SatDyn& d, float drive, float warmth, float mix) {  // TubeSaturation::new (saturation.rs:68-91)
  drive = clampf(drive, 0.0f, 1.0f); warmth = clampf(warmth, 0.0f, 1.0f); mix = clampf(mix, 0.0f, 1.0f);
  for (int c = 0; c < 2; c++) { d.drive[c] = {drive, drive}; d.warmth[c] = {warmth, warmth}; d.mix[c] = {mix, mix}; d.dc_x1[c] = d.dc_y1[c] = 0.0f; }
  d.t_drive = drive; d.t_warmth = warmth; d.t_mix = mix;
}
G_HD void comp_init(CompDyn& d, float th, float ratio, float att, float rel, float mix) {  // TubeCompressor::new (compressor.rs:55-96)
  th = clampf(th, -60.0f, 0.0f); ratio = clampf(ratio, 1.0f, 20.0f); att = clampf(att, 0.1f, 100.0f); rel = clampf(rel, 5.0f, 1000.0f); mix = clampf(mix, 0.0f, 1.0f);
  for (int c = 0; c < 2; c++) {
    d.th[c] = {th, th}; d.ratio[c] = {ratio, ratio}; d.att[c] = {att, att}; d.rel[c] = {rel, rel}; d.mix[c] = {mix, mix};
    d.env[c] = 0.0f; d.gain[c] = 1.0f; d.dc_x1[c] = d.dc_y1[c] = 0.0f;
  }
  d.t_th = th; d.t_ratio = ratio; d.t_att = att; d.t_rel = rel; d.t_mix = mix;
}
G_HD void fbsmall_init(FbSmall& w, float sr, float drive, float fb, float cutoff, float mix) {  // FeedbackWaveshaper::new; same arithmetic as fbws_init
  w.drive = clampf(drive, 1.0f, 100.0f); w.mix = clampf(mix, 0.0f, 1.0f); w.feedback = clampf(fb, 0.0f, 0.98f);
  w.cutoff = clampf(cutoff, 200.0f, 20000.0f);
  w.filter_coeff = fbws_filter_coeff(w.cutoff, sr);
  w.env_att = gm::g_expf(-1.0f / (1.0f / 1000.0f * sr));
  w.env_rel = gm::g_expf(-1.0f / (120.0f / 1000.0f * sr));
  w.last_out = w.filter_state = w.dc_x1 = w.dc_y1 = w.env = 0.0f;
  w.memo_drive = -1.0f; w.memo_fb = -1.0f; w.memo_makeup = 1.0f;
}
// effect_chain.rs:57-109 defaults for rack effects vs ffi.rs:852-884 defaults for the global instances
G_HD void fx_construct(FxDyn& f, uint32_t kind, bool rack, float sr, float bpm) {
  for (int i = 0; i < 40; i++) f.w[i] = 0;
  switch (kind) {
    case FXK_LOWPASS: lp_init(f.lp, 20000.0f, 0.0f); break;
    case FXK_SATURATION: sat_init(f.sat, 0.3f, 0.4f, 0.5f); break;
    case FXK_COMPRESSOR: comp_init(f.comp, -12.0f, 4.0f, 5.0f, 100.0f, 0.5f); break;
    case FXK_WAVESHAPER: for (int c = 0; c < 2; c++) { f.ws.drive[c] = 1.0f; f.ws.mix[c] = 0.0f; } f.ws.shared = rack ? 0u : 1u; break;
    case FXK_FBWS: for (int c = 0; c < 2; c++) fbsmall_init(f.fbws.s[c], sr, 1.0f, 0.0f, 2000.0f, 0.0f); f.fbws.shared = rack ? 0u : 1u; break;
    case FXK_TILT: tilt_init(f.tilt, sr); break;
    case FXK_DELAY: if (rack) delay_init(f.delay, 2, bpm, 0.3f, 0.3f, 8000.0f); else delay_init(f.delay, 2, bpm, 0.0f, 0.0f, 20000.0f); break;
    case FXK_SPRING: spring_init(f.spring, 0.5f, rack ? 0.3f : 0.0f, 0.5f); break;
    case FXK_PLATE: plate_init(f.plate, 0.5f, rack ? 0.3f : 0.0f, 0.5f); break;
    default: break;
  }
}
// `set_param` of each effect (ffi.rs:2988-3075 == effect_chain.rs:152-232): raw FFI value -> clamped atomic target
G_HD void fx_set_param(FxDyn& f, uint32_t kind, uint32_t p, float v, float sr) {
  switch (kind) {
    case FXK_LOWPASS: if (p == 0) f.lp.cutoff_target = clampf(v, 20.0f, 20000.0f); else if (p == 1) f.lp.res_target = clampf(v, 0.0f, 0.95f); break;
    case FXK_SATURATION: v = clampf(v, 0.0f, 1.0f); if (p == 0) f.sat.t_drive = v; else if (p == 1) f.sat.t_warmth = v; else if (p == 2) f.sat.t_mix = v; break;
    case FXK_COMPRESSOR:
      switch (p) { case 0: f.comp.t_th = clampf(v, -60.0f, 0.0f); break; case 1: f.comp.t_ratio = clampf(v, 1.0f, 20.0f); break; case 2: f.comp.t_att = clampf(v, 0.1f, 100.0f); break;
        case 3: f.comp.t_rel = clampf(v, 5.0f, 1000.0f); break; case 4: f.comp.t_mix = clampf(v, 0.0f, 1.0f); break; }
      break;
    case FXK_WAVESHAPER:   // Waveshaper::set_drive / set_mix act immediately (waveshaper.rs:29-46); rack: both channel instances
      for (int c = 0; c < 2; c++) { if (p == 0) f.ws.drive[c] = clampf(v, 1.0f, 10.0f); else if (p == 1) f.ws.mix[c] = clampf(v, 0.0f, 1.0f); }
      break;
    case FXK_FBWS:         // feedback_waveshaper.rs:171-200
      for (int c = 0; c < 2; c++) {
        FbSmall& w = f.fbws.s[c];
        if (p == 0) w.drive = clampf(v, 1.0f, 100.0f); else if (p == 1) w.feedback = clampf(v, 0.0f, 0.98f);
        else if (p == 2) { w.cutoff = clampf(v, 200.0f, 20000.0f); w.filter_coeff = fbws_filter_coeff(w.cutoff, sr); }
        else if (p == 3) w.mix = clampf(v, 0.0f, 1.0f);
      }
      break;
    case FXK_TILT: if (p == 0) f.tilt.cutoff_target = clampf(v, 0.0f, 1.0f); else if (p == 1) f.tilt.res_target = clampf(v, 0.0f, 1.0f); break;
    case FXK_DELAY:
      switch (p) {
        case 0: { uint64_t t = f32_to_u64_sat(v); if (t <= 8) f.delay.timing_target = (uint32_t)t; } break;
        case 1: f.delay.fb_target = clampf(v, 0.0f, 0.95f); break;
        case 2: f.delay.mix_target = clampf(v, 0.0f, 1.0f); break;
        case 3: f.delay.cutoff_target = clampf(v, 20.0f, 20000.0f); break;
        case 4: f.delay.pingpong = v >= 0.5f; break;
      }
      break;
    case FXK_SPRING: v = clampf(v, 0.0f, 1.0f); if (p == 0) f.spring.decay_target = v; else if (p == 1) f.spring.mix_target = v; else if (p == 2) f.spring.damping_target = v; break;
    case FXK_PLATE:
      v = clampf(v, 0.0f, 1.0f);
      switch (p) { case 0: f.plate.t_decay = v; break; case 1: f.plate.t_mix = v; break; case 2: f.plate.t_damping = v; break;
        case 3: f.plate.t_predelay = v; break; case 4: f.plate.t_width = v; break; case 5: f.plate.t_size = v; break; }
      break;
    default: break;
  }
}

#ifdef __CUDACC__
// ---------------------------------------------------------------- per-sample effect processing ----
// x mod n for 0 <= x < 2n (every ring index here): a compare and a subtract instead of the ~20-instruction integer division
// (ncu r1: the `% len` of the spring's six index increments alone was 10 % of the mix kernel's instructions).
__device__ __forceinline__ uint32_t wrap2(uint32_t x, uint32_t n) { return x >= n ? x - n : x; }
struct RingRef { float* base; long long cap; int es; __device__ __forceinline__ float& at(uint32_t j) const { return base[(long long)j * cap + es]; } };

__device__ __forceinline__ float tilt_one(TiltDyn& d, int c, float in, const RateCtx& rc) {  // tilt_filter.rs:87-139
  sm_set(d.cutoff[c], d.cutoff_target, 0.0f, 1.0f);
  sm_set(d.res[c], d.res_target, 0.0f, 1.0f);
  float knob = sm_tick(d.cutoff[c], rc.smooth30);
  float resonance = sm_tick(d.res[c], rc.smooth30);
  float mix, freq; bool lp;
  // the powf is a pure function of the knob: re-evaluated only when the smoothed knob moves (bit-identical)
  if (knob != d.memo_t[c]) { d.memo_t[c] = knob; d.memo_pow[c] = knob < 0.5f ? gm::g_powf(20000.0f / 80.0f, knob * 2.0f) : gm::g_powf(8000.0f / 20.0f, (knob - 0.5f) * 2.0f); }
  if (knob < 0.5f) { mix = 1.0f - (knob * 2.0f); freq = 80.0f * d.memo_pow[c]; lp = true; }
  else { mix = (knob - 0.5f) * 2.0f; freq = 20.0f * d.memo_pow[c]; lp = false; }
  if (mix < 0.001f) return in;
  float q = 0.5f + resonance * 8.0f;
  tpt_set(d.svf[c], rc.sr, freq, q);
  float lo, bd, hi;
  tpt_process(d.svf[c], in, lo, bd, hi);
  float wet = lp ? lo : hi;
  float out = in * (1.0f - mix) + wet * mix;
  if (!isfinite(out)) { d.svf[c].ic1 = d.svf[c].ic2 = 0.0f; return 0.0f; }
  if (fabsf(out) < 1e-15f) return 0.0f;
  return out;
}

struct DelayStep { float filtered, feedback, mix; };
// The ring reads of a frame have addresses that depend on state only, never on this frame's audio, so every effect
// first computes its addresses (`*_prep`), then issues ALL its loads back to back, and only then runs the dependent
// arithmetic: the L2 / HBM latency is paid once per effect and frame instead of once per tap (the reference order of
// the arithmetic is untouched; the taps read cells written >= 1 frame earlier, the writes of this frame come after).
struct DelayPrep { uint32_t r1, r2; float df, feedback, mix, cutoff; };
__device__ __forceinline__ DelayPrep delay_prep(DelayDyn& d, int c, const RingRef& r, uint32_t len, const RateCtx& rc) {  // delay.rs:321-360
  DelayCh& s = d.ch[c];
  const uint32_t base = c * len;
  uint32_t tc = d.timing_target;
  float time_target = delay_seconds(tc <= 8 ? tc : 2, d.bpm_target);
  if (tc != s.prev_timing) {
    s.prev_timing = tc;
    for (uint32_t j = 0; j < len; j++) r.at(base + j) = 0.0f;
    s.z1 = s.z2 = 0.0f;
    float tcl = clampf(time_target, 0.0f, 5.0f);
    s.time = {tcl, tcl};
  }
  sm_set(s.time, time_target, 0.0f, 5.0f); sm_set(s.fb, d.fb_target, 0.0f, 0.95f); sm_set(s.mix, d.mix_target, 0.0f, 1.0f); sm_set(s.cutoff, d.cutoff_target, 20.0f, 20000.0f);
  DelayPrep p;
  float time = sm_tick(s.time, rc.smooth50);
  p.feedback = sm_tick(s.fb, rc.smooth30); p.mix = sm_tick(s.mix, rc.smooth30); p.cutoff = sm_tick(s.cutoff, rc.smooth30);
  float ds = time * rc.sr;
  uint32_t di = (uint32_t)f32_to_u64_sat(ds);
  p.df = ds - (float)di;
  p.r1 = base + wrap2(s.write_index + len - di, len);          // di <= 5 s * sr = len - 1
  p.r2 = base + wrap2(s.write_index + len - di - 1, len);
  return p;
}
__device__ __forceinline__ DelayStep delay_filter(DelayDyn& d, int c, const DelayPrep& p, float s1, float s2, const RateCtx& rc) {  // :361-399
  DelayCh& s = d.ch[c];
  float delayed = s1 * (1.0f - p.df) + s2 * p.df;
  if (p.cutoff != d.memo_cut[c]) { d.memo_cut[c] = p.cutoff; d.memo_g[c] = 1.0f - gm::g_expf(-2.0f * PI_F * p.cutoff / rc.sr); }
  float g = d.memo_g[c];
  float rfb = 0.3f * (s.z1 - s.z2);
  s.z1 = s.z1 + g * (delayed + rfb - s.z1);
  s.z2 = s.z2 + g * (s.z1 - s.z2);
  float filtered = s.z2;
  if (fabsf(s.z1) < 1e-15f) s.z1 = 0.0f;
  if (fabsf(s.z2) < 1e-15f) s.z2 = 0.0f;
  return {filtered, p.feedback, p.mix};
}
__device__ __forceinline__ float delay_write(DelayDyn& d, int c, const RingRef& r, uint32_t len, float dry, float inject, const DelayStep& st, float tap) {  // :407-439
  DelayCh& s = d.ch[c];
  float w = inject + tap * st.feedback;
  w = (isfinite(w) && fabsf(w) > 1e-15f) ? w : 0.0f;
  r.at(c * len + s.write_index) = w;
  s.write_index = wrap2(s.write_index + 1, len);
  float out = dry * (1.0f - st.mix) + st.filtered * st.mix;
  return isfinite(out) ? out : dry;
}
__device__ __forceinline__ void delay_stereo(DelayDyn& d, const RingRef& r, uint32_t len, float& l, float& rr, const RateCtx& rc) {  // :460-491
  const float li = isfinite(l) ? l : 0.0f, ri = isfinite(rr) ? rr : 0.0f;
  const DelayPrep pa = delay_prep(d, 0, r, len, rc), pb = delay_prep(d, 1, r, len, rc);
  const float a1 = r.at(pa.r1), a2 = r.at(pa.r2), b1 = r.at(pb.r1), b2 = r.at(pb.r2);   // the two channels own disjoint halves
  const DelayStep a = delay_filter(d, 0, pa, a1, a2, rc), b = delay_filter(d, 1, pb, b1, b2, rc);
  if (!d.pingpong) {
    l = delay_write(d, 0, r, len, li, li, a, a.filtered);
    rr = delay_write(d, 1, r, len, ri, ri, b, b.filtered);
    return;
  }
  l = delay_write(d, 0, r, len, li, li, a, b.filtered);
  rr = delay_write(d, 1, r, len, ri, 0.0f, b, a.filtered);
}

__device__ __forceinline__ float spring_one(SpringDyn& d, int c, const RingRef& r, const FxGeom& g, float in, const RateCtx& rc, const float* dl) {  // reverb.rs:162-217
  const float G[6] = {0.70f, 0.68f, 0.65f, 0.62f, 0.60f, 0.58f};
  SpringCh& s = d.ch[c];
  in = isfinite(in) ? in : 0.0f;
  sm_set(s.decay, d.decay_target, 0.0f, 1.0f); sm_set(s.mix, d.mix_target, 0.0f, 1.0f); sm_set(s.damping, d.damping_target, 0.0f, 1.0f);
  float decay = sm_tick(s.decay, rc.smooth15), mix = sm_tick(s.mix, rc.smooth15), damping = sm_tick(s.damping, rc.smooth15);
  if (decay != d.memo_decay[c]) { d.memo_decay[c] = decay; d.memo_fb[c] = gm::g_powf(decay, 0.4f) * 0.95f; }
  float feedback = d.memo_fb[c];
  float d1 = damping, d2 = 1.0f - damping;
  float sig = in + s.fb;
#pragma unroll
  for (int i = 0; i < 6; i++) {
    const uint32_t off = g.spring_off[c * 6 + i], len = g.spring_len[c * 6 + i];
    const float delayed = dl[i];          // loaded by the caller for both channels before either chain starts
    float v = sig - G[i] * delayed;
    sig = G[i] * v + delayed;
    r.at(off + s.idx[i]) = v;
    s.idx[i] = wrap2(s.idx[i] + 1, len);
  }
  s.damp = sig * d2 + s.damp * d1;
  if (fabsf(s.damp) < 1e-15f) s.damp = 0.0f;
  s.fb = s.damp * feedback;
  if (fabsf(s.fb) < 1e-15f) s.fb = 0.0f;
  float res = in * (1.0f - mix) + sig * mix;
  return isfinite(res) ? res : in;
}

struct PlateLine {
  const RingRef& r; uint32_t off, cap; uint32_t& idx;
  __device__ __forceinline__ void write(float x) { r.at(off + idx) = x; idx = wrap2(idx + 1, cap); }
  __device__ __forceinline__ float read_frac(float o) const {
    o = clampf(o, 1.0f, (float)(cap - 2));
    uint32_t w = (uint32_t)o; float fr = o - (float)w;
    float a = r.at(off + wrap2(idx + cap - w, cap)), b = r.at(off + wrap2(idx + cap - w - 1, cap));      // 1 <= w <= cap - 2
    return a + fr * (b - a);
  }
  __device__ __forceinline__ float tap_frac(float o) const {
    o = clampf(o, 0.0f, (float)(cap - 2));
    uint32_t w = (uint32_t)o; float fr = o - (float)w;
    float a = r.at(off + wrap2(idx + cap - 1 - w, cap)), b = r.at(off + wrap2(idx + cap - 2 - w, cap));  // 0 <= w <= cap - 2
    return a + fr * (b - a);
  }
  __device__ __forceinline__ float allpass(float in, float g, float d) { float dl = read_frac(d); float v = in - g * dl; write(v); return g * v + dl; }
};
__device__ __forceinline__ void flush_dn(float& x) { if (fabsf(x) < 1e-15f) x = 0.0f; }
__device__ __forceinline__ void plate_tank(PlateDyn& d, const RingRef& r, const FxGeom& g, float in, float& wl, float& wr, float& mix, const RateCtx& rc) {  // plate_reverb.rs:406-534
  in = isfinite(in) ? in : 0.0f;
  sm_set(d.decay, d.t_decay, 0, 1); sm_set(d.mix, d.t_mix, 0, 1); sm_set(d.damping, d.t_damping, 0, 1);
  sm_set(d.predelay, d.t_predelay, 0, 1); sm_set(d.width, d.t_width, 0, 1); sm_set(d.size, d.t_size, 0, 1);
  float decay_knob = sm_tick(d.decay, rc.smooth15); mix = sm_tick(d.mix, rc.smooth15); float damping = sm_tick(d.damping, rc.smooth15);
  float predelay_knob = sm_tick(d.predelay, rc.smooth15); float width = sm_tick(d.width, rc.smooth15);
  float sz = sm_tick(d.size, rc.smooth15);
  if (sz != d.memo_sz) { d.memo_sz = sz; d.memo_size = sz <= 0.5f ? gm::g_powf(4.0f, 2.0f * sz - 1.0f) : gm::g_powf(2.0f, 2.0f * sz - 1.0f); }
  float size = d.memo_size;
  float decay_gain = decay_knob * 0.95f;
  float dd2 = clampf(decay_gain + 0.15f, 0.25f, 0.50f);
  float damp = damping * 0.95f;
#define PL(i) PlateLine{r, g.plate_off[i], g.plate_cap[i], d.idx[i]}
  PlateLine predelay = PL(0);
  predelay.write(in);
  float pds = predelay_knob * 200.0f * 0.001f * rc.sr;
  float delayed = predelay.tap_frac(pds);
  d.bandwidth += 0.9995f * (delayed - d.bandwidth);
  flush_dn(d.bandwidth);
  float sig = d.bandwidth;
  const float IAG[4] = {0.750f, 0.750f, 0.625f, 0.625f};
#pragma unroll
  for (int i = 0; i < 4; i++) { PlateLine ap = PL(1 + i); sig = ap.allpass(sig, IAG[i], g.plate_in_delay[i]); }
  d.lfo_pa = fract(d.lfo_pa + g.plate_lfo_ia); d.lfo_pb = fract(d.lfo_pb + g.plate_lfo_ib);
  const float TAU_F = 6.28318530717958647692f;
  float lfo_a = gm::g_sinf(TAU_F * d.lfo_pa), lfo_b = gm::g_sinf(TAU_F * d.lfo_pb);
  float in_a = sig + d.fb_b, in_b = sig + d.fb_a;
  PlateLine mod_a = PL(5), d1a_l = PL(6), ap2a = PL(7), d2a_l = PL(8), mod_b = PL(9), d1b_l = PL(10), ap2b = PL(11), d2b_l = PL(12);
  float a1 = mod_a.allpass(in_a, 0.70f, g.plate_len[0] * size + lfo_a * g.plate_excursion);
  float d1a = d1a_l.read_frac(g.plate_len[1] * size);
  d1a_l.write(a1);
  d.damp_a = d1a * (1.0f - damp) + d.damp_a * damp; flush_dn(d.damp_a);
  float a2 = ap2a.allpass(d.damp_a * decay_gain, dd2, g.plate_len[2] * size);
  float d2a = d2a_l.read_frac(g.plate_len[3] * size);
  d2a_l.write(a2);
  float b1 = mod_b.allpass(in_b, 0.70f, g.plate_len[4] * size + lfo_b * g.plate_excursion);
  float d1b = d1b_l.read_frac(g.plate_len[5] * size);
  d1b_l.write(b1);
  d.damp_b = d1b * (1.0f - damp) + d.damp_b * damp; flush_dn(d.damp_b);
  float b2 = ap2b.allpass(d.damp_b * decay_gain, dd2, g.plate_len[6] * size);
  float d2b = d2b_l.read_frac(g.plate_len[7] * size);
  d2b_l.write(b2);
  d.fb_a = d2a * decay_gain; flush_dn(d.fb_a);
  d.fb_b = d2b * decay_gain; flush_dn(d.fb_b);
  float ts = g.plate_sr_scale * size;
  float yl = 0.6f * (d1b_l.tap_frac(266.0f * ts) + d1b_l.tap_frac(2974.0f * ts) - ap2b.tap_frac(1913.0f * ts) + d2b_l.tap_frac(1996.0f * ts)
                     - d1a_l.tap_frac(1990.0f * ts) - ap2a.tap_frac(187.0f * ts) - d2a_l.tap_frac(1066.0f * ts));
  float yr = 0.6f * (d1a_l.tap_frac(353.0f * ts) + d1a_l.tap_frac(3627.0f * ts) - ap2a.tap_frac(1228.0f * ts) + d2a_l.tap_frac(2673.0f * ts)
                     - d1b_l.tap_frac(2111.0f * ts) - ap2b.tap_frac(335.0f * ts) - d2b_l.tap_frac(121.0f * ts));
#undef PL
  float mid = 0.5f * (yl + yr);
  float side = 0.5f * (yl - yr) * width;
  wl = mid + side; wr = mid - side;
}
__device__ __forceinline__ void plate_stereo(PlateDyn& d, const RingRef& r, const FxGeom& g, float& l, float& rr, const RateCtx& rc) {  // :552-565
  float li = isfinite(l) ? l : 0.0f, ri = isfinite(rr) ? rr : 0.0f;
  float wl, wr, mix;
  plate_tank(d, r, g, 0.5f * (li + ri), wl, wr, mix, rc);
  float ol = li * (1.0f - mix) + wl * mix, orr = ri * (1.0f - mix) + wr * mix;
  l = isfinite(ol) ? ol : li; rr = isfinite(orr) ? orr : ri;
}

// ---- effects whose oversampler history lives in the slot's ring arena (OS_WORDS floats per instance at `base`) ----
__device__ __forceinline__ void os_ring_load(Oversamp& o, const RingRef& r, uint32_t base) {
  float* w = reinterpret_cast<float*>(&o);
#pragma unroll 8
  for (uint32_t i = 0; i < OS_WORDS; i++) w[i] = r.at(base + i);
  o.mode = 4;                             // no FFI call changes the mode of an effect-slot oversampler: always X4
}
__device__ __forceinline__ void os_ring_store(const Oversamp& o, const RingRef& r, uint32_t base) {
  const float* w = reinterpret_cast<const float*>(&o);
#pragma unroll 8
  for (uint32_t i = 0; i < OS_WORDS; i++) r.at(base + i) = w[i];
}
__device__ __forceinline__ void os_ring_clear(const RingRef& r, uint32_t base) { for (uint32_t i = 0; i < OS_WORDS; i++) r.at(base + i) = 0.0f; }
static_assert(sizeof(Hb8) * 4 == OS_WORDS * 4 && offsetof(Oversamp, mode) == OS_WORDS * 4, "Oversamp = 64 history words + mode");

__device__ __forceinline__ float lowpass_one(LpDyn& d, int c, float in, const RateCtx& rc) {  // lowpass_filter.rs:129-194
  sm_set(d.cutoff[c], d.cutoff_target, 20.0f, 20000.0f);
  sm_set(d.res[c], d.res_target, 0.0f, 0.95f);
  const float cutoff = sm_tick(d.cutoff[c], rc.smooth30), resonance = sm_tick(d.res[c], rc.smooth30);
  const float max_cutoff = rc.sr * 0.40f;
  const float safe_cutoff = fminf(cutoff, max_cutoff);
  if (safe_cutoff != d.memo_c[c]) {           // g is a pure function of the smoothed cutoff: one expf per change, not per sample
    d.memo_c[c] = safe_cutoff;
    const float nf = safe_cutoff / rc.sr;
    d.memo_g[c] = clampf(1.0f - gm::g_expf(-2.0f * PI_F * nf), 0.0f, 0.90f);
  }
  const float g = d.memo_g[c];
  const float freq_ratio = fminf(safe_cutoff / 5000.0f, 1.0f);
  const float resonance_scale = 1.0f - (freq_ratio * freq_ratio * 0.7f);
  const float feedback = (resonance * resonance_scale) * 3.5f;
  const float fbs = d.stage2[c] * feedback;
  const float iwf = in - gm::g_tanhf(fbs) * fminf(feedback, 1.0f);
  d.stage1[c] += g * (iwf - d.stage1[c]);
  d.stage2[c] += g * (d.stage1[c] - d.stage2[c]);
  const float out = gm::g_tanhf(d.stage2[c]);
  if (fabsf(d.stage1[c]) < 1e-15f) d.stage1[c] = 0.0f;
  if (fabsf(d.stage2[c]) < 1e-15f) d.stage2[c] = 0.0f;
  if (!isfinite(out)) { d.stage1[c] = d.stage2[c] = 0.0f; return 0.0f; }
  return out;
}
__device__ __forceinline__ float dc_block(float in, float& x1, float& y1) {  // saturation.rs:135-146 == compressor.rs:120-130
  const float out = in - x1 + 0.995f * y1;
  x1 = in;
  y1 = fabsf(out) < 1e-15f ? 0.0f : out;
  return out;
}
constexpr float FRAC_2_PI_F = 0.63661977236758134308f;
// atanf: CUDA's (1 ulp) instead of a glibc port — it feeds half-band decimators, a DC blocker and a dry/wet mix only
// (bounded gain, no recurrence), like the tanh of the scan back ends (DESIGN.md "where approximation is allowed").
__device__ __forceinline__ float sat_shape(float in, float drive, float bias) {  // saturation.rs:104-123
  const float driven = in * drive;
  const float biased = driven + bias * fabsf(driven);
  const float soft = atanf(biased) * FRAC_2_PI_F;
  const float second = (soft * soft) * copysignf(1.0f, soft) * 0.15f;
  return soft + second * bias;
}
__device__ __forceinline__ float sat_one(SatDyn& d, int c, const RingRef& r, float in, const RateCtx& rc) {  // saturation.rs:202-255
  const uint32_t base = (uint32_t)c * OS_WORDS;
  if (!isfinite(in)) { d.dc_x1[c] = d.dc_y1[c] = 0.0f; os_ring_clear(r, base); return 0.0f; }
  sm_set(d.drive[c], d.t_drive, 0.0f, 1.0f); sm_set(d.warmth[c], d.t_warmth, 0.0f, 1.0f); sm_set(d.mix[c], d.t_mix, 0.0f, 1.0f);
  const float drive = 1.0f + sm_tick(d.drive[c], rc.smooth30) * 7.0f;
  const float warmth = sm_tick(d.warmth[c], rc.smooth30) * 0.4f;
  const float mix = sm_tick(d.mix[c], rc.smooth30);
  if (mix < 0.0001f) return in;
  Oversamp os;
  os_ring_load(os, r, base);
  const float sat = os_process(os, in, [&](float x) { return sat_shape(x, drive, warmth); });
  const float dcb = dc_block(sat, d.dc_x1[c], d.dc_y1[c]);
  const float out = in * (1.0f - mix) + dcb * mix;
  if (!isfinite(out)) { d.dc_x1[c] = d.dc_y1[c] = 0.0f; os_ring_clear(r, base); return 0.0f; }
  os_ring_store(os, r, base);
  return out;
}
__device__ __forceinline__ float comp_gr_db(float over_db, float ratio) {  // compressor.rs:103-117, 6 dB soft knee
  const float slope = 1.0f - 1.0f / ratio;
  if (over_db <= -3.0f) return 0.0f;
  if (over_db >= 3.0f) return over_db * slope;
  const float x = over_db + 3.0f;
  return x * x / (2.0f * 6.0f) * slope;
}
__device__ __forceinline__ float comp_one(CompDyn& d, int c, const RingRef& r, float in, float sidechain, const RateCtx& rc) {  // compressor.rs:133-250
  if (!isfinite(in) || !isfinite(sidechain)) return 0.0f;
  sm_set(d.th[c], d.t_th, -60.0f, 0.0f); sm_set(d.ratio[c], d.t_ratio, 1.0f, 20.0f); sm_set(d.att[c], d.t_att, 0.1f, 100.0f);
  sm_set(d.rel[c], d.t_rel, 5.0f, 1000.0f); sm_set(d.mix[c], d.t_mix, 0.0f, 1.0f);
  const float threshold_db = sm_tick(d.th[c], rc.smooth30), ratio = sm_tick(d.ratio[c], rc.smooth30), attack_ms = sm_tick(d.att[c], rc.smooth30);
  const float release_ms = sm_tick(d.rel[c], rc.smooth30), mix = sm_tick(d.mix[c], rc.smooth30);
  if (mix < 0.0001f) return in;
  const float sc = fabsf(sidechain);
  const float tms = sc > d.env[c] ? attack_ms : release_ms;
  const float coeff = gm::g_expf(-1.0f / (tms * 0.001f * rc.sr));
  d.env[c] = coeff * d.env[c] + (1.0f - coeff) * sc;
  if (d.env[c] < 1e-15f) d.env[c] = 0.0f;
  const float env_db = 20.0f * log10f(d.env[c] + 1e-20f);          // CUDA log10f (2 ulp): a level in dB that becomes a smoothed gain
  const float gr = comp_gr_db(env_db - threshold_db, ratio);
  const float gain_linear = gm::g_powf(10.0f, -gr * 0.05f);
  d.gain[c] += 0.05f * (gain_linear - d.gain[c]);
  const float compressed = in * d.gain[c];
  const uint32_t base = (uint32_t)c * OS_WORDS;
  Oversamp os;
  os_ring_load(os, r, base);
  const float colored_os = os_process(os, compressed, [](float x) { return atanf(x) * FRAC_2_PI_F * 1.1f; });
  os_ring_store(os, r, base);
  const float colored = d.gain[c] < 0.99f ? colored_os : compressed;
  const float dcb = dc_block(colored, d.dc_x1[c], d.dc_y1[c]);
  const float out = in * (1.0f - mix) + dcb * mix;
  if (!isfinite(out)) { d.dc_x1[c] = d.dc_y1[c] = 0.0f; d.env[c] = 0.0f; d.gain[c] = 1.0f; return 0.0f; }
  return out;
}
__device__ __forceinline__ float wsfx_one(WsDyn& d, int c, const RingRef& r, float in) {  // waveshaper.rs:48-72 on instance c
  if (isfinite(in) && (d.mix[c] <= 0.0001f || d.drive[c] <= 1.0f)) return in;   // bypass leaves the half-band history untouched
  const uint32_t base = (uint32_t)c * OS_WORDS;
  Oversamp os;
  os_ring_load(os, r, base);
  const float y = ws_core(d.drive[c], d.mix[c], os, in);
  os_ring_store(os, r, base);
  return y;
}
__device__ __forceinline__ float fbwsfx_one(FbwsDyn& d, int c, const RingRef& r, float in) {  // feedback_waveshaper.rs:109-169 on instance c
  FbSmall& w = d.s[c];
  if (isfinite(in) && (w.mix <= 0.0001f || w.drive <= 1.0f)) return in;
  const uint32_t base = (uint32_t)c * OS_WORDS;
  Oversamp os;
  os_ring_load(os, r, base);
  const float y = fbws_core(w, os, in);
  os_ring_store(os, r, base);
  return y;
}
// `reset()` of each reorderable effect, as gooey_engine_set_effect_order / move_effect call it (ffi.rs:1417-1425): saturation,
// low-pass, tilt, delay, compressor, spring, plate.  The two waveshapers are not in that list.
__device__ __forceinline__ void fx_reset(FxDyn& f, uint32_t kind, const RingRef& r, const FxGeom& g) {
  // a slot whose effect was never enabled has no ring arena yet (it is allocated zero-filled on first use): only its scalar state is reset
  const bool ring = r.base != nullptr;
  switch (kind) {
    case FXK_SATURATION: for (int c = 0; c < 2; c++) { f.sat.dc_x1[c] = f.sat.dc_y1[c] = 0.0f; if (ring) os_ring_clear(r, c * OS_WORDS); } break;
    case FXK_LOWPASS: for (int c = 0; c < 2; c++) f.lp.stage1[c] = f.lp.stage2[c] = 0.0f; break;
    case FXK_TILT: for (int c = 0; c < 2; c++) f.tilt.svf[c].ic1 = f.tilt.svf[c].ic2 = 0.0f; break;
    case FXK_DELAY:
      if (ring) for (uint32_t j = 0; j < 2u * g.delay_len; j++) r.at(j) = 0.0f;
      for (int c = 0; c < 2; c++) { f.delay.ch[c].write_index = 0; f.delay.ch[c].z1 = f.delay.ch[c].z2 = 0.0f; }
      break;
    case FXK_COMPRESSOR: for (int c = 0; c < 2; c++) { f.comp.env[c] = 0.0f; f.comp.gain[c] = 1.0f; f.comp.dc_x1[c] = f.comp.dc_y1[c] = 0.0f; if (ring) os_ring_clear(r, c * OS_WORDS); } break;
    case FXK_SPRING:
      if (ring) for (uint32_t j = 0; j < g.ring_words[2]; j++) r.at(j) = 0.0f;
      for (int c = 0; c < 2; c++) { for (int i = 0; i < 6; i++) f.spring.ch[c].idx[i] = 0; f.spring.ch[c].fb = f.spring.ch[c].damp = 0.0f; }
      break;
    case FXK_PLATE:
      if (ring) for (uint32_t j = 0; j < g.ring_words[3]; j++) r.at(j) = 0.0f;
      for (int i = 0; i < 13; i++) f.plate.idx[i] = 0;
      f.plate.bandwidth = f.plate.damp_a = f.plate.damp_b = f.plate.fb_a = f.plate.fb_b = f.plate.lfo_pa = f.plate.lfo_pb = 0.0f;
      break;
    default: break;
  }
}

__device__ __forceinline__ void fx_process(FxDyn& f, uint32_t kind, const RingRef& r, const FxGeom& g, float& l, float& rr, const RateCtx& rc, float sidechain = 0.0f, bool has_sidechain = false) {
  switch (kind) {
    case FXK_LOWPASS: l = lowpass_one(f.lp, 0, l, rc); rr = lowpass_one(f.lp, 1, rr, rc); break;
    case FXK_SATURATION: l = sat_one(f.sat, 0, r, l, rc); rr = sat_one(f.sat, 1, r, rr, rc); break;
    case FXK_COMPRESSOR: {
      const float sl = has_sidechain ? sidechain : l, sr_ = has_sidechain ? sidechain : rr;
      l = comp_one(f.comp, 0, r, l, sl, rc); rr = comp_one(f.comp, 1, r, rr, sr_, rc);
    } break;
    case FXK_WAVESHAPER: l = wsfx_one(f.ws, 0, r, l); rr = wsfx_one(f.ws, f.ws.shared ? 0 : 1, r, rr); break;
    case FXK_FBWS: l = fbwsfx_one(f.fbws, 0, r, l); rr = fbwsfx_one(f.fbws, f.fbws.shared ? 0 : 1, r, rr); break;
    case FXK_TILT: l = tilt_one(f.tilt, 0, l, rc); rr = tilt_one(f.tilt, 1, rr, rc); break;
    case FXK_DELAY: delay_stereo(f.delay, r, g.delay_len, l, rr, rc); break;
    case FXK_SPRING: {
      float dl[2][6];
#pragma unroll
      for (int c = 0; c < 2; c++)
#pragma unroll
        for (int i = 0; i < 6; i++) dl[c][i] = r.at(g.spring_off[c * 6 + i] + f.spring.ch[c].idx[i]);
      l = spring_one(f.spring, 0, r, g, l, rc, dl[0]); rr = spring_one(f.spring, 1, r, g, rr, rc, dl[1]);
    } break;
    case FXK_PLATE: plate_stereo(f.plate, r, g, l, rr, rc); break;
    default: break;
  }
}

__device__ __forceinline__ void mix_event(MixState& s, const MixCfg& cfg, const VoiceEvent& e, const RateCtx& rc) {
  switch (e.kind) {
    case MX_SET: {
      const uint32_t p = e.param;
      if (p < MP_CH_MUTE) sm_set(s.ch_gain[p - MP_CH_GAIN], e.value, 0.0f, 1.0f);
      else if (p < MP_CH_PAN) sm_set(s.ch_mute[p - MP_CH_MUTE], e.value, 0.0f, 1.0f);
      else if (p < MP_TR_GAIN) sm_set(s.ch_pan[p - MP_CH_PAN], e.value, 0.0f, 1.0f);
      else if (p < MP_TR_PAN) sm_set(s.tr_gain[p - MP_TR_GAIN], e.value, 0.0f, 2.0f);
      else if (p < MP_TR_MUTE) sm_set(s.tr_pan[p - MP_TR_PAN], e.value, 0.0f, 1.0f);
      else if (p < MP_MASTER) sm_set(s.tr_mute[p - MP_TR_MUTE], e.value, 0.0f, 1.0f);
      else if (p == MP_MASTER) sm_set(s.master, e.value, 0.0f, 2.0f);
    } break;
    case MX_SNAP:
      if (e.param == 0) { for (int i = 0; i < N_VOICE_CH; i++) { s.ch_mute[i].c = s.ch_mute[i].t; s.ch_gain[i].c = s.ch_gain[i].t; s.ch_pan[i].c = s.ch_pan[i].t; } }
      else if (e.param == 1) { for (int i = 0; i < MAX_TRACKS; i++) { s.tr_gain[i].c = s.tr_gain[i].t; s.tr_pan[i].c = s.tr_pan[i].t; s.tr_mute[i].c = s.tr_mute[i].t; } }
      else s.master.c = s.master.t;
      break;
    case MX_FX_SET: { uint32_t slot = e.param >> 8; if (slot < MAX_FX) fx_set_param(s.fx[slot], cfg.fx_kind[slot], e.param & 0xff, e.value, rc.sr); } break;
    case MX_FX_INIT: if (e.param < MAX_FX) fx_construct(s.fx[e.param], e.aux & 0xff, (e.aux >> 8) & 1u, rc.sr, e.value); break;   // aux bit 8: rack variant
    case MX_FX_BPM: if (e.param < MAX_FX && cfg.fx_kind[e.param] == FXK_DELAY) s.fx[e.param].delay.bpm_target = e.value; break;
    case MX_TRACK_INIT: if (e.param < MAX_TRACKS) { s.tr_gain[e.param] = {1.0f, 1.0f}; s.tr_pan[e.param] = {0.5f, 0.5f}; s.tr_mute[e.param] = {1.0f, 1.0f}; } break;
    default: break;
  }
}

#ifndef GOOEY_OWN_KERNELS_TU   // rs_chain.cu and poly_wave.cu compile only their own kernels
// One engine per thread.  Voice rows come in and the mix goes out through 32 engines x 32 frames shared-memory tiles,
// so every global access is a 128-byte row segment.
constexpr int MIX_CH = 7;
constexpr size_t MIX_DYN_SMEM = 32 * (sizeof(MixState) + sizeof(MixCfg));
__global__ void __launch_bounds__(32) mix_kernel(const MixLaunch L) {
  __shared__ float tin[MIX_CH][TILE * 33];
  __shared__ float tout[2][TILE * 33];
  __shared__ float tpre[2][TILE * 33];
  const int i = blockIdx.x * 32 + threadIdx.x;
  const int lane = threadIdx.x;
  const int warp_i0 = i - lane;
  if (warp_i0 >= L.n) return;
  const uint8_t fmode = (i < L.n && L.fast) ? L.fast[i] : 0;
  const bool valid = i < L.n && fmode != 1;
  const bool pre = valid && fmode == 2;          // strips / graph / master already mixed by mix_fast_kernel: only the global chain runs here
  const uint32_t row_mask = __ballot_sync(0xffffffffu, valid);
  if (row_mask == 0) return;
  const bool any_pre = __any_sync(0xffffffffu, pre), any_full = __any_sync(0xffffffffu, valid && !pre);
  const int n_rows = min(32, L.n - warp_i0);
  // The per-engine mixer state (414 words) and configuration are indexed with run-time slots (effect order, racks,
  // routes), which would put them in local memory — 3.7 MB for 2048 engines, thrashing L1 on every access.  They live in
  // dynamic shared memory instead (one struct per lane, 58 KB per CTA; MIX_DYN_SMEM).
  extern __shared__ __align__(16) unsigned char mix_dyn_smem[];
  MixState& st = reinterpret_cast<MixState*>(mix_dyn_smem)[lane];
  MixCfg& cfg = reinterpret_cast<MixCfg*>(mix_dyn_smem + 32 * sizeof(MixState))[lane];
  uint32_t ev = 0, ev_end = 0;
  int es = 0;
  if (valid) {
    es = (int)L.slots[i];
    load_words(st, L.state, es, L.state_cap, 0);
    cfg = L.cfg[es];
    ev = L.ev_begin[i]; ev_end = L.ev_begin[i + 1];
    if (pre) ev = ev_end;                          // mix_prepare_kernel consumed them (all at frame 0)
  }
  const RateCtx& rc = L.rc;
  // pan trig cache (pan is constant during a bounce; recomputed when the smoothed value moves)
  float pan_v[N_VOICE_CH], pan_cos[N_VOICE_CH], pan_sin[N_VOICE_CH];
#pragma unroll
  for (int c = 0; c < N_VOICE_CH; c++) { pan_v[c] = -1.0f; pan_cos[c] = pan_sin[c] = 0.0f; }
  float pk[N_VOICE_CH], tpk[MAX_TRACKS];   // record_peak: `if level > prev` (NaN never wins)
#pragma unroll
  for (int c = 0; c < N_VOICE_CH; c++) pk[c] = 0.0f;
#pragma unroll
  for (int t = 0; t < MAX_TRACKS; t++) tpk[t] = 0.0f;
  for (int f0 = 0; f0 < L.frames; f0 += TILE) {
    const int nf = min(TILE, L.frames - f0);
    if (any_full)
      for (int c = 0; c < MIX_CH; c++)
        if ((L.chan_mask >> c) & 1u) load_tile_rows_any(tin[c], L.voice_buf, L.voice_stride, c * L.n_lpad + warp_i0, n_rows, f0, nf, lane);
    if (any_pre)
      for (int c = 0; c < 2; c++) load_tile_rows_any(tpre[c], L.premix + (long long)c * L.n_lpad * L.premix_stride, L.premix_stride, warp_i0, n_rows, f0, nf, lane);
    __syncwarp();
    if (valid) {
      for (int j = 0; j < nf; j++) {
        const uint32_t frame = f0 + j;
        while (ev < ev_end && L.events[ev].frame <= frame) {
          const VoiceEvent& e = L.events[ev];
          if (e.kind == MX_FX_RESET) {   // reset_effect_states (ffi.rs:1417-1425): needs the ring arenas
            for (int s = 0; s < MAX_FX; s++) if (cfg.fx_kind[s] != FXK_NONE && !((cfg.fx_rack >> s) & 1u)) fx_reset(st.fx[s], cfg.fx_kind[s], RingRef{L.ring[s], L.ring_cap, es}, L.geo);
          } else {
            mix_event(st, cfg, e, rc);
            if (e.kind == MX_FX_INIT && e.param < MAX_FX && L.ring[e.param]) {   // a (re)built effect starts from silent delay lines
              const RingRef r{L.ring[e.param], L.ring_cap, es};
              const uint32_t k = e.aux & 0xff;
              const uint32_t words = k == FXK_DELAY ? L.geo.ring_words[1] : k == FXK_SPRING ? L.geo.ring_words[2] : k == FXK_PLATE ? L.geo.ring_words[3]
                                   : (k == FXK_SATURATION || k == FXK_COMPRESSOR || k == FXK_WAVESHAPER || k == FXK_FBWS) ? 2u * OS_WORDS : 0u;
              for (uint32_t j = 0; j < words; j++) r.at(j) = 0.0f;
            }
          }
          ev++;
        }
        float ml = 0.0f, mr = 0.0f;
        float channel_outs[N_VOICE_CH];
        if (pre) {
          ml = tpre[0][lane * 33 + j]; mr = tpre[1][lane * 33 + j];
#pragma unroll
          for (int c = 0; c < N_VOICE_CH; c++) channel_outs[c] = 0.0f;
        } else {
        float kit_l = 0.0f, kit_r = 0.0f, bass_l = 0.0f, bass_r = 0.0f;
#pragma unroll
        for (int c = 0; c < N_VOICE_CH; c++) {  // ffi.rs:1268-1283
          float x = tin[c][lane * 33 + j] * sm_tick(st.ch_gain[c], rc.smooth10) * sm_tick(st.ch_mute[c], rc.smooth10);
          channel_outs[c] = x;
          if (fabsf(x) > pk[c]) pk[c] = fabsf(x);
          float pan = sm_tick(st.ch_pan[c], rc.smooth10);
          if (pan != pan_v[c]) { float ang = clampf(pan, 0.0f, 1.0f) * 1.57079632679489661923f; pan_v[c] = pan; pan_cos[c] = gm::g_cosf(ang); pan_sin[c] = gm::g_sinf(ang); }
          float pl = x * pan_cos[c], pr = x * pan_sin[c];
          if (c < 4) { kit_l += pl; kit_r += pr; } else { bass_l += pl; bass_r += pr; }
        }
        float src_l[9] = {kit_l, bass_l, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f}, src_r[9] = {kit_r, bass_r, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
        if (cfg.src_poly) { float x = tin[5][lane * 33 + j]; src_l[2] = x * L.center_l; src_r[2] = x * L.center_r; }
        if (cfg.src_gran) { float x = tin[6][lane * 33 + j]; src_l[3] = x * L.center_l; src_r[3] = x * L.center_r; }
        if (cfg.src_ext && L.ext) {   // loop mixer and sampler racks: already stereo (ffi.rs:1289-1308)
#pragma unroll
          for (int s = 0; s < 5; s++)
            if ((cfg.src_ext >> s) & 1u) { const float* p = L.ext + (long long)(2u * cfg.ext_row[s]) * L.ext_stride + frame; src_l[4 + s] = p[0]; src_r[4 + s] = p[L.ext_stride]; }
        }
        for (uint32_t t = 0; t < cfg.n_tracks; t++) {  // graph.rs:344-350, 385-399
          float fl = 0.0f, fr = 0.0f;
#pragma unroll
          for (int s = 0; s < 5; s++) if (cfg.route[s] == (int32_t)t) { fl += src_l[s]; fr += src_r[s]; }
          if (cfg.src_ext >> 1) {
#pragma unroll
            for (int s = 5; s < 9; s++) if (cfg.route[s] == (int32_t)t) { fl += src_l[s]; fr += src_r[s]; }
          }
          float gain = sm_tick(st.tr_gain[t], rc.smooth10) * sm_tick(st.tr_mute[t], rc.smooth10);
          fl *= gain; fr *= gain;
          float pan = clampf(sm_tick(st.tr_pan[t], rc.smooth10), 0.0f, 1.0f);
          fl *= fminf(2.0f * (1.0f - pan), 1.0f);
          fr *= fminf(2.0f * pan, 1.0f);
          for (uint32_t k = 0; k < cfg.rack_n[t]; k++) {
            const uint32_t slot = cfg.rack_slot[t][k];
            fx_process(st.fx[slot], cfg.fx_kind[slot], RingRef{L.ring[slot], L.ring_cap, es}, L.geo, fl, fr, rc);
          }
          {
            const float lv = fmaxf(fabsf(fl), fabsf(fr));
#pragma unroll
            for (int q = 0; q < MAX_TRACKS; q++) if ((uint32_t)q == t && lv > tpk[q]) tpk[q] = lv;
          }
          ml += fl; mr += fr;
        }
        const float mg = sm_tick(st.master, rc.smooth30);
        ml *= mg; mr *= mg;
        }
#pragma unroll 1
        for (int o = 0; o < 9; o++) {  // ffi.rs:1317-1364
          const uint32_t id = cfg.order[o];
          const uint32_t slot = id < 12u ? cfg.gslot[id] : 0xffu;
          if (slot >= (uint32_t)MAX_FX || !cfg.fx_enabled[slot]) continue;
          float sc = 0.0f; bool has_sc = false;
          if (id == FXK_COMPRESSOR && cfg.comp_sidechain < (uint32_t)N_VOICE_CH) {   // ffi.rs:1331-1343
            has_sc = true;
#pragma unroll
            for (int c = 0; c < N_VOICE_CH; c++) if ((uint32_t)c == cfg.comp_sidechain) sc = channel_outs[c];
          }
          fx_process(st.fx[slot], id, RingRef{L.ring[slot], L.ring_cap, es}, L.geo, ml, mr, rc, sc, has_sc);
        }
        if (cfg.limiter_on) { ml = gm::g_tanhf(ml * cfg.lim_inv) * cfg.lim_th; mr = gm::g_tanhf(mr * cfg.lim_inv) * cfg.lim_th; }
        if (L.out_mode == 0) tout[0][lane * 33 + j] = 0.5f * (ml + mr);
        else { tout[0][lane * 33 + j] = ml; tout[1][lane * 33 + j] = mr; }
      }
    }
    __syncwarp();
    if (L.out_mode == 0) {
      store_tile_voice_major(tout[0], L.out, L.out_stride, warp_i0, L.out_rows ? L.out_rows + warp_i0 : nullptr, row_mask, f0, nf, lane);
    } else {
      // interleave L/R: row r, frame f -> out[row*stride + 2*(f0+f) + ch]; 64 consecutive floats per row
      for (int r = 0; r < n_rows; r++) {
        if (!((row_mask >> r) & 1u)) continue;     // rows of the time-parallel mixer (or past the end) are not this kernel's
        const long long row = L.out_rows ? (long long)L.out_rows[warp_i0 + r] : (long long)(warp_i0 + r);
        float* dst = L.out + row * L.out_stride + 2LL * f0;
        for (int k = lane; k < 2 * nf; k += 32) dst[k] = (k & 1) ? tout[1][r * 33 + (k >> 1)] : tout[0][r * 33 + (k >> 1)];
      }
    }
    __syncwarp();
  }
  if (valid) {
    store_words(st, L.state, es, L.state_cap, 0);
    if (L.peaks) {
      float* pp = L.peaks + (size_t)i * N_PEAKS;
#pragma unroll
      for (int c = 0; c < N_VOICE_CH; c++) if (pk[c] > pp[c]) pp[c] = pk[c];
#pragma unroll
      for (int t = 0; t < MAX_TRACKS; t++) if (tpk[t] > pp[N_VOICE_CH + t]) pp[N_VOICE_CH + t] = tpk[t];
    }
  }
}

// ---- time-parallel mixer ------------------------------------------------------------------------------------------
// With no effect in the chain or in any rack, the mixer's only memory is its smoothed parameters.  Once they have
// settled (cur == tgt, so SmoothedParam::tick returns the same value every sample) every output frame is the same
// pure function of that frame's voice samples, evaluated here in the reference's operation order — one thread per
// (engine, 4 frames) instead of one thread per engine.  mix_prepare_kernel (thread per engine) applies the launch's
// frame-0 events, decides eligibility and freezes the constants; events later in the launch disqualify the engine.
__global__ void __launch_bounds__(128) mix_prepare_kernel(const MixLaunch L) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= L.n) return;
  const int es = (int)L.slots[i];
  const MixCfg cfg = L.cfg[es];
  const uint32_t ev0 = L.ev_begin[i], ev1 = L.ev_begin[i + 1];
  bool ok = true, chain = false;
  for (int s = 0; s < MAX_FX; s++) chain = chain || (cfg.fx_kind[s] != FXK_NONE && cfg.fx_enabled[s] && !((cfg.fx_rack >> s) & 1u));
  for (uint32_t t = 0; t < cfg.n_tracks; t++) ok = ok && cfg.rack_n[t] == 0;
  for (uint32_t e = ev0; e < ev1; e++) ok = ok && L.events[e].frame == 0 && L.events[e].kind != MX_FX_INIT && L.events[e].kind != MX_FX_RESET;
  // a global chain does not disqualify the engine: its strips / graph / master still run time-parallel (fast = 2) and only
  // the chain is left to the per-engine kernel — unless the compressor listens to a voice strip (ffi.rs:1331-1343)
  if (chain && cfg.comp_sidechain < (uint32_t)N_VOICE_CH) ok = false;
  if (chain && !L.premix) ok = false;
  if (!ok) { L.fast[i] = 0; return; }
  MixState st;
  load_words(st, L.state, es, L.state_cap, 0);
  for (uint32_t e = ev0; e < ev1; e++) mix_event(st, cfg, L.events[e], L.rc);
  for (int c = 0; c < N_VOICE_CH; c++) ok = ok && st.ch_gain[c].c == st.ch_gain[c].t && st.ch_mute[c].c == st.ch_mute[c].t && st.ch_pan[c].c == st.ch_pan[c].t;
  for (uint32_t t = 0; t < cfg.n_tracks; t++) ok = ok && st.tr_gain[t].c == st.tr_gain[t].t && st.tr_mute[t].c == st.tr_mute[t].t && st.tr_pan[t].c == st.tr_pan[t].t;
  ok = ok && st.master.c == st.master.t;
  L.fast[i] = ok ? (chain ? 2 : 1) : 0;
  if (!ok) return;                                   // state untouched: the general kernel re-applies the events itself
  store_words(st, L.state, es, L.state_cap, 0);      // events consumed
  MixConst k;
  for (int c = 0; c < N_VOICE_CH; c++) {
    k.g[c] = st.ch_gain[c].c; k.m[c] = st.ch_mute[c].c;
    const float ang = clampf(st.ch_pan[c].c, 0.0f, 1.0f) * 1.57079632679489661923f;
    k.pc[c] = gm::g_cosf(ang); k.ps[c] = gm::g_sinf(ang);
  }
  for (int t = 0; t < MAX_TRACKS; t++) {
    k.tgain[t] = st.tr_gain[t].c * st.tr_mute[t].c;
    const float pan = clampf(st.tr_pan[t].c, 0.0f, 1.0f);
    k.tbl[t] = fminf(2.0f * (1.0f - pan), 1.0f); k.tbr[t] = fminf(2.0f * pan, 1.0f);
  }
  k.master = st.master.c; k.lim_th = cfg.lim_th; k.lim_inv = cfg.lim_inv;
  k.n_tracks = cfg.n_tracks; k.limiter_on = chain ? 0u : cfg.limiter_on; k.src_poly = cfg.src_poly; k.src_gran = cfg.src_gran;   // the limiter follows the chain
  for (int s = 0; s < 9; s++) k.route[s] = cfg.route[s];
  k.src_ext = L.ext ? cfg.src_ext : 0u;
  for (int s = 0; s < 5; s++) k.ext_row[s] = cfg.ext_row[s];
  L.consts[i] = k;
}

__device__ __forceinline__ void mix_fast_frame(const MixConst& k, const float* x, const float* ext_l, const float* ext_r, float center_l, float center_r,
                                               float& ml, float& mr, float* pk) {
  float kit_l = 0.0f, kit_r = 0.0f, bass_l = 0.0f, bass_r = 0.0f;
#pragma unroll
  for (int c = 0; c < N_VOICE_CH; c++) {
    const float v = x[c] * k.g[c] * k.m[c];
    if (fabsf(v) > pk[c]) pk[c] = fabsf(v);
    const float pl = v * k.pc[c], pr = v * k.ps[c];
    if (c < 4) { kit_l += pl; kit_r += pr; } else { bass_l += pl; bass_r += pr; }
  }
  float src_l[9] = {kit_l, bass_l, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f}, src_r[9] = {kit_r, bass_r, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
  if (k.src_poly) { src_l[2] = x[5] * center_l; src_r[2] = x[5] * center_r; }
  if (k.src_gran) { src_l[3] = x[6] * center_l; src_r[3] = x[6] * center_r; }
  if (k.src_ext) {
#pragma unroll
    for (int s = 0; s < 5; s++) if ((k.src_ext >> s) & 1u) { src_l[4 + s] = ext_l[s]; src_r[4 + s] = ext_r[s]; }
  }
  ml = 0.0f; mr = 0.0f;
  for (uint32_t t = 0; t < k.n_tracks; t++) {
    float fl = 0.0f, fr = 0.0f;
#pragma unroll
    for (int s = 0; s < 5; s++) if (k.route[s] == (int32_t)t) { fl += src_l[s]; fr += src_r[s]; }
    if (k.src_ext >> 1) {
#pragma unroll
      for (int s = 5; s < 9; s++) if (k.route[s] == (int32_t)t) { fl += src_l[s]; fr += src_r[s]; }
    }
    fl *= k.tgain[t]; fr *= k.tgain[t];
    fl *= k.tbl[t]; fr *= k.tbr[t];
    {
      const float lv = fmaxf(fabsf(fl), fabsf(fr));
#pragma unroll
      for (int q = 0; q < MAX_TRACKS; q++) if ((uint32_t)q == t && lv > pk[N_VOICE_CH + q]) pk[N_VOICE_CH + q] = lv;
    }
    ml += fl; mr += fr;
  }
  ml *= k.master; mr *= k.master;
  if (k.limiter_on) { ml = gm::g_tanhf(ml * k.lim_inv) * k.lim_th; mr = gm::g_tanhf(mr * k.lim_inv) * k.lim_th; }
}

// grid = (ceil(frames / 1024), n engines), 256 threads, 4 frames per thread
__global__ void __launch_bounds__(256) mix_fast_kernel(const MixLaunch L) {
  const int i = blockIdx.y;
  if (!L.fast[i]) return;
  const int f = (blockIdx.x * 256 + threadIdx.x) * 4;
  __shared__ MixConst ks;
  if (threadIdx.x == 0) ks = L.consts[i];
  __syncthreads();
  if (f >= L.frames) return;
  const int nf = min(4, L.frames - f);
  const bool vec_in = nf == 4 && (L.voice_stride & 3) == 0;
  float x[MIX_CH][4];
#pragma unroll
  for (int c = 0; c < MIX_CH; c++) {
    x[c][0] = x[c][1] = x[c][2] = x[c][3] = 0.0f;
    if (!((L.chan_mask >> c) & 1u)) continue;
    if (c == 5 && !ks.src_poly) continue;
    if (c == 6 && !ks.src_gran) continue;
    const float* row = L.voice_buf + (long long)(c * L.n_lpad + i) * L.voice_stride + f;
    if (vec_in) { const float4 v = *reinterpret_cast<const float4*>(row); x[c][0] = v.x; x[c][1] = v.y; x[c][2] = v.z; x[c][3] = v.w; }
    else for (int q = 0; q < nf; q++) x[c][q] = row[q];
  }
  float ol[4], orr[4], pk[N_PEAKS];
#pragma unroll
  for (int q = 0; q < N_PEAKS; q++) pk[q] = 0.0f;
#pragma unroll
  for (int q = 0; q < 4; q++) {
    float xs[MIX_CH];
#pragma unroll
    for (int c = 0; c < MIX_CH; c++) xs[c] = x[c][q];
    float junk[N_PEAKS];
    float el[5] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f}, er[5] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    if (ks.src_ext && q < nf) {
#pragma unroll
      for (int s = 0; s < 5; s++)
        if ((ks.src_ext >> s) & 1u) { const float* p = L.ext + (long long)(2u * ks.ext_row[s]) * L.ext_stride + f + q; el[s] = p[0]; er[s] = p[L.ext_stride]; }
    }
    mix_fast_frame(ks, xs, el, er, L.center_l, L.center_r, ol[q], orr[q], q < nf ? pk : junk);
  }
  if (L.peaks) {   // maxima of non-negative floats compare like their bit patterns: warp reduce, then one atomic per value
    unsigned* pp = reinterpret_cast<unsigned*>(L.peaks + (size_t)i * N_PEAKS);
    const unsigned act = __activemask();
#pragma unroll
    for (int q = 0; q < N_PEAKS; q++) {
      if (q >= N_VOICE_CH + (int)ks.n_tracks) break;
      const unsigned m = __reduce_max_sync(act, __float_as_uint(pk[q]));
      if ((threadIdx.x & 31) == (__ffs(act) - 1) && m > pp[q]) atomicMax(pp + q, m);
    }
  }
  if (L.fast[i] == 2) {          // pre-chain mix for the general kernel
    float* pl = L.premix + (long long)i * L.premix_stride + f;
    float* pr = pl + (long long)L.n_lpad * L.premix_stride;
    if (nf == 4 && (L.premix_stride & 3) == 0) { *reinterpret_cast<float4*>(pl) = make_float4(ol[0], ol[1], ol[2], ol[3]); *reinterpret_cast<float4*>(pr) = make_float4(orr[0], orr[1], orr[2], orr[3]); }
    else for (int q = 0; q < nf; q++) { pl[q] = ol[q]; pr[q] = orr[q]; }
    return;
  }
  const long long row = L.out_rows ? (long long)L.out_rows[i] : (long long)i;
  if (L.out_mode == 0) {
    float* dst = L.out + row * L.out_stride + f;
    if (nf == 4 && (L.out_stride & 3) == 0 && (reinterpret_cast<uintptr_t>(L.out) & 15) == 0)
      *reinterpret_cast<float4*>(dst) = make_float4(0.5f * (ol[0] + orr[0]), 0.5f * (ol[1] + orr[1]), 0.5f * (ol[2] + orr[2]), 0.5f * (ol[3] + orr[3]));
    else for (int q = 0; q < nf; q++) dst[q] = 0.5f * (ol[q] + orr[q]);
  } else {
    float* dst = L.out + row * L.out_stride + 2LL * f;
    for (int q = 0; q < nf; q++) { dst[2 * q] = ol[q]; dst[2 * q + 1] = orr[q]; }
  }
}
// 16-bit PCM of rows of f32 samples: `(s * 32767.0).round() as i16` (bounce.rs:105-113, ffi.rs:7968-7972: f32::round = half
// away from zero, saturating cast, NaN -> 0).  grid = (ceil(cols / 1024), rows), 256 threads, 4 samples per thread.
__device__ __forceinline__ int16_t pcm16_of(float s) {
  const float r = roundf(s * 32767.0f);
  return (int16_t)(r != r ? 0 : (r >= 32767.0f ? 32767 : (r <= -32768.0f ? -32768 : (int)r)));
}
__global__ void __launch_bounds__(256) quantize_pcm16_kernel(const float* __restrict__ in, long long in_stride, int16_t* __restrict__ out, long long out_stride,
                                                             int col0, int cols) {
  const int c = (blockIdx.x * 256 + threadIdx.x) * 4;
  if (c >= cols) return;
  const float* src = in + (long long)blockIdx.y * in_stride + col0 + c;
  int16_t* dst = out + (long long)blockIdx.y * out_stride + col0 + c;
  const int nq = min(4, cols - c);
  if (nq == 4 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0) && ((reinterpret_cast<uintptr_t>(dst) & 7) == 0)) {
    const float4 v = *reinterpret_cast<const float4*>(src);
    short4 q; q.x = pcm16_of(v.x); q.y = pcm16_of(v.y); q.z = pcm16_of(v.z); q.w = pcm16_of(v.w);
    *reinterpret_cast<short4*>(dst) = q;
  } else for (int k = 0; k < nq; k++) dst[k] = pcm16_of(src[k]);
}
#endif  // GOOEY_OWN_KERNELS_TU
#endif  // __CUDACC__

}  // namespace gd
