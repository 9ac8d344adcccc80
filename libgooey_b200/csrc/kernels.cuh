// kernels.cuh — the voice render kernels.
//
// A voice's render is split three ways (DESIGN.md "A/B/C"):
//   plan_kernel  (A) one thread per voice: applies the call's events to the control half of the state, checks that
//                    every smoothed parameter is settled, and emits one Span per event-free stretch: a snapshot of the
//                    control half plus the analytically advanced envelope latches.
//   front_kernel (B) one thread per (voice, frame): the pure part of the tick — additive oscillators, SipHash noise,
//                    envelope curves — evaluated from the span snapshot, written to per-voice planes.  This is where
//                    the FP32/FP64 work is; it scales over time, not just over voices.
//   back_kernel  (C) one thread per voice, sample-serial: filters, oversampled waveshapers, RNG-driven oscillators;
//                    reads the planes through 32x32 shared-memory tiles and writes the output the same way
//                    (128-bit coalesced stores).
//   slow_kernel  (S) one thread per voice, the reference's whole tick per sample.  Used for voices whose parameters
//                    are still gliding when the call starts or are edited without a snap (A marks them), for
//                    LFO-routed basses, and for basses and poly synths under GOOEY_B200_BACKEND=serial (pool.cuh launch_back).
// Output layout: out[row * stride + frame] (voice-major).  State layout: word-interleaved SoA, state[w * n_pad + slot].
#pragma once
#include <cuda_runtime.h>
#include "voices2.cuh"
#include "../../include/gooey_batch.h"

namespace gd {

constexpr int TILE = 32;

template <class S> __device__ __forceinline__ void load_words(S& s, const uint32_t* base, int slot, int n_pad, int w0) {
  constexpr int W = sizeof(S) / 4;
  uint32_t* w = reinterpret_cast<uint32_t*>(&s);
#pragma unroll
  for (int i = 0; i < W; i++) w[i] = base[(size_t)(w0 + i) * n_pad + slot];
}
template <class S> __device__ __forceinline__ void store_words(const S& s, uint32_t* base, int slot, int n_pad, int w0) {
  constexpr int W = sizeof(S) / 4;
  const uint32_t* w = reinterpret_cast<const uint32_t*>(&s);
#pragma unroll
  for (int i = 0; i < W; i++) base[(size_t)(w0 + i) * n_pad + slot] = w[i];
}

// ------------------------------------------------------------------------------------------- voice traits ----
// ID: the instrument id (GooeyVoicePatch::instrument) that selects the type.
struct KickV {
  using State = KickState; using Ctl = KickCtl; using Aud = KickAud; using Span = KickSpan;
  static constexpr bool FAST = true; static constexpr int NPL = KICK_PLANES; static constexpr uint32_t ID = GOOEY_INSTRUMENT_KICK;
  struct Run { KickDer d; int j_act; };
  static __device__ __forceinline__ float tick(State& s, const double* tt, const RateCtx& rc) { return kick_tick(s, tt, rc); }
  static __device__ __forceinline__ void slow_event(State& s, const VoiceEvent& e, const double* tt, const RateCtx&) {
    uint32_t r = 0; kick_event(s.c, e, tt, r); kick_span_begin(s.a, s.c, r);
  }
  static __device__ __forceinline__ bool settled(const Ctl& c) { return params_settled<K_NP>(c.cur, c.tgt); }
  static __device__ __forceinline__ void event(Ctl& c, const VoiceEvent& e, const double* tt, uint32_t& r) { kick_event(c, e, tt, r); }
  static __device__ __forceinline__ void plan(Ctl& c, uint32_t r, const double* tt, int ja, int jb, Span& sp) { kick_plan(c, r, tt, ja, jb, sp); }
  static __device__ __forceinline__ int front_end(const Span& sp) { return sp.j_act; }
  static __device__ __forceinline__ void front(const Span& sp, double now, uint32_t, float sr, float* o) {
    // ~1-ulp sine in the additive oscillators unless the feedback waveshaper's drive would amplify that ulp past the
    // parity margin (its tanh has slope `drive` at the origin, up to 100)
    KickFront f = sp.d.drive <= 8.0f ? kick_front<true>(sp.c, sp.d, now, sr) : kick_front<false>(sp.c, sp.d, now, sr);
    o[0] = f.p1; o[1] = f.raw_click; o[2] = f.ne; o[3] = f.amp;
  }
  static __device__ __forceinline__ void span_begin(Aud& a, const Span& sp, Run& r, float) { kick_span_begin(a, sp.c, sp.resets); r.d = sp.d; r.j_act = sp.j_act; }
  static __device__ __forceinline__ void span_resume(const Span& sp, Run& r) { r.d = sp.d; r.j_act = sp.j_act; }
  static __device__ __forceinline__ bool wants_planes(const Aud&, const Run& r, int j) { return j < r.j_act; }
  static __device__ __forceinline__ bool is_active(const Aud&, const Run& r, int j) { return j < r.j_act; }
  static __device__ __forceinline__ float back(Aud& a, const Run& r, int j, const float* p, const RateCtx& rc) {
    if (j >= r.j_act) return 0.0f;
    KickFront f; f.p1 = p[0]; f.raw_click = p[1]; f.ne = p[2]; f.amp = p[3];
    return kick_back(a, r.d, f, rc);
  }
};
struct SnareV {
  using State = SnareState; using Ctl = SnareCtl; using Aud = SnareAud; using Span = SnareSpan;
  static constexpr bool FAST = true; static constexpr int NPL = SNARE_PLANES; static constexpr uint32_t ID = GOOEY_INSTRUMENT_SNARE;
  struct Run { SnareDer d; int j_act; };
  static __device__ __forceinline__ float tick(State& s, const double* tt, const RateCtx& rc) { return snare_tick(s, tt, rc); }
  static __device__ __forceinline__ void slow_event(State& s, const VoiceEvent& e, const double* tt, const RateCtx&) {
    uint32_t r = 0; snare_event(s.c, e, tt, r); snare_span_begin(s.a, s.c, r);
  }
  static __device__ __forceinline__ bool settled(const Ctl& c) { return params_settled<S_NP>(c.cur, c.tgt); }
  static __device__ __forceinline__ void event(Ctl& c, const VoiceEvent& e, const double* tt, uint32_t& r) { snare_event(c, e, tt, r); }
  static __device__ __forceinline__ void plan(Ctl& c, uint32_t r, const double* tt, int ja, int jb, Span& sp) { snare_plan(c, r, tt, ja, jb, sp); }
  static __device__ __forceinline__ int front_end(const Span& sp) { return sp.j_act; }
  static __device__ __forceinline__ void front(const Span& sp, double now, uint32_t, float sr, float* o) {
    SnareFront f = snare_front<true>(sp.c, sp.d, now, sr);      // the snare's waveshaper drive is at most 10
    o[0] = f.tonal_out; o[1] = f.raw_noise; o[2] = f.cne; o[3] = f.crack_out; o[4] = f.amp;
  }
  static __device__ __forceinline__ void span_begin(Aud& a, const Span& sp, Run& r, float) { snare_span_begin(a, sp.c, sp.resets); r.d = sp.d; r.j_act = sp.j_act; }
  static __device__ __forceinline__ void span_resume(const Span& sp, Run& r) { r.d = sp.d; r.j_act = sp.j_act; }
  static __device__ __forceinline__ bool wants_planes(const Aud&, const Run& r, int j) { return j < r.j_act; }
  static __device__ __forceinline__ bool is_active(const Aud&, const Run& r, int j) { return j < r.j_act; }
  static __device__ __forceinline__ float back(Aud& a, const Run& r, int j, const float* p, const RateCtx& rc) {
    if (j >= r.j_act) return 0.0f;
    SnareFront f; f.tonal_out = p[0]; f.raw_noise = p[1]; f.cne = p[2]; f.crack_out = p[3]; f.amp = p[4];
    return snare_back(a, r.d, f, rc);
  }
};
struct HatV {
  using State = HatState; using Ctl = HatCtl; using Aud = HatAud; using Span = HatSpan;
  static constexpr bool FAST = true; static constexpr int NPL = HAT_PLANES; static constexpr uint32_t ID = GOOEY_INSTRUMENT_HIHAT;
  struct Run { HatDer d; int j_env; float env_final; };
  static __device__ __forceinline__ float tick(State& s, const double* tt, const RateCtx& rc) { return hat_tick(s, tt, rc); }
  static __device__ __forceinline__ void slow_event(State& s, const VoiceEvent& e, const double* tt, const RateCtx&) {
    uint32_t r = 0; hat_event(s.c, e, tt, r); hat_span_begin(s.a, s.c, r);
  }
  static __device__ __forceinline__ bool settled(const Ctl& c) { return params_settled<H_NP>(c.cur, c.tgt); }
  static __device__ __forceinline__ void event(Ctl& c, const VoiceEvent& e, const double* tt, uint32_t& r) { hat_event(c, e, tt, r); }
  static __device__ __forceinline__ void plan(Ctl& c, uint32_t r, const double* tt, int ja, int jb, Span& sp) { hat_plan(c, r, tt, ja, jb, sp); }
  static __device__ __forceinline__ int front_end(const Span& sp) { return sp.j_env < sp.j1 ? sp.j_env : sp.j1; }
  static __device__ __forceinline__ void front(const Span& sp, double now, uint32_t, float sr, float* o) { o[0] = hat_front(sp.c, sp.d, now, sr).env; }
  static __device__ __forceinline__ void span_begin(Aud& a, const Span& sp, Run& r, float) { hat_span_begin(a, sp.c, sp.resets); span_resume(sp, r); }
  static __device__ __forceinline__ void span_resume(const Span& sp, Run& r) { r.d = sp.d; r.j_env = sp.j_env; r.env_final = sp.env_final; }
  static __device__ __forceinline__ bool wants_planes(const Aud& a, const Run& r, int j) { return a.active && j < r.j_env; }
  static __device__ __forceinline__ bool is_active(const Aud& a, const Run&, int) { return a.active != 0; }
  static __device__ __forceinline__ float back(Aud& a, const Run& r, int j, const float* p, const RateCtx& rc) {
    if (!a.active) return 0.0f;
    HatFront f; f.env = j < r.j_env ? p[0] : r.env_final;
    return hat_back(a, r.d, f, j >= r.j_env, rc);
  }
};
struct TomV {
  using State = TomState; using Ctl = TomCtl; using Aud = TomAud; using Span = TomSpan;
  static constexpr bool FAST = true; static constexpr int NPL = TOM_PLANES; static constexpr uint32_t ID = GOOEY_INSTRUMENT_TOM;
  struct Run { TomDer d; int j_env; float env_final; };
  static __device__ __forceinline__ float tick(State& s, const double* tt, const RateCtx& rc) { return tom_tick(s, tt, rc); }
  static __device__ __forceinline__ void slow_event(State& s, const VoiceEvent& e, const double* tt, const RateCtx& rc) {
    uint32_t r = 0; tom_event(s.c, e, tt, r); tom_span_begin(s.a, s.c.mem_q_scale, s.c.mem_gain_scale, s.c.mem_dirty, r, rc.sr); s.c.mem_dirty = 0;
  }
  static __device__ __forceinline__ bool settled(const Ctl&) { return true; }   // Tom2 parameters are not smoothed (tom2.rs:66-79)
  static __device__ __forceinline__ void event(Ctl& c, const VoiceEvent& e, const double* tt, uint32_t& r) { tom_event(c, e, tt, r); }
  static __device__ __forceinline__ void plan(Ctl& c, uint32_t r, const double* tt, int ja, int jb, Span& sp) { tom_plan(c, r, tt, ja, jb, sp); }
  // the hash planes are needed for as long as the voice may ring (membrane), i.e. the whole span
  static __device__ __forceinline__ int front_end(const Span& sp) { return sp.d.membrane > 0.0f ? sp.j1 : (sp.j_env < sp.j1 ? sp.j_env + 1 : sp.j1); }
  static __device__ __forceinline__ void front(const Span& sp, double now, uint32_t k, float, float* o) {
    TomFront f = tom_front(sp.c, sp.d, now, k); o[0] = f.env; o[1] = f.noise; o[2] = f.rnd;
  }
  static __device__ __forceinline__ void span_begin(Aud& a, const Span& sp, Run& r, float sr) {
    tom_span_begin(a, sp.mem_q_scale, sp.mem_gain_scale, sp.mem_dirty, sp.resets, sr); span_resume(sp, r);
  }
  static __device__ __forceinline__ void span_resume(const Span& sp, Run& r) { r.d = sp.d; r.j_env = sp.j_env; r.env_final = sp.env_final; }
  static __device__ __forceinline__ bool wants_planes(const Aud& a, const Run&, int) { return a.active != 0; }
  static __device__ __forceinline__ bool is_active(const Aud& a, const Run&, int) { return a.active != 0; }
  static __device__ __forceinline__ float back(Aud& a, const Run& r, int j, const float* p, const RateCtx& rc) {
    if (!a.active) return 0.0f;
    TomFront f; f.env = j < r.j_env ? p[0] : r.env_final; f.noise = p[1]; f.rnd = p[2];
    return tom_back(a, r.d, f, j >= r.j_env, rc);
  }
};
struct BassV { using State = BassState; static constexpr bool FAST = false; static constexpr uint32_t ID = GOOEY_INSTRUMENT_BASS;
  static __device__ __forceinline__ float tick(State& s, const double* tt, const RateCtx& rc) { return bass_tick(s, tt, rc); }
  static __device__ __forceinline__ void slow_event(State& s, const VoiceEvent& e, const double* tt, const RateCtx&) { bass_event(s, e, tt); } };
struct PolyV { using State = PolyState; static constexpr bool FAST = false; static constexpr uint32_t ID = GOOEY_B200_VOICE_POLY;
  static __device__ __forceinline__ float tick(State& s, const double* tt, const RateCtx& rc) { return poly_tick(s, tt, rc); }
  static __device__ __forceinline__ void slow_event(State& s, const VoiceEvent& e, const double* tt, const RateCtx&) { poly_event(s, e, tt); } };
struct GranV { using State = GranState; static constexpr bool FAST = false; static constexpr uint32_t ID = GOOEY_B200_VOICE_GRANULATOR;
  static __device__ __forceinline__ float tick(State& s, const double* tt, const RateCtx& rc) { return gran_tick(s, tt, rc); }
  static __device__ __forceinline__ void slow_event(State& s, const VoiceEvent& e, const double* tt, const RateCtx&) { gran_event(s, e, tt); } };

// ------------------------------------------------------------------------------------------- launch records ----
// One LFO route of a voice (ffi.rs:1238-1251): every frame, after the frame's events and before the tick, the voice's parameter
// `param` (internal index) receives `apply_modulation(plane[frame] * depth)` (ffi.rs:322-405).
//   mode 0: smoothed parameter, set_bipolar (smoother.rs:105-115): target = (clamp(m, -1, 1) + 1) * 0.5
//   mode 1: Tom2 plain parameter: set_*(m * 100), clamped to 0..100          mode 2: Tom2 tuning: clamp(m, 0, 1)
struct ModRoute { uint32_t param, mode; float depth; uint32_t plane; };
struct LfoStream { float phase, inc, amount, offset; int plane; };   // plane: row of the value planes, -1 = enabled but unrouted (the phase still runs)

struct VoiceLaunch {
  uint32_t* state;           // [words][n_pad]
  int n, n_pad;
  const uint32_t* slots;     // launch index -> pool slot (nullptr = identity)
  const uint32_t* rows;      // launch index -> output row (nullptr = row0 + index)
  int row0;
  const VoiceEvent* events;  // per-voice lists, sorted by frame; frames are relative to the call
  const uint32_t* ev_begin;  // [n+1]
  const double* tt;          // engine clock table
  int frames;                // frames in the call
  float* out; long long stride;
  RateCtx rc;
  // fast path
  uint8_t* mode;             // [n] 0 = fast (A/B/C), 1 = general (S)
  void* spans;               // Span[ span_off[n] ]
  const uint32_t* span_off;  // [n+1]
  uint32_t* n_spans;         // [n]
  uint32_t* span_cursor;     // [n] current span of each voice across chunked C launches
  float* planes;             // [NPL][n_rows_pad][pitch] for the current chunk
  long long plane_stride;    // floats between planes
  int pitch;                 // floats between rows of a plane (chunk capacity, multiple of 32)
  int chunk0, chunk_frames;  // frames [chunk0, chunk0 + chunk_frames) of the call
  // LFO modulation (nullptr = none): routes of voice v = routes[route_begin[v] .. route_begin[v + 1]); LFO values of the call's
  // frame j at mod_planes[plane * mod_pitch + mod_frame0 + j]
  const ModRoute* routes; const uint32_t* route_begin;
  const float* mod_planes; long long mod_pitch; int mod_frame0;
};

// Warp-cooperative store of a 32x32 tile (tile[lane][frame]) to voice-major output; row_mask = rows to write.
__device__ __forceinline__ void store_tile_voice_major(const float* tile /*[32][33]*/, float* out, long long stride, int row0,
                                                        const uint32_t* rows, uint32_t row_mask, int f0, int nf, int lane) {
  const bool vec_ok = (nf == TILE) && ((stride & 3) == 0) && ((f0 & 3) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
  if (vec_ok) {
    const int c = (lane & 7) * 4;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const int r = k * 4 + (lane >> 3);
      if ((row_mask >> r) & 1u) {
        const float* src = tile + r * 33 + c;
        float4 v = make_float4(src[0], src[1], src[2], src[3]);
        const long long row = rows ? (long long)rows[r] : (long long)(row0 + r);
        *reinterpret_cast<float4*>(out + row * stride + f0 + c) = v;
      }
    }
  } else {
    for (int r = 0; r < 32; r++) {
      if (!((row_mask >> r) & 1u)) continue;
      const long long row = rows ? (long long)rows[r] : (long long)(row0 + r);
      if (lane < nf) out[row * stride + f0 + lane] = tile[r * 33 + lane];
    }
  }
}
// Warp-cooperative load of a 32 rows x 32 floats tile from a row-major plane (pitch multiple of 4, 16B-aligned rows).
__device__ __forceinline__ void load_tile_rows(float* tile /*[32][33]*/, const float* plane, int pitch, int row0, int n_rows, int c0, int lane) {
  const int c = (lane & 7) * 4;
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const int r = k * 4 + (lane >> 3);
    if (r < n_rows) {
      const float4 v = *reinterpret_cast<const float4*>(plane + (size_t)(row0 + r) * pitch + c0 + c);
      float* dst = tile + r * 33 + c;
      dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
    }
  }
}

// Same for any pitch / alignment / partial width (scalar loads, still one 128-byte segment per row).
__device__ __forceinline__ void load_tile_rows_any(float* tile /*[32][33]*/, const float* plane, long long pitch, int row0, int n_rows, int c0, int nf, int lane) {
  for (int r = 0; r < n_rows; r++)
    if (lane < nf) tile[r * 33 + lane] = plane[(long long)(row0 + r) * pitch + c0 + lane];
}

// ------------------------------------------------------------------------------------------- S: general path ----
template <class V, int BLOCK>
__global__ void __launch_bounds__(BLOCK) slow_kernel(const VoiceLaunch L) {
  __shared__ float tiles[BLOCK / 32][TILE * 33];
  const int v = blockIdx.x * BLOCK + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warp_v0 = v - lane;
  if (warp_v0 >= L.n) return;
  bool mine = v < L.n;
  if (V::FAST && mine) mine = L.mode[v] != 0;
  const uint32_t row_mask = __ballot_sync(0xffffffffu, mine);
  if (row_mask == 0) return;
  typename V::State st;
  uint32_t ev = 0, ev_end = 0;
  int sv = v;
  if (mine) {
    if (L.slots) sv = (int)L.slots[v];
    load_words(st, L.state, sv, L.n_pad, 0);
    ev = L.ev_begin[v];
    ev_end = L.ev_begin[v + 1];
  }
  uint32_t r0 = 0, r1 = 0;
  if (mine && L.routes) { r0 = L.route_begin[v]; r1 = L.route_begin[v + 1]; }
  float* tile = tiles[warp];
  for (int f0 = 0; f0 < L.frames; f0 += TILE) {
    const int nf = min(TILE, L.frames - f0);
    if (mine) {
      for (int j = 0; j < nf; j++) {
        const uint32_t frame = f0 + j;
        while (ev < ev_end && L.events[ev].frame <= frame) { V::slow_event(st, L.events[ev], L.tt, L.rc); ev++; }
        for (uint32_t q = r0; q < r1; q++) {       // LFO pool: after the triggers, before the tick
          const ModRoute r = L.routes[q];
          const float m = L.mod_planes[(long long)r.plane * L.mod_pitch + L.mod_frame0 + (int)frame] * r.depth;
          VoiceEvent e; e.frame = frame; e.kind = EV_SET_TARGET; e.param = (uint16_t)r.param; e.aux = 0;
          e.value = r.mode == 0 ? (clampf(m, -1.0f, 1.0f) + 1.0f) * 0.5f : (r.mode == 1 ? m * 100.0f : clampf(m, 0.0f, 1.0f));
          V::slow_event(st, e, L.tt, L.rc);
        }
        tile[lane * 33 + j] = V::tick(st, L.tt, L.rc);
      }
    }
    __syncwarp();
    store_tile_voice_major(tile, L.out, L.stride, L.row0 + warp_v0, L.rows ? L.rows + warp_v0 : nullptr, row_mask, f0, nf, lane);
    __syncwarp();
  }
  if (mine) store_words(st, L.state, sv, L.n_pad, 0);
}

// ------------------------------------------------------------------------------------------- A: plan ----
template <class V>
__global__ void __launch_bounds__(64) plan_kernel(const VoiceLaunch L) {
  using Ctl = typename V::Ctl; using Span = typename V::Span;
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= L.n) return;
  const int sv = L.slots ? (int)L.slots[v] : v;
  Ctl c;
  load_words(c, L.state, sv, L.n_pad, 0);
  Span* sp = reinterpret_cast<Span*>(L.spans) + L.span_off[v];
  uint32_t e = L.ev_begin[v];
  const uint32_t ee = L.ev_begin[v + 1];
  uint32_t ns = 0;
  bool fast = V::settled(c);
  if (L.routes && L.route_begin[v + 1] > L.route_begin[v]) fast = false;     // an LFO writes a new target every frame: per-sample path
  int j = 0;
  while (fast && j < L.frames) {
    uint32_t resets = 0;
    while (e < ee && L.events[e].frame <= (uint32_t)j) { V::event(c, L.events[e], L.tt, resets); e++; }
    if (!V::settled(c)) { fast = false; break; }
    int jn = L.frames;
    if (e < ee && L.events[e].frame < (uint32_t)jn) jn = (int)L.events[e].frame;
    V::plan(c, resets, L.tt, j, jn, sp[ns]);
    ns++;
    j = jn;
  }
  L.mode[v] = fast ? 0 : 1;
  L.n_spans[v] = fast ? ns : 0;
  L.span_cursor[v] = 0xffffffffu;
  if (fast) store_words(c, L.state, sv, L.n_pad, 0);
}

// ------------------------------------------------------------------------------------------- B: front ----
template <class V, int BLOCK>
__global__ void __launch_bounds__(BLOCK) front_kernel(const VoiceLaunch L, const int blocks_per_voice) {
  using Span = typename V::Span;
  const int v = blockIdx.x / blocks_per_voice;
  if (L.mode[v]) return;
  const int jc = (blockIdx.x - v * blocks_per_voice) * BLOCK + threadIdx.x;   // frame within the chunk
  const int j = L.chunk0 + jc;
  if (jc >= L.chunk_frames || j >= L.frames) return;
  const Span* spans = reinterpret_cast<const Span*>(L.spans) + L.span_off[v];
  int lo = 0, hi = (int)L.n_spans[v] - 1;
  while (lo < hi) { int mid = (lo + hi + 1) >> 1; if (spans[mid].j0 <= j) lo = mid; else hi = mid - 1; }
  const Span& sp = spans[lo];
  if (j >= V::front_end(sp)) return;
  float o[V::NPL];
  const uint32_t k = sp.kbase + (uint32_t)j;
  V::front(sp, L.tt[k], k, L.rc.sr, o);
  float* dst = L.planes + (size_t)v * L.pitch + jc;
#pragma unroll
  for (int p = 0; p < V::NPL; p++) dst[(size_t)p * L.plane_stride] = o[p];
}

// ------------------------------------------------------------------------------------------- C: back ----
template <class V, int BLOCK>
__global__ void __launch_bounds__(BLOCK) back_kernel(const VoiceLaunch L) {
  using Span = typename V::Span; using Aud = typename V::Aud;
  constexpr int WC = sizeof(typename V::Ctl) / 4;
  __shared__ float tiles[BLOCK / 32][V::NPL + 1][TILE * 33];
  const int v = blockIdx.x * BLOCK + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warp_v0 = v - lane;
  if (warp_v0 >= L.n) return;
  const bool mine = v < L.n && L.mode[v] == 0;
  const uint32_t row_mask = __ballot_sync(0xffffffffu, mine);
  if (row_mask == 0) return;
  const int n_rows = min(32, L.n - warp_v0);
  Aud a;
  typename V::Run run;
  const Span* spans = nullptr;
  uint32_t cur = 0xffffffffu, ns = 0;
  int next_j0 = 0x7fffffff;
  int sv = v;
  if (mine) {
    if (L.slots) sv = (int)L.slots[v];
    load_words(a, L.state, sv, L.n_pad, WC);
    spans = reinterpret_cast<const Span*>(L.spans) + L.span_off[v];
    ns = L.n_spans[v];
    cur = L.span_cursor[v];
    if (cur != 0xffffffffu) V::span_resume(spans[cur], run);
    const uint32_t nx = cur + 1u;   // 0 when no span has begun yet
    next_j0 = nx < ns ? spans[nx].j0 : 0x7fffffff;
  }
  float (*tl)[TILE * 33] = tiles[warp];
  float* tout = tl[V::NPL];
  const int cend = min(L.chunk_frames, L.frames - L.chunk0);
  for (int f0 = 0; f0 < cend; f0 += TILE) {
    const int nf = min(TILE, cend - f0);
    // does any voice of the warp read planes in this tile?  (first frame of the tile decides for kick/snare; hat and
    // tom can only switch ON at a span start, which forces a load as well)
    bool want = false;
    if (mine) want = V::wants_planes(a, run, L.chunk0 + f0) || next_j0 < L.chunk0 + f0 + nf;
    if (__any_sync(0xffffffffu, want)) {
#pragma unroll
      for (int p = 0; p < V::NPL; p++) load_tile_rows(tl[p], L.planes + (size_t)p * L.plane_stride, L.pitch, warp_v0, n_rows, f0, lane);
    }
    __syncwarp();
    if (mine) {
      for (int jj = 0; jj < nf; jj++) {
        const int j = L.chunk0 + f0 + jj;
        while (j == next_j0) {
          cur += 1u;
          V::span_begin(a, spans[cur], run, L.rc.sr);
          next_j0 = cur + 1u < ns ? spans[cur + 1u].j0 : 0x7fffffff;
        }
        float p[V::NPL];
#pragma unroll
        for (int q = 0; q < V::NPL; q++) p[q] = tl[q][lane * 33 + jj];
        tout[lane * 33 + jj] = V::back(a, run, j, p, L.rc);
      }
    }
    __syncwarp();
    store_tile_voice_major(tout, L.out, L.stride, L.row0 + warp_v0, L.rows ? L.rows + warp_v0 : nullptr, row_mask, L.chunk0 + f0, nf, lane);
    __syncwarp();
  }
  if (mine) {
    store_words(a, L.state, sv, L.n_pad, WC);
    L.span_cursor[v] = cur;
  }
}

#ifndef GOOEY_OWN_KERNELS_TU   // rs_chain.cu and poly_wave.cu compile only their own kernels
// The LFO pool of a batch (engine/lfo.rs:170-185): one thread per (engine, enabled LFO) walks the call's frames —
// value = sin(phase * 2 * pi); phase += inc, wrapped at 1; out = offset + value * amount — and leaves the final phase.
__global__ void __launch_bounds__(64) lfo_kernel(LfoStream* __restrict__ streams, int n, float* __restrict__ planes, long long pitch, int frames) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  LfoStream s = streams[i];
  float* out = s.plane >= 0 ? planes + (long long)s.plane * pitch : nullptr;
  for (int f = 0; f < frames; f++) {
    const float value = gm::g_sinf(s.phase * 2.0f * PI_F);
    s.phase += s.inc;
    if (s.phase >= 1.0f) s.phase -= 1.0f;
    if (out) out[f] = s.offset + (value * s.amount);
  }
  streams[i].phase = s.phase;
}
#endif

}  // namespace gd
