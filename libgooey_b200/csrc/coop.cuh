// coop.cuh — kernel K: the CTA-cooperative back end of the drum voices.
//
// wave.cuh gives one voice to one warp (lane = frame) and REPLAYS every exact-order recurrence (f32 phase accumulators,
// RNGs, direct-form-I biquads with thresholded coefficient pick-up, envelope followers ...) on all 32 lanes of that warp:
// each replayed frame costs the warp one issue slot per instruction although only one lane's worth of work is done.
// ncu (profiles/r1_o): 75 % of the tom back end's warp-instructions are such replays, 2 670 thread-instructions per
// voice-frame against ~600 algorithmic, 8 one-warp CTAs per SM at 242 registers, issue_active 0.38.
//
// Here a CTA owns NV voices.  A voice's timeline still advances in blocks of up to 32 frames, but a block is processed in
// PHASES separated by CTA barriers, and the two kinds of work are laid out differently:
//   * P phases (memoryless per-frame work and the LTI sections evaluated as Kogge-Stone scans): warp w owns voice w,
//     lane = frame — exactly the arithmetic of wave.cuh, whose scan helpers are reused;
//   * S phases (exact-order recurrences): ONE warp runs the loop over the block's frames with lane = VOICE, reading the
//     per-frame inputs the P phase left in shared memory (stash[slot][voice][frame], pitch 33 -> conflict free both ways)
//     and writing per-frame results back.  The replay of NV voices costs what the replay of one voice cost before, and
//     the five membrane resonators of the tom run as (filter, voice) pairs on lanes.
// The audio state of the CTA's voices lives in shared memory (one Aud struct per voice, loaded from / stored to the pool
// once per launch), so a P warp and the S lanes see the same state without replication in registers: the kernel fits 2-3
// CTAs per SM, and the serial phases of one CTA overlap the parallel phases of its neighbours.
// Blocks are NOT aligned between the voices of a CTA: every voice takes its next block (shortened at span boundaries and
// at deactivation) each round; a voice without work just attends the barriers.
//
// Exactness: the S phases execute the reference's operations in the reference's order (same as the replays they
// replace); the P phases are the scans / memoryless stages of wave.cuh unchanged.  tests/test_backend_choice_gpu.py
// renders enough toms for this back end to be chosen and compares it with the per-sample-order back end
// (GOOEY_B200_BACKEND=serial) and with the oracle.
#pragma once
#include <climits>
#include <type_traits>
#include "wave.cuh"

namespace gd { namespace coop {
using namespace gd::wave;     // warp-wide scan helpers: scan1 / ap_sec / hb_run / os_scan / lin2_scan / biquad_scan / tpt_scan ...

constexpr unsigned FULL = 0xffffffffu;
constexpr int SP = 33;        // stash row pitch (floats)
enum { M_IDLE = 0, M_NORMAL = 1, M_TAIL = 2, M_GENERIC = 3, M_SERIAL = 4 };
enum { F_NORMAL = 1u << M_NORMAL, F_TAIL = 1u << M_TAIL, F_GENERIC = 1u << M_GENERIC, F_SERIAL = 1u << M_SERIAL, F_MEMBRANE = 1u << 8 };
struct RoundInfo { int j, nl, nv, mode; };
struct Empty {};

template <class C, int NV> struct Smem {
  typename std::conditional<C::GEO, GeoTables, Empty>::type T;
  typename C::V::Aud aud[NV];
  typename C::V::Run run[NV];
  typename C::Span2 w2[NV];
  RoundInfo ri[NV];
  unsigned wflags[2][NV];      // per round parity, per voice: mode bits of the voice's block
  Lin2 lin[C::NLIN > 0 ? NV : 1][C::NLIN > 0 ? C::NLIN : 1];
  float st[C::NST][NV][SP];
};

// max over the warp of an int (uniform loop bounds of the S phases)
__device__ __forceinline__ int warp_max(int x) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) x = max(x, __shfl_xor_sync(FULL, x, d));
  return x;
}

// ---- tom -------------------------------------------------------------------------------------------------------------
// Phases of a round (tom2.rs:450-585 split by what depends on history):
//   A  (P) envelope / pitch per frame, attack + completion ballots, mode of the block, click table, phase increments
//   S1 (S) the three phase accumulators + rand~ sample-and-hold (morph_osc.rs:137-202) and the band-pass's coefficient
//          change detector (biquad_bandpass.rs:73-87: a chain through last_freq only) -> update mask of the block;
//          GENERIC voices: the reference's whole tick per sample
//   B  (P) sines / triangles / morph mix; band-pass coefficient sets at the frames that update (biquad_bandpass.rs:88-119),
//          every frame picks the set in effect and forms the FEED-FORWARD half of the direct-form-I section
//          (b0 x[n] + b1 x[n-1]) + b2 x[n-2] — inputs only, same operation order as the reference
//   S2 (S) the FEEDBACK half: out = (ffwd - a1 y1) - a2 y2 — the only part that is a recurrence (4 flops per frame)
//   C  (P) membrane input filtered * env and the feed-forward halves of the five membrane resonators
//   S3 (S) their feedback halves, lanes = (filter, voice) (membrane_resonator.rs:189-200)
//   D  (P) sum of the five, tanh, ring-level input
//   S4 (S) ring level; in the ringing TAIL also the deactivation test (tom2.rs:488-493)
// TAIL = main oscillator done (envelope complete), membrane still ringing: only C / S3 / D / S4 run.  Everything else the
// reference keeps ticking there (phases, click, band-pass memory) is reset by the next trigger before it can be observed;
// the band-pass coefficient memory, which survives a trigger, is brought to where the per-sample bp_set calls would leave it.
struct TomC {
  using V = TomV;
  struct Span2 { int dummy; };
  static constexpr bool GEO = false;
  static constexpr int NLIN = 0;
  static constexpr int NST = 12;
  enum { ST_INC = 0, ST_FFWD = 0, ST_RND = 1, ST_A1 = 1, ST_FF = 2, ST_A2 = 2, ST_TP = 3, ST_FILT = 3, ST_FSP = 4, ST_RIN = 4, ST_RV = 5, ST_Y0 = 5,
         ST_ENV = 10, ST_NOISE = 11, ST_RLEV = 11 };
  static constexpr int MIN_CTAS = 2;     // resident 16-voice CTAs per SM the register allocation must allow
  static __device__ __forceinline__ int active_end(const TomV::Run&) { return 0x7fffffff; }
  template <class SM> static __device__ __forceinline__ void span_setup(SM&, int, int, const RateCtx&) {}

  template <int NV, class SM>
  static __device__ __forceinline__ void round(SM& S, const int warp, const int lane, const bool work, const float* p, const int j, int& nout, float& y,
                                               const RateCtx& rc, const unsigned rnd_idx) {
    TomAud& a = S.aud[warp];
    const TomV::Run& r = S.run[warp];
    const TomDer& d = r.d;
    const float sr = rc.sr;
    float (*st)[NV][SP] = S.st;
    const int nl = nout;
    int mode = M_IDLE, nv = 0;
    float env_l = 0.0f, noise_l = 0.0f, fade = 1.0f, mf_l = 40.0f, click = 0.0f;
    const unsigned le = (2u << lane) - 1u;     // lanes 0..lane
    // ------------------------------------------------------------------------------------------------ phase A
    if (work) {
      env_l = (j + lane) < r.j_env ? p[0] : r.env_final;
      noise_l = p[1];
      const float rnd_l = p[2];
      const bool complete_l = (j + lane) >= r.j_env;
      const unsigned valid = nl >= 32 ? FULL : ((1u << nl) - 1u);
      const float eb = env_l * d.bend_scaled;
      const float raw_freq = d.base_frequency * (1.0f + eb * eb);
      const unsigned m_att = __ballot_sync(FULL, env_l > 0.9f) & valid;
      const bool past0 = a.past_attack != 0u, done0 = a.main_done != 0u;
      const float ring0 = a.ring_level;
      const bool merged = a.tri_phase == a.main_sine_phase && a.tri_phase == a.mtri_phase && a.tri_phase == a.gated_sine_phase;
      const uint32_t cp = a.click_pos; const bool playing = a.click_playing != 0u;
      const bool past_l = past0 || (m_att & le) != 0u;
      const unsigned m_done = __ballot_sync(FULL, complete_l || (past_l && raw_freq < 20.0f)) & valid;
      const int first_done = done0 ? 0 : (m_done ? __ffs(m_done) - 1 : 32);
      __syncwarp();                                // every lane has read the voice's flags
      if (first_done == 0) {
        if (d.membrane > 0.0f && j >= r.j_env) {   // ringing tail (or about to die: S4 decides frame by frame)
          mode = M_TAIL; nv = nl;
          if (lane == 0) {
            a.main_done = 1;
            const float eb0 = r.env_final * d.bend_scaled;
            const float ff = fmaxf(fmaxf(d.base_frequency * (1.0f + eb0 * eb0), 40.0f), 20.0f);
            bp_set(a.bp, sr, ff, d.fq, 1.1f);      // where the per-sample bp_set calls of the tail leave the coefficient memory
          }
        } else if (!(d.membrane > 0.0f) && !(ring0 > 0.0001f)) {   // no tail: the voice ends at this frame (tom2.rs:488-493)
          mode = M_IDLE; nv = 0;
          if (lane == 0) { a.main_done = 1; a.active = 0; if (m_att & 1u) a.past_attack = 1; }
        } else { mode = M_GENERIC; nv = nl; }
      } else if (!merged) { mode = M_GENERIC; nv = nl; }
      else {
        mode = M_NORMAL; nv = first_done < nl ? first_done : nl;
        fade = (past_l && raw_freq < 40.0f) ? (raw_freq - 20.0f) / (40.0f - 20.0f) : 1.0f;
        mf_l = fmaxf(raw_freq, 40.0f);
        if (playing) { const uint32_t idx = cp + (uint32_t)lane; if (idx < 64u) click = c_tom_impulse[idx]; }
        if (lane == 0) {
          if ((m_att & (nv >= 32 ? FULL : ((1u << nv) - 1u))) != 0u) a.past_attack = 1;
          if (playing) { const uint32_t c2 = min(64u, cp + (uint32_t)nv); a.click_pos = c2; if (c2 >= 64u) a.click_playing = 0; }
        }
        st[ST_INC][warp][lane] = mf_l / sr;
        st[ST_FF][warp][lane] = fmaxf(mf_l, 20.0f);
      }
      if (mode == M_NORMAL || mode == M_GENERIC) st[ST_RND][warp][lane] = rnd_l;
      if (mode == M_GENERIC) { st[ST_ENV][warp][lane] = env_l; st[ST_NOISE][warp][lane] = noise_l; }
      if (lane == 0) {
        S.ri[warp].nv = nv; S.ri[warp].mode = mode;
      }
    }
    if (lane == 0) S.wflags[rnd_idx & 1u][warp] = mode == M_IDLE ? 0u : ((1u << mode) | ((d.membrane > 0.0f && mode != M_GENERIC) ? F_MEMBRANE : 0u));
    __syncthreads();                                                                                   // b1
    const unsigned fl = __reduce_or_sync(FULL, lane < NV ? S.wflags[rnd_idx & 1u][lane] : 0u);
    // ------------------------------------------------------------------------------------------------ phase S1
    if (fl & (F_NORMAL | F_GENERIC)) {
      if (warp == 0 && (fl & F_NORMAL)) {
        const int vv = lane < NV ? lane : 0;
        const bool on = lane < NV && S.ri[vv].mode == M_NORMAL;
        const int n_v = on ? S.ri[vv].nv : 0;
        TomAud& b = S.aud[vv];
        float ph = b.tri_phase, fx = b.fixed_sine_phase, rph = b.rand_phase, rcu = b.rand_current, rtg = b.rand_target;
        const float inc_fixed = 190.0f / sr, inc_rand = S.run[vv].d.rand_freq / sr;
        const float fq = S.run[vv].d.fq;
        float lf = b.bp.last_freq;
        bool qg_ok = fabsf(fq - b.bp.last_q) < 0.001f && fabsf(1.1f - b.bp.last_gain) < 0.001f;   // an update makes both terms true
        unsigned mask = 0u;
        const int nmax = warp_max(n_v);
        // Register-blocked: the block's inputs are loaded eight frames at a time before the dependent arithmetic starts, so
        // the shared-memory latency is paid once per eight frames instead of once per frame (the compiler cannot hoist the
        // loads itself: it has to assume the loop's stores alias them).
        const float* r_inc = &st[ST_INC][vv][0]; const float* r_rnd = &st[ST_RND][vv][0]; const float* r_ff = &st[ST_FF][vv][0];
        float* w_tp = &st[ST_TP][vv][0]; float* w_fsp = &st[ST_FSP][vv][0]; float* w_rv = &st[ST_RV][vv][0];
        for (int n0 = 0; n0 < nmax; n0 += 8) {
          float inc[8], rnd[8], ffn[8];
#pragma unroll
          for (int k = 0; k < 8; k++) { inc[k] = r_inc[n0 + k]; rnd[k] = r_rnd[n0 + k]; ffn[k] = r_ff[n0 + k]; }
#pragma unroll
          for (int k = 0; k < 8; k++) {
            if (n0 + k < n_v) {
              w_tp[n0 + k] = ph; w_fsp[n0 + k] = fx;
              ph += inc[k]; if (ph >= 1.0f) ph -= 1.0f;
              fx += inc_fixed; if (fx >= 1.0f) fx -= 1.0f;
              const float prev = rph;
              rph += inc_rand; if (rph >= 1.0f) rph -= 1.0f;
              const bool wrap = rph < prev;
              rcu = wrap ? rtg : rcu; rtg = wrap ? rnd[k] : rtg;
              w_rv[n0 + k] = rcu + (rtg - rcu) * rph;          // rand_value (morph_osc.rs: memoryless given the state)
              const bool upd = !(fabsf(ffn[k] - lf) < 0.01f && qg_ok);   // !bp_unchanged
              lf = upd ? ffn[k] : lf; qg_ok = qg_ok || upd;
              mask |= upd ? (1u << (n0 + k)) : 0u;
            }
          }
        }
        if (on) {
          b.tri_phase = b.main_sine_phase = b.mtri_phase = b.gated_sine_phase = ph;
          b.fixed_sine_phase = fx; b.rand_phase = rph; b.rand_current = rcu; b.rand_target = rtg;
          b.bp.last_freq = lf;
          if (mask) { b.bp.last_q = fq; b.bp.last_gain = 1.1f; }
          S.ri[vv].nl = (int)mask;                                 // (nl is not read again this round: carries the update mask to phase B)
        }
      }
      if (warp == (NV > 1 ? 1 : 0) && (fl & F_GENERIC)) {        // the reference's whole tick per sample, lane = voice
        const int vv = lane < NV ? lane : 0;
        if (lane < NV && S.ri[vv].mode == M_GENERIC) {
          TomAud& b = S.aud[vv];
          const TomV::Run& rr = S.run[vv];
          const int jv = S.ri[vv].j, n_v = S.ri[vv].nv;
          int got = n_v;
          for (int n = 0; n < n_v; n++) {
            TomFront f; f.env = st[ST_ENV][vv][n]; f.noise = st[ST_NOISE][vv][n]; f.rnd = st[ST_RND][vv][n];
            const float yy = tom_back(b, rr.d, f, (jv + n) >= rr.j_env, rc);
            st[ST_TP][vv][n] = yy;
            if (!b.active) { got = n + 1; break; }
          }
          S.ri[vv].nv = got;
        }
      }
      __syncthreads();                                                                                 // b2
    }
    // ------------------------------------------------------------------------------------------------ phases B, S2
    float filtered = 0.0f;
    if (fl & F_NORMAL) {
      if (mode == M_NORMAL) {
        const float tp = st[ST_TP][warp][lane], fsp = st[ST_FSP][warp][lane], rand_value = st[ST_RV][warp][lane];
        const float ffl = st[ST_FF][warp][lane];
        const unsigned mask = (unsigned)S.ri[warp].nl;
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
        // coefficient set in effect at this frame: the set computed at the latest update frame <= lane, else the carried one
        float b0 = a.bp.b0, b1 = a.bp.b1, b2 = a.bp.b2, a1 = a.bp.a1, a2 = a.bp.a2;
        const float x1c = a.bp.x1, x2c = a.bp.x2;
        if (mask) {
          Biquad spec;
          bp_compute(spec, sr, ffl, d.fq, 1.1f);
          const unsigned m = mask & le;
          const int src = m ? 31 - __clz(m) : 0;
          const float sb0 = __shfl_sync(FULL, spec.b0, src), sb1 = __shfl_sync(FULL, spec.b1, src), sb2 = __shfl_sync(FULL, spec.b2, src);
          const float sa1 = __shfl_sync(FULL, spec.a1, src), sa2 = __shfl_sync(FULL, spec.a2, src);
          if (m) { b0 = sb0; b1 = sb1; b2 = sb2; a1 = sa1; a2 = sa2; }
        }
        float xm1 = __shfl_up_sync(FULL, x, 1), xm2 = __shfl_up_sync(FULL, x, 2);
        if (lane == 0) { xm1 = x1c; xm2 = x2c; } else if (lane == 1) xm2 = x1c;
        const float ffwd = b0 * x + b1 * xm1 + b2 * xm2;
        __syncwarp();                                // ST_TP .. ST_RV, ST_FF and the carried band-pass state have been read by every lane
        st[ST_FFWD][warp][lane] = ffwd; st[ST_A1][warp][lane] = a1; st[ST_A2][warp][lane] = a2;
        if (lane == nv - 1) { Biquad& o = a.bp; o.b0 = b0; o.b1 = b1; o.b2 = b2; o.a1 = a1; o.a2 = a2; o.x1 = x; o.x2 = xm1; }
      }
      __syncthreads();                                                                                 // b3
      if (warp == 0) {   // S2
        const int vv = lane < NV ? lane : 0;
        const bool on = lane < NV && S.ri[vv].mode == M_NORMAL;
        const int n_v = on ? S.ri[vv].nv : 0;
        float y1 = S.aud[vv].bp.y1, y2 = S.aud[vv].bp.y2;
        const int nmax = warp_max(n_v);
        const float* r_f = &st[ST_FFWD][vv][0]; const float* r_a1 = &st[ST_A1][vv][0]; const float* r_a2 = &st[ST_A2][vv][0];
        float* w_y = &st[ST_FILT][vv][0];
        for (int n0 = 0; n0 < nmax; n0 += 8) {
          float f[8], c1[8], c2[8], o[8];
#pragma unroll
          for (int k = 0; k < 8; k++) { f[k] = r_f[n0 + k]; c1[k] = r_a1[n0 + k]; c2[k] = r_a2[n0 + k]; }
#pragma unroll
          for (int k = 0; k < 8; k++) {
            o[k] = 0.0f;
            if (n0 + k < n_v) {
              const float out = f[k] - c1[k] * y1 - c2[k] * y2;
              y2 = y1; y1 = out;
              o[k] = fabsf(out) < 1e-15f ? 0.0f : out;
            }
          }
#pragma unroll
          for (int k = 0; k < 8; k++) if (n0 + k < n_v) w_y[n0 + k] = o[k];
        }
        if (on) { S.aud[vv].bp.y1 = y1; S.aud[vv].bp.y2 = y2; }
      }
      __syncthreads();                                                                                 // b4
      if (mode == M_NORMAL) filtered = st[ST_FILT][warp][lane];
    }
    // ------------------------------------------------------------------------------------------------ phases C, S3, D, S4
    float mem_out = 0.0f, rlev = 0.0f;
    if (fl & F_MEMBRANE) {
      if ((mode == M_NORMAL || mode == M_TAIL) && d.membrane > 0.0f) {   // C
        const float mi = mode == M_NORMAL ? filtered * env_l : 0.0f;
        const float u1 = __shfl_up_sync(FULL, mi, 1), u2 = __shfl_up_sync(FULL, mi, 2);
        float ffw[5], xp[5];
#pragma unroll
        for (int f = 0; f < 5; f++) {
          const Biquad& m = a.mem[f];
          const float xm1 = lane == 0 ? m.x1 : u1, xm2 = lane == 0 ? m.x2 : (lane == 1 ? m.x1 : u2);
          ffw[f] = m.b0 * mi + m.b1 * xm1 + m.b2 * xm2;
          xp[f] = xm1;
        }
        __syncwarp();                                // the carried x history has been read by lanes 0 and 1
#pragma unroll
        for (int f = 0; f < 5; f++) {
          st[ST_Y0 + f][warp][lane] = ffw[f];
          if (lane == nv - 1) { a.mem[f].x1 = mi; a.mem[f].x2 = xp[f]; }
        }
      }
      __syncthreads();                                                                                 // b5
      {   // S3: q = (filter, voice) pairs on lanes
        const int q = warp * 32 + lane;
        const int f = q / NV, vv = q - f * NV;
        if (f < 5) {
          const int m = S.ri[vv].mode;
          const bool on = (m == M_NORMAL || m == M_TAIL) && S.run[vv].d.membrane > 0.0f;
          const int n_v = on ? S.ri[vv].nv : 0;
          const Biquad& bq = S.aud[vv].mem[f];
          const float a1 = bq.a1, a2 = bq.a2;
          float y1 = bq.y1, y2 = bq.y2;
          float* row = &st[ST_Y0 + f][vv][0];
          for (int n0 = 0; n0 < n_v; n0 += 8) {
            float in[8], o[8];
#pragma unroll
            for (int k = 0; k < 8; k++) in[k] = row[n0 + k];
#pragma unroll
            for (int k = 0; k < 8; k++) {
              o[k] = 0.0f;
              if (n0 + k < n_v) {
                const float out = in[k] - a1 * y1 - a2 * y2;
                y2 = y1; y1 = out;
                o[k] = fabsf(out) < 1e-15f ? 0.0f : out;
              }
            }
#pragma unroll
            for (int k = 0; k < 8; k++) if (n0 + k < n_v) row[n0 + k] = o[k];
          }
          if (on) { Biquad& o = S.aud[vv].mem[f]; o.y1 = y1; o.y2 = y2; }
        }
      }
      __syncthreads();                                                                                 // b6
      if ((mode == M_NORMAL || mode == M_TAIL) && d.membrane > 0.0f) {   // D
        float acc = 0.0f;
#pragma unroll
        for (int i = 0; i < 5; i++) acc += st[ST_Y0 + i][warp][lane];
        mem_out = w_tanh(acc);
        st[ST_RIN][warp][lane] = fabsf(mem_out) * 0.001f;
      }
      __syncthreads();                                                                                 // b7
      if (warp == NV - 1) {   // S4
        const int vv = lane < NV ? lane : 0;
        const int m = S.ri[vv].mode;
        const bool on = lane < NV && (m == M_NORMAL || m == M_TAIL) && S.run[vv].d.membrane > 0.0f;
        const int n_v = on ? S.ri[vv].nv : 0;
        float ring = S.aud[vv].ring_level;
        if (m == M_TAIL) {
          int dead = -1;
          const float* r_in = &st[ST_RIN][vv][0]; float* w_lev = &st[ST_RLEV][vv][0];
          for (int n0 = 0; n0 < n_v && dead < 0; n0 += 8) {
            float in[8], lev[8];
#pragma unroll
            for (int k = 0; k < 8; k++) in[k] = r_in[n0 + k];
#pragma unroll
            for (int k = 0; k < 8; k++) {
              lev[k] = 0.0f;
              if (n0 + k < n_v && dead < 0) {
                if (!(ring > 0.0001f)) dead = n0 + k;            // tom2.rs:488-493, tested before the frame's membrane tick
                else { ring = ring * 0.999f + in[k]; lev[k] = ring; }
              }
            }
#pragma unroll
            for (int k = 0; k < 8; k++) if (n0 + k < n_v) w_lev[n0 + k] = lev[k];
          }
          if (on && dead >= 0) { S.ri[vv].nv = dead; S.aud[vv].active = 0; }
        } else {
          const float* r_in = &st[ST_RIN][vv][0];
          for (int n0 = 0; n0 < n_v; n0 += 8) {
            float in[8];
#pragma unroll
            for (int k = 0; k < 8; k++) in[k] = r_in[n0 + k];
#pragma unroll
            for (int k = 0; k < 8; k++) if (n0 + k < n_v) ring = ring * 0.999f + in[k];
          }
        }
        if (on) S.aud[vv].ring_level = ring;
      }
      __syncthreads();                                                                                 // b8
      if (mode == M_TAIL) rlev = st[ST_RLEV][warp][lane];
    }
    // ------------------------------------------------------------------------------------------------ output
    if (mode == M_NORMAL) {
      const float dry_gain = 1.0f - d.mm;
      const float dry = filtered * env_l;
      const float fs = dry * dry_gain + mem_out * d.mm;
      y = fs * fade * 0.7f * d.vol;
      nout = nv;        // a block that ended at the main oscillator's last frame: the next round starts in the tail (or ends the voice)
    } else if (mode == M_TAIL) {
      const float fd = rlev >= 0.005f ? 1.0f : (rlev <= 0.0001f ? 0.0f : (rlev - 0.0001f) / (0.005f - 0.0001f));
      y = mem_out * d.mm * fd * 0.7f * d.vol;
      nout = S.ri[warp].nv;
    } else if (mode == M_GENERIC) {
      y = st[ST_TP][warp][lane];
      nout = S.ri[warp].nv;
    } else nout = 0;
  }
};

// ---- the kernel --------------------------------------------------------------------------------------------------------
template <class C, int NV>
__global__ void __launch_bounds__(NV * 32, C::MIN_CTAS) coop_kernel(const VoiceLaunch L) {
  using V = typename C::V; using Span = typename V::Span; using Aud = typename V::Aud;
  constexpr int WC = sizeof(typename V::Ctl) / 4;
  constexpr int WA = sizeof(Aud) / 4;
  extern __shared__ __align__(16) unsigned char coop_smem_raw[];
  Smem<C, NV>& S = *reinterpret_cast<Smem<C, NV>*>(coop_smem_raw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if constexpr (C::GEO) geo_tables_init(S.T, L.rc, threadIdx.x, NV * 32);
  const int v = blockIdx.x * NV + warp;
  const bool alive = v < L.n && L.mode[v] == 0;
  const int sv = alive ? (L.slots ? (int)L.slots[v] : v) : 0;
  Aud& a = S.aud[warp];
  typename V::Run& run = S.run[warp];
  const Span* spans = nullptr;
  uint32_t ns = 0, cur = 0xffffffffu;
  bool ready = false;
  int next_j0 = 0x7fffffff;
  float* out = nullptr;
  const float* planes = nullptr;
  {
    uint32_t* aw = reinterpret_cast<uint32_t*>(&a);
    for (int w = lane; w < WA; w += 32) aw[w] = alive ? L.state[(size_t)(WC + w) * L.n_pad + sv] : 0u;
  }
  if (alive) {
    spans = reinterpret_cast<const Span*>(L.spans) + L.span_off[v];
    ns = L.n_spans[v];
    cur = L.span_cursor[v];
    if (cur != 0xffffffffu && lane == 0) V::span_resume(spans[cur], run);
    next_j0 = cur + 1u < ns ? spans[cur + 1u].j0 : 0x7fffffff;
    const long long row = L.rows ? (long long)L.rows[v] : (long long)(L.row0 + v);
    out = L.out + row * L.stride;
    planes = L.planes + (size_t)v * L.pitch;
  }
  if (lane == 0) S.ri[warp] = RoundInfo{0, 0, 0, M_IDLE};
  __syncthreads();
  const int c1 = L.chunk0 + min(L.chunk_frames, L.frames - L.chunk0);
  int j = L.chunk0;
  float pn[V::NPL];
  int pj = -1;
#pragma unroll
  for (int q = 0; q < V::NPL; q++) pn[q] = 0.0f;
  for (unsigned rnd_idx = 0;; rnd_idx++) {
    const bool more = alive && j < c1;
    bool work = false;
    int nl = 0;
    float p[V::NPL];
#pragma unroll
    for (int q = 0; q < V::NPL; q++) p[q] = 0.0f;
    if (more) {
      while (j == next_j0) {
        cur += 1u;
        if (lane == 0) V::span_begin(a, spans[cur], run, L.rc.sr);
        __syncwarp();
        ready = false;
        next_j0 = cur + 1u < ns ? spans[cur + 1u].j0 : 0x7fffffff;
      }
      const int span_end = min(next_j0, c1);
      const int act_end = min(span_end, C::active_end(run));
      if (cur == 0xffffffffu || !V::is_active(a, run, j) || j >= act_end) {      // silent until the next span: zero-fill
        for (int k = j + lane; k < span_end; k += 32) out[k] = 0.0f;
        j = span_end;
      } else {
        if (!ready) { __syncwarp(); C::span_setup(S, warp, lane, L.rc); __syncwarp(); ready = true; }
        nl = min(32, act_end - j);
        if (pj == j) {                              // prefetched during the previous round
#pragma unroll
          for (int q = 0; q < V::NPL; q++) { const float t = __shfl_sync(FULL, pn[q], nl - 1); p[q] = lane < nl ? pn[q] : t; }
        } else {
          const int jj = j + min(lane, nl - 1);     // lanes past the block re-read its last frame: finite, never stored
#pragma unroll
          for (int q = 0; q < V::NPL; q++) p[q] = planes[(size_t)q * L.plane_stride + (jj - L.chunk0)];
        }
        work = true;
        // planes of the block that follows if this one is not shortened: issued now, consumed next round, so the L2 latency
        // overlaps this round's phases (frames past the chunk are clamped; lanes past the next block are fixed up above)
        pj = j + nl;
        if (pj < c1) {
          const int jn = min(pj + lane, c1 - 1);
#pragma unroll
          for (int q = 0; q < V::NPL; q++) pn[q] = planes[(size_t)q * L.plane_stride + (jn - L.chunk0)];
        }
      }
    }
    __syncwarp();                                  // the previous round's readers of ri[warp] are done
    if (lane == 0) S.ri[warp] = RoundInfo{j, nl, nl, work ? M_NORMAL : M_IDLE};
    if (!__syncthreads_or(more ? 1 : 0)) break;                                                         // b0
    float y = 0.0f;
    int nout = nl;
    C::template round<NV>(S, warp, lane, work, p, j, nout, y, L.rc, rnd_idx);
    if (work) {
      if (lane < nout) out[j + lane] = y;
      j += nout;
    }
  }
  __syncthreads();
  if (alive) {
    const uint32_t* aw = reinterpret_cast<const uint32_t*>(&a);
    for (int w = lane; w < WA; w += 32) L.state[(size_t)(WC + w) * L.n_pad + sv] = aw[w];
    if (lane == 0) L.span_cursor[v] = cur;
  }
}

} }  // namespace gd::coop
