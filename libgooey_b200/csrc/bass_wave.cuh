// bass_wave.cuh — the bass voice, one warp per voice, lane = frame (reference: src/instruments/bass.rs:793-877).
//
// A bass tick is three f64 phase accumulators -> f64 sine + two polyBLEP saw/square pairs -> optional oversampled
// waveshaper -> TPT low-pass whose cutoff follows the filter envelope (coefficients recomputed, through a change
// threshold, while the envelope moves) -> amp envelope.  Per 32-frame block the warp
//   * replays the phase accumulators and the state-variable filter in the reference's order (cheap recurrences),
//   * evaluates everything else one frame per lane: sines, polyBLEPs, both envelopes (from lane-local copies whose
//     latches are advanced analytically, dsp.cuh env_advance), tan() of the filter coefficients, the waveshaper through
//     the half-band scans of wave.cuh.
// Blocks are cut at event frames and at the frame where the amp envelope ends.  Whenever a parameter is still gliding
// (the smoothers then change the tick's inputs every sample) or the voice is idle, lane 0 simply runs the per-sample
// path (voices2.cuh bass_tick) for the block, so the two paths share one state and alternate freely.
#pragma once
#include "wave.cuh"

namespace gd {

constexpr int BASS_WORDS = sizeof(BassState) / 4;

// Warp-cooperative form of env_advance (dsp.cuh) over the block's frames [0, nl): every lane tests the (monotone) latch
// predicates at ITS frame and a ballot finds the first frame, instead of one binary search over the clock table per lane and
// envelope (ncu r2_b: those searches were 14 % of the kernel's instructions and a third of its stall samples).
struct EnvBlk { int j1, j2; double rel_start; };   // j1: frame at whose tick the release began, j2: frame at whose tick the envelope ended (J_NONE: not in this block)
__device__ __forceinline__ EnvBlk env_block(const Env& e, double now_l, int nl, int lane) {
  EnvBlk b; b.j1 = J_NONE; b.j2 = J_NONE; b.rel_start = e.rel_start;
  if (!(e.flags & 1)) return b;
  int start = 0;
  if (!(e.flags & 2)) {
    if (e.sustain != 0.0f) return b;
    const EnvPastDecay p{&e, e.attack + e.decay};
    const unsigned m = __ballot_sync(0xffffffffu, lane < nl && p(now_l));
    if (!m) return b;
    b.j1 = __ffs(m) - 1;
    b.rel_start = __shfl_sync(0xffffffffu, now_l, b.j1);
    start = b.j1 + 1;
  }
  const float r = (float)(now_l - b.rel_start);
  const unsigned m2 = __ballot_sync(0xffffffffu, lane < nl && lane >= start && !(r < e.release));
  if (m2) b.j2 = __ffs(m2) - 1;
  return b;
}
// the envelope as ticking frames [0, n) of the block leaves it (== env_advance(e, tt, k0, 0, n))
__device__ __forceinline__ Env env_after(const Env& e, const EnvBlk& b, int n) {
  Env x = e;
  if (b.j1 != J_NONE && b.j1 < n) { x.flags |= 2u; x.rel_start = b.rel_start; }
  if (b.j2 != J_NONE && b.j2 < n) x.flags &= ~1u;
  return x;
}

template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) bass_wave_kernel(const VoiceLaunch L) {
  __shared__ wave::GeoTables T;
  __shared__ BassState states[WARPS];
  __shared__ float stashes[WARPS][6][32];
  __shared__ double phase_stash[WARPS][3][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  wave::geo_tables_init(T, L.rc, threadIdx.x, WARPS * 32);
  __syncthreads();
  const int v = blockIdx.x * WARPS + warp;
  if (v >= L.n) return;
  const int sv = L.slots ? (int)L.slots[v] : v;
  BassState& s = states[warp];
  float (*st)[32] = stashes[warp];
  double (*pst)[32] = phase_stash[warp];
  {
    uint32_t* w = reinterpret_cast<uint32_t*>(&s);
    for (int i = lane; i < BASS_WORDS; i += 32) w[i] = L.state[(size_t)i * L.n_pad + sv];
  }
  __syncwarp();
  uint32_t ev = L.ev_begin[v];
  const uint32_t ev_end = L.ev_begin[v + 1];
  const long long row = L.rows ? (long long)L.rows[v] : (long long)(L.row0 + v);
  float* out = L.out + row * L.stride;
  const RateCtx& rc = L.rc;
  const float sr = rc.sr;
  const double dt = 1.0 / (double)sr;
  // per-span constants: pure functions of the settled parameters and of the triggered frequency, recomputed after events and
  // after per-sample blocks only (they were ~10 % of the kernel when evaluated per block: three powf / exp and two tanh)
  bool stale = true;
  float freq = 0.0f, sub_level = 0.0f, osc_level = 0.0f, detune_level = 0.0f, osc_shape = 0.0f, od = 0.0f, drive = 1.0f, comp = 1.0f;
  float base_cutoff = 0.0f, fenv_amt = 0.0f, nr = 0.5f;
  double sub_inc = 0.0, det_inc = 0.0;
  int j = 0;
  while (j < L.frames) {
    // events due at frame j, then the block runs up to the next event
    if (ev < ev_end && L.events[ev].frame <= (uint32_t)j) {
      if (lane == 0) while (ev < ev_end && L.events[ev].frame <= (uint32_t)j) { bass_event(s, L.events[ev], L.tt); ev++; }
      ev = __shfl_sync(0xffffffffu, ev, 0);
      stale = true;
      __syncwarp();
    }
    const int next_ev = ev < ev_end ? (int)L.events[ev].frame : L.frames;
    bool ok = lane < B_NP ? s.cur[lane] == s.tgt[lane] : true;
    const bool settled = __all_sync(0xffffffffu, ok);
    if (settled && s.active == 0) {       // idle and nothing gliding: the tick only counts frames (bass.rs:800-803) until the next event
      const int n_idle = next_ev - j;
      for (int q = j + lane; q < next_ev; q += 32) out[q] = 0.0f;
      __syncwarp();
      if (lane == 0) s.k += (uint32_t)n_idle;
      __syncwarp();
      j = next_ev;
      continue;
    }
    int end = min(min(j + 32, L.frames), next_ev);
    int nl = end - j;
    bool parallel = settled;
    const uint32_t k0 = s.k;
    float y = 0.0f;
    // ---- parallel block ----
    if (parallel) {
      if (stale) {
        freq = s.trig_freq * tuning_to_multiplier(s.cur[B_TUNING]);
        sub_level = s.cur[B_SUB]; osc_level = s.cur[B_OSC]; detune_level = s.cur[B_DETUNE_LEVEL];
        const float detune_cents = denorm(s.cur[B_DETUNE_AMT], 0.0f, 30.0f);
        osc_shape = s.cur[B_SHAPE];
        const float detune_ratio = gm::g_powf(2.0f, detune_cents / 1200.0f);
        const float detune_freq = freq * detune_ratio;
        sub_inc = (double)freq * dt; det_inc = (double)detune_freq * dt;
        od = s.cur[B_OVERDRIVE];
        drive = clampf(1.0f + od * 9.0f, 1.0f, 10.0f);
        comp = gm::g_tanhf(0.5f) / gm::g_tanhf(0.5f * drive);
        base_cutoff = exp_denorm(s.cur[B_CUTOFF], 20.0f, 18000.0f);
        fenv_amt = s.cur[B_FENV_AMT];
        nr = fmaxf(denorm(s.cur[B_RES], 0.5f, 15.0f), 0.5f);
        stale = false;
      }
      // the frame whose tick ends the amp envelope cuts the block
      const double now_l = L.tt[k0 + (uint32_t)min(lane, nl - 1)];
      const EnvBlk ab = env_block(s.amp_env, now_l, nl, lane);
      if (ab.j2 != J_NONE) nl = ab.j2 + 1;
      const int last = nl - 1;
      const EnvBlk fb = env_block(s.flt_env, now_l, nl, lane);
      // f64 phase accumulators: lanes 0 / 1 / 2 replay sub / osc / detune in the reference's order (bass.rs:820-828: advance, then read)
      const double osc_inc = sub_inc;
      {
        double ph = lane == 0 ? s.sub_phase : (lane == 1 ? s.osc_phase : s.detune_phase);
        const double inc = lane == 0 ? sub_inc : (lane == 1 ? osc_inc : det_inc);
        const int pl = min(lane, 2);
#pragma unroll 4
        for (int n = 0; n < nl; n++) {
          ph += inc; ph -= floor(ph);
          if (lane < 3) pst[pl][n] = ph;
        }
      }
      __syncwarp();
      const double my_sp = pst[0][min(lane, last)], my_op = pst[1][min(lane, last)], my_dp = pst[2][min(lane, last)];
      const double sp = pst[0][last], op = pst[1][last], dp = pst[2][last];
      const float sub_out = (float)sin(my_sp * 6.283185307179586476925286766559);
      const float saw_m = polyblep_saw(my_op, osc_inc), sq_m = polyblep_square(my_op, osc_inc);
      const float osc_out = saw_m * (1.0f - osc_shape) + sq_m * osc_shape;
      const float saw_d = polyblep_saw(my_dp, det_inc), sq_d = polyblep_square(my_dp, det_inc);
      const float det_out = saw_d * (1.0f - osc_shape) + sq_d * osc_shape;
      const float mix = sub_out * sub_level + osc_out * osc_level + det_out * detune_level;
      const bool shaping = od > 0.001f && !(s.ws.mix <= 0.0001f || drive <= 1.0f);
      const bool finite = __all_sync(0xffffffffu, lane >= nl || isfinite(mix));
      if (od > 0.001f && !finite) parallel = false;     // Waveshaper resets on a non-finite input: per-sample order (nothing was written yet)
      else {
        float sat = mix;
        Oversamp os = s.ws.os;
        if (shaping) {
          const float wmix = s.ws.mix, d_ = drive, c_ = comp;
          const float shaped = wave::os_scan(os, mix, [d_, c_](float x) { return wave::w_tanh(x * d_) * c_; }, T, lane, last);
          sat = mix * (1.0f - wmix) + shaped * wmix;
        }
        // envelopes: lane-local copies as the frames before mine leave them
        const Env fe = env_after(s.flt_env, fb, lane), ae = env_after(s.amp_env, ab, lane);
        const float fenv = env_value(fe, now_l);
        const float amp_env = env_value(ae, now_l);
        const float env_offset = (18000.0f - base_cutoff) * fenv_amt * fenv;
        const float cutoff = clampf(base_cutoff + env_offset, 20.0f, 18000.0f);
        // filter coefficients this frame would get if the change threshold lets them through (state_variable_tpt.rs:83-92)
        Tpt spec;
        spec.cutoff = clampf(cutoff, 20.0f, sr * 0.45f);
        spec.res = nr;
        spec.ic1 = spec.ic2 = 0.0f;
        tpt_update(spec, sr);
        __syncwarp();
        st[0][lane] = spec.cutoff; st[4][lane] = sat;
        __syncwarp();
        Tpt f = s.filter;
        // the change threshold is a sample-and-hold through f.cutoff alone (f.res == nr after the first update): replayed as its own
        // short chain, leaving the block's update mask
        unsigned mask = 0u;
        {
          float fc = f.cutoff;
          bool res_ok = !(fabsf(nr - f.res) > 0.001f);
#pragma unroll 4
          for (int n = 0; n < nl; n++) {
            const float nc = st[0][n];
            const bool upd = fabsf(nc - fc) > 0.001f || !res_ok;
            fc = upd ? nc : fc; res_ok = res_ok || upd;
            mask |= upd ? (1u << n) : 0u;
          }
          f.cutoff = fc;
        }
        // coefficient set in effect at this lane's frame: that of the latest update frame <= lane, else the carried one
        float g_l = f.g, h_l = f.h;
        if (mask) {
          const unsigned m = mask & ((2u << lane) - 1u);
          const int src = m ? 31 - __clz(m) : 0;
          const float sg = __shfl_sync(0xffffffffu, spec.g, src), sh = __shfl_sync(0xffffffffu, spec.h, src);
          if (m) { g_l = sg; h_l = sh; }
          const int lu = 31 - __clz(mask);                       // the block's last update leaves its coefficients in the state
          f.res = nr; f.g = __shfl_sync(0xffffffffu, spec.g, lu); f.r = __shfl_sync(0xffffffffu, spec.r, lu); f.h = __shfl_sync(0xffffffffu, spec.h, lu);
        }
        __syncwarp();
        st[1][lane] = g_l; st[3][lane] = h_l;
        __syncwarp();
        float lo_l = 0.0f;
        {
          float ic1 = f.ic1, ic2 = f.ic2;
#pragma unroll 4
          for (int n = 0; n < nl; n++) {        // tpt_process (dsp.cuh) with the frame's coefficients; only the low-pass output is used
            const float g = st[1][n], h = st[3][n], in = st[4][n];
            const float v1 = (g * (in - ic2) + ic1) * h;
            const float v2 = ic2 + g * v1;
            ic1 = 2.0f * v1 - ic1;
            ic2 = 2.0f * v2 - ic2;
            if (n == lane) lo_l = v2;
          }
          f.ic1 = ic1; f.ic2 = ic2;
        }
        y = lo_l * amp_env * sqrtf(s.velocity) * s.cur[B_VOLUME];
        __syncwarp();
        if (lane == 0) {                  // commit the block
          s.sub_phase = sp; s.osc_phase = op; s.detune_phase = dp;
          s.filter = f;
          s.ws.drive = drive;
          if (shaping) s.ws.os = os;
          const Env fe2 = env_after(s.flt_env, fb, nl), ae2 = env_after(s.amp_env, ab, nl);
          s.flt_env = fe2; s.amp_env = ae2;
          if (!env_active(ae2)) s.active = 0;
          s.k = k0 + (uint32_t)nl;
        }
        __syncwarp();
      }
    }
    const int last = nl - 1;
    // ---- per-sample path for this block (gliding parameters, idle voice, non-finite waveshaper input) ----
    if (!parallel) {
      if (lane == 0) for (int n = 0; n < nl; n++) st[5][n] = bass_tick(s, L.tt, rc);
      stale = true;
      __syncwarp();
      y = st[5][min(lane, last)];
      __syncwarp();
    }
    if (lane < nl) out[j + lane] = y;
    j += nl;
  }
  __syncwarp();
  {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(&s);
    for (int i = lane; i < BASS_WORDS; i += 32) L.state[(size_t)i * L.n_pad + sv] = w[i];
  }
}

}  // namespace gd
