// poly_wave.cu — the poly synth, one warp per voice, lane = frame (reference: src/instruments/poly_synth.rs:437-525).
//
// A PolySynth tick walks six sub-voices; each active one is two f64 phase accumulators -> two polyBLEP saw/square pairs ->
// TPT low-pass whose cutoff follows the filter envelope (coefficients recomputed, through a change threshold, while the
// envelope moves) -> amp envelope.  That is the bass's structure six times over (bass_wave.cuh), and the block walk is the
// same.  Per block of up to 32 frames the warp
//   * replays the recurrences in the reference's order, each chain on a lane of its own: the 12 phase accumulators on
//     lanes 0-11, then each sub-voice's change-threshold chain and its filter state on lane k;
//   * evaluates everything else one frame per lane: both envelopes of every sub-voice (lane-local copies whose latches are
//     advanced by the ballots of env_block), the polyBLEPs, tan() of the coefficient updates, the sum over sub-voices.
// Blocks are cut at event frames and after the frame whose tick ends an amp envelope (that frame's tick latches the
// sub-voice inactive and leaves its phases, filter and filter envelope untouched).  While a parameter glides, or no
// sub-voice is active, lane 0 runs poly_tick for the block, so the two paths share one state and alternate freely.
// Nothing is re-associated: the output is bit-identical to slow_kernel<PolyV>.
#define GOOEY_OWN_KERNELS_TU
#include "device_rt.h"
#include "bass_wave.cuh"
#include "poly_wave.cuh"

namespace gd {

constexpr int POLY_WORDS = sizeof(PolyState) / 4;

template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) poly_wave_kernel(const VoiceLaunch L) {
  __shared__ PolyState states[WARPS];
  __shared__ double phase_stash[WARPS][12][32];     // [2k + b][n]: phase_a / phase_b of sub-voice k read by the tick of frame n
  __shared__ float stash[WARPS][5][6][32];          // filter input, cutoff, g, h, low-pass output per sub-voice and frame
  __shared__ float coef[WARPS][6][3];               // g, r, h the block's last coefficient update leaves in sub-voice k's filter
  __shared__ float ticks[WARPS][32];                // outputs of the per-sample path
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int v = blockIdx.x * WARPS + warp;
  if (v >= L.n) return;
  const int sv = L.slots ? (int)L.slots[v] : v;
  PolyState& s = states[warp];
  double (*pst)[32] = phase_stash[warp];
  float (*in_s)[32] = stash[warp][0];
  float (*nc_s)[32] = stash[warp][1];
  float (*g_s)[32] = stash[warp][2];
  float (*h_s)[32] = stash[warp][3];
  float (*lo_s)[32] = stash[warp][4];
  {
    uint32_t* w = reinterpret_cast<uint32_t*>(&s);
    for (int i = lane; i < POLY_WORDS; i += 32) w[i] = L.state[(size_t)i * L.n_pad + sv];
  }
  __syncwarp();
  uint32_t ev = L.ev_begin[v];
  const uint32_t ev_end = L.ev_begin[v + 1];
  const long long row = L.rows ? (long long)L.rows[v] : (long long)(L.row0 + v);
  float* out = L.out + row * L.stride;
  const RateCtx& rc = L.rc;
  const float sr = rc.sr;
  const double dt = 1.0 / (double)sr;
  // per-span constants: pure functions of the settled parameters, recomputed after events and after per-sample blocks
  bool stale = true;
  float osc_shape = 0.0f, volume = 0.0f, base_cutoff = 0.0f, fenv_amt = 0.0f, nr = 0.5f;
  double detune_ratio = 1.0;
  int j = 0;
  while (j < L.frames) {
    // events due at frame j, then the block runs up to the next event
    if (ev < ev_end && L.events[ev].frame <= (uint32_t)j) {
      if (lane == 0) while (ev < ev_end && L.events[ev].frame <= (uint32_t)j) { poly_event(s, L.events[ev], L.tt); ev++; }
      ev = __shfl_sync(0xffffffffu, ev, 0);
      stale = true;
      __syncwarp();
    }
    const int next_ev = ev < ev_end && L.events[ev].frame < (uint32_t)L.frames ? (int)L.events[ev].frame : L.frames;
    const bool settled = __all_sync(0xffffffffu, lane < P_NP ? s.cur[lane] == s.tgt[lane] : true);
    const bool any_active = __any_sync(0xffffffffu, lane < 6 && s.v[lane].active != 0);
    if (settled && !any_active) {   // idle and nothing gliding: the tick only advances the clock (poly_synth.rs:512-525)
      const int n_idle = next_ev - j;
      for (int q = j + lane; q < next_ev; q += 32) out[q] = 0.0f;
      __syncwarp();
      if (lane == 0) { s.k += (uint32_t)n_idle; s.last_tick_time = L.tt[s.k - 1]; }
      __syncwarp();
      j = next_ev;
      continue;
    }
    int nl = min(min(j + 32, L.frames), next_ev) - j;
    const uint32_t k0 = s.k;
    float y = 0.0f;
    if (settled) {
      if (stale) {
        osc_shape = s.cur[P_SHAPE]; volume = s.cur[P_VOLUME];
        detune_ratio = 1.0 + (double)s.cur[P_DETUNE] * 0.0175;
        base_cutoff = 20.0f * gm::g_powf(18000.0f / 20.0f, s.cur[P_CUTOFF]);
        fenv_amt = s.cur[P_FENV_AMT];
        nr = fmaxf(0.5f + s.cur[P_RES] * 14.5f, 0.5f);
        stale = false;
      }
      const double now_l = L.tt[k0 + (uint32_t)min(lane, nl - 1)];
      // the first frame whose tick ends an amp envelope closes the block
      EnvBlk ab[6];
#pragma unroll
      for (int k = 0; k < 6; k++) {
        ab[k].j1 = ab[k].j2 = J_NONE;
        if (s.v[k].active) { ab[k] = env_block(s.v[k].amp_env, now_l, nl, lane); if (ab[k].j2 != J_NONE) nl = min(nl, ab[k].j2 + 1); }
      }
      // frames [0, live[k]) tick sub-voice k in full; at frame live[k] < nl its amp envelope ends
      int live[6];
#pragma unroll
      for (int k = 0; k < 6; k++) live[k] = !s.v[k].active ? 0 : (ab[k].j2 < nl ? ab[k].j2 : nl);
      const int pk = min(lane >> 1, 5);
      int my_live = 0;                                // live[] of the sub-voice this lane's chains belong to (lanes 0-11: pk, lanes 0-5: lane)
      int chain_live = 0;
#pragma unroll
      for (int k = 0; k < 6; k++) { if (k == pk) my_live = live[k]; if (k == lane) chain_live = live[k]; }
      if (lane >= 12) my_live = 0;
      // f64 phase accumulators: lane 2k + b replays phase_a (b = 0) / phase_b (b = 1) of sub-voice k (:458-466: read, then advance)
      double ph = 0.0;
      {
        const PolyVoice& pv = s.v[pk];
        const double inc = (lane & 1) ? pv.frequency * detune_ratio * dt : pv.frequency * dt;
        ph = (lane & 1) ? pv.phase_b : pv.phase_a;
        for (int n = 0; n < my_live; n++) { pst[lane][n] = ph; ph += inc; ph -= floor(ph); }
      }
      __syncwarp();
      // per frame and sub-voice: envelopes, oscillators, the cutoff the filter is asked for
      EnvBlk fb[6];
      float amp[6];
#pragma unroll
      for (int k = 0; k < 6; k++) {
        fb[k].j1 = fb[k].j2 = J_NONE; amp[k] = 0.0f;
        if (!s.v[k].active) continue;
        const PolyVoice& pv = s.v[k];
        const Env ae = env_after(pv.amp_env, ab[k], lane);
        amp[k] = env_value(ae, now_l);
        fb[k] = env_block(pv.flt_env, now_l, live[k], lane);
        if (lane < live[k]) {
          const Env fe = env_after(pv.flt_env, fb[k], lane);
          const float flt_env = env_value(fe, now_l);
          const double inc_a = pv.frequency * dt, inc_b = pv.frequency * detune_ratio * dt;
          const double pa = pst[2 * k][lane], pb = pst[2 * k + 1][lane];
          const float saw_a = polyblep_saw(pa, inc_a), sq_a = polyblep_square(pa, inc_a);
          const float osc_a = saw_a * (1.0f - osc_shape) + sq_a * osc_shape;
          const float saw_b = polyblep_saw(pb, inc_b), sq_b = polyblep_square(pb, inc_b);
          const float osc_b = saw_b * (1.0f - osc_shape) + sq_b * osc_shape;
          in_s[k][lane] = (osc_a + osc_b) * 0.5f;
          const float mod_cutoff = base_cutoff + fenv_amt * flt_env * (18000.0f - base_cutoff);
          nc_s[k][lane] = clampf(clampf(mod_cutoff, 20.0f, 18000.0f), 20.0f, sr * 0.45f);   // tpt_set's nc
        }
      }
      __syncwarp();
      // change threshold (state_variable_tpt.rs:83-92): lane k replays sub-voice k's sample-and-hold through the cutoff and
      // leaves the frames whose tick recomputes the coefficients
      unsigned mask = 0u;
      float fc = 0.0f;
      if (lane < 6 && chain_live > 0) {
        const Tpt& f = s.v[lane].filter;
        fc = f.cutoff;
        bool res_ok = !(fabsf(nr - f.res) > 0.001f);
        for (int n = 0; n < chain_live; n++) {
          const float nc = nc_s[lane][n];
          const bool upd = fabsf(nc - fc) > 0.001f || !res_ok;
          fc = upd ? nc : fc; res_ok = res_ok || upd;
          mask |= upd ? (1u << n) : 0u;
        }
      }
      // coefficient set in effect at each frame: that of the latest update frame <= the frame, else the carried one
#pragma unroll
      for (int k = 0; k < 6; k++) {
        if (!s.v[k].active) continue;
        const unsigned mk = __shfl_sync(0xffffffffu, mask, k);
        const Tpt& f = s.v[k].filter;
        float g_l = f.g, h_l = f.h;
        if (mk) {
          Tpt spec; spec.g = spec.r = spec.h = 0.0f;
          if ((mk >> lane) & 1u) { spec.cutoff = nc_s[k][lane]; spec.res = nr; tpt_update(spec, sr); }
          const unsigned m = mk & ((2u << lane) - 1u);
          const int src = m ? 31 - __clz(m) : 0;
          const float sg = __shfl_sync(0xffffffffu, spec.g, src), sh = __shfl_sync(0xffffffffu, spec.h, src);
          if (m) { g_l = sg; h_l = sh; }
          const int lu = 31 - __clz(mk);
          const float lg = __shfl_sync(0xffffffffu, spec.g, lu), lr = __shfl_sync(0xffffffffu, spec.r, lu), lh = __shfl_sync(0xffffffffu, spec.h, lu);
          if (lane == k) { coef[warp][k][0] = lg; coef[warp][k][1] = lr; coef[warp][k][2] = lh; }
        }
        if (lane < live[k]) { g_s[k][lane] = g_l; h_s[k][lane] = h_l; }
      }
      __syncwarp();
      // filter state: lane k runs tpt_process (dsp.cuh) of sub-voice k with each frame's coefficients; only the low-pass is used
      float ic1 = 0.0f, ic2 = 0.0f;
      if (lane < 6 && s.v[lane].active) {
        ic1 = s.v[lane].filter.ic1; ic2 = s.v[lane].filter.ic2;
        for (int n = 0; n < chain_live; n++) {
          const float g = g_s[lane][n], h = h_s[lane][n], in = in_s[lane][n];
          const float v1 = (g * (in - ic2) + ic1) * h;
          const float v2 = ic2 + g * v1;
          ic1 = 2.0f * v1 - ic1;
          ic2 = 2.0f * v2 - ic2;
          lo_s[lane][n] = v2;
        }
      }
      __syncwarp();
      float acc = 0.0f;
#pragma unroll
      for (int k = 0; k < 6; k++) {
        float yk = 0.0f;
        if (s.v[k].active && lane < live[k]) yk = lo_s[k][lane] * amp[k] * sqrtf(s.v[k].velocity) * volume;
        acc += yk;
      }
      y = acc * (1.0f / 4.0f);
      __syncwarp();
      // commit the block: each chain lane its own result, lane 0 the latches and the clock
      if (lane < 12 && my_live > 0) { if (lane & 1) s.v[pk].phase_b = ph; else s.v[pk].phase_a = ph; }
      if (lane < 6 && s.v[lane].active) {
        Tpt& f = s.v[lane].filter;
        if (mask) { f.cutoff = fc; f.res = nr; f.g = coef[warp][lane][0]; f.r = coef[warp][lane][1]; f.h = coef[warp][lane][2]; }
        f.ic1 = ic1; f.ic2 = ic2;
      }
      __syncwarp();
      if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 6; k++) {
          if (!s.v[k].active) continue;
          s.v[k].flt_env = env_after(s.v[k].flt_env, fb[k], live[k]);
          s.v[k].amp_env = env_after(s.v[k].amp_env, ab[k], nl);
          if (!env_active(s.v[k].amp_env)) s.v[k].active = 0;
        }
        s.k = k0 + (uint32_t)nl;
        s.last_tick_time = L.tt[k0 + (uint32_t)nl - 1];
      }
      __syncwarp();
    } else {
      // ---- per-sample path for this block (gliding parameters) ----
      if (lane == 0) for (int n = 0; n < nl; n++) ticks[warp][n] = poly_tick(s, L.tt, rc);
      stale = true;
      __syncwarp();
      y = ticks[warp][min(lane, nl - 1)];
      __syncwarp();
    }
    if (lane < nl) out[j + lane] = y;
    j += nl;
  }
  __syncwarp();
  {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(&s);
    for (int i = lane; i < POLY_WORDS; i += 32) L.state[(size_t)i * L.n_pad + sv] = w[i];
  }
}

void poly_wave_launch(const VoiceLaunch& L, cudaStream_t st) {
  // Every kernel of a render runs at the maximum shared-memory carve-out (pool.cuh same_carveout): kernels whose
  // carve-outs differ cannot share an SM.
  auto kernel = poly_wave_kernel<POLY_WAVE_WARPS>;
  gh::func_attr_once((const void*)kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  kernel<<<(L.n + POLY_WAVE_WARPS - 1) / POLY_WAVE_WARPS, POLY_WAVE_WARPS * 32, 0, st>>>(L);
}
void poly_wave_set_midi_freq(const double mf[128]) { GH_CUDA(cudaMemcpyToSymbol(c_midi_freq, mf, 128 * sizeof(double))); }

}  // namespace gd
