// gran_wave.cuh — the granulator, one warp per instance (reference: src/instruments/granulator.rs:511-742).
//
// A granulator tick is: parameter smoothers -> spawn due grains (f64 schedule, xorshift32 draws, slot search / steal) ->
// gain compensation 1/sqrt(active) through a 10 ms smoother -> for each of the 64 + 16 grain slots a cubic read of the
// source buffer, a sin^shape window (sinf + powf), fades, overlap-add -> drive waveshaper -> volume.
// The per-grain work is ~95 % of the instructions and grains do not interact, so the warp's lanes own the slots
// (lane l: slots l, l + 32, l + 64) and the overlap-add is a warp-shuffle reduction; the rare control events (spawn /
// steal at <= 80 per second, parameter glides, cloud end) are run by lane 0 on the shared-memory copy of the state with
// the very functions the per-sample path uses (voices2.cuh), so their arithmetic and order are the reference's.
// The only re-association is the overlap-add itself: 80 f32 terms summed as a fixed shuffle tree instead of slot order
// (<= 1e-7 of full scale).
#pragma once
#include "kernels.cuh"

namespace gd {

constexpr int GRAN_WORDS = sizeof(GranState) / 4;

template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) gran_wave_kernel(const VoiceLaunch L) {
  __shared__ GranState states[WARPS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int v = blockIdx.x * WARPS + warp;
  if (v >= L.n) return;
  const int sv = L.slots ? (int)L.slots[v] : v;
  GranState& s = states[warp];
  {
    uint32_t* w = reinterpret_cast<uint32_t*>(&s);
    for (int i = lane; i < GRAN_WORDS; i += 32) w[i] = L.state[(size_t)i * L.n_pad + sv];
  }
  __syncwarp();
  uint32_t ev = L.ev_begin[v];
  const uint32_t ev_end = L.ev_begin[v + 1];
  const long long row = L.rows ? (long long)L.rows[v] : (long long)(L.row0 + v);
  float* out = L.out + row * L.stride;
  const RateCtx& rc = L.rc;
  const float sr = rc.sr;
  bool settled = false;                       // re-derived after every event
  int tg_n = -1; float tg = 1.0f;             // lane 0: active-grain count of the last gain-compensation target and the target
  for (int f0 = 0; f0 < L.frames; f0 += 32) {
    const int nf = min(32, L.frames - f0);
    float mine = 0.0f;
    for (int j = 0; j < nf; j++) {
      const uint32_t frame = (uint32_t)(f0 + j);
      // ---- control part: lane 0, on the shared state, with the per-sample path's own code ----
      if (ev < ev_end && L.events[ev].frame <= frame) {
        if (lane == 0) while (ev < ev_end && L.events[ev].frame <= frame) { gran_event(s, L.events[ev], L.tt); ev++; }
        ev = __shfl_sync(0xffffffffu, ev, 0);
        settled = false;
        __syncwarp();
      }
      const double now = L.tt[s.k];
      bool spawn_check = false;
      if (lane == 0) {
        s.k += 1;
        if (!settled) {
#pragma unroll
          for (int i = 0; i < G_NP; i++) smooth_tick(s.cur[i], s.tgt[i], rc.smooth15);
        }
        if (s.cloud_active) {
          if (now > s.cloud_end) s.cloud_active = 0;
          else spawn_check = now + 1e-12 >= s.next_grain;
        }
        if (spawn_check) {      // spawn_due_grains (granulator.rs:511-544), verbatim from gran_tick
          const float* buf = reinterpret_cast<const float*>(((uint64_t)s.buf_hi << 32) | s.buf_lo);
          const float density = clampf(s.cur[G_DENSITY], 0.0f, 1.0f) * 80.0f;
          if (density > 0.0f && buf != nullptr && s.buf_len > 0) {
            const double interval = 1.0 / (double)density;
            const double random_timing = (double)clampf(s.cur[G_RAND_TIMING], 0.0f, 1.0f);
            int guard = 0;
            while (s.cloud_active && now + 1e-12 >= s.next_grain && guard < 8) {
              gran_spawn(s, sr);
              s.next_grain += interval;
              if (random_timing > 0.0) {
                const double jitter = ((double)gran_next_f32(s) * 2.0 - 1.0) * interval * random_timing;
                s.next_grain = fmax(s.next_grain + jitter, now);
              }
              if (s.next_grain > s.cloud_end) s.cloud_active = 0;
              guard++;
            }
          }
        }
      }
      __syncwarp();
      if (!settled) {
        bool st = true;
        if (lane < G_NP) st = s.cur[lane] == s.tgt[lane];
        settled = __all_sync(0xffffffffu, st);
      }
      // ---- tick_grains (granulator.rs:661-718): lanes own slots lane, lane + 32, lane + 64 ----
      int n_act = 0;
#pragma unroll
      for (int q = 0; q < 3; q++) { const int i = lane + 32 * q; if (i < 80) n_act += (int)s.grains[i].active; }
      n_act = __reduce_add_sync(0xffffffffu, n_act);                       // one redux.sync instead of a five-step shuffle tree
      float raw = 0.0f;
      if (lane == 0) {
        if (n_act != tg_n) { tg_n = n_act; tg = n_act == 0 ? 1.0f : clampf(1.0f / sqrtf((float)n_act), 0.0f, 1.0f); }   // pure function of the count: once per change
        if (fabsf(s.gc_tgt - tg) > 1e-8f) s.gc_tgt = tg;
        smooth_tick(s.gc_cur, s.gc_tgt, rc.smooth10);
      }
      __syncwarp();
      if (n_act > 0) {
        const float gc = s.gc_cur;
        const float* buf = reinterpret_cast<const float*>(((uint64_t)s.buf_hi << 32) | s.buf_lo);
        const uint32_t blen = s.buf_len;
        float part = 0.0f;
#pragma unroll
        for (int q = 0; q < 3; q++) {
          const int i = lane + 32 * q;
          if (i >= 80) continue;
          Grain& g = s.grains[i];
          if (!g.active) continue;
          if (g.age >= g.duration) { g.active = 0; continue; }
          const float phase = clampf(__fdividef(g.age, g.duration), 0.0f, 1.0f);     // 2-ulp quotient: the argument of a memoryless window (below)
          // window = max(sin(pi phase), 0) ^ shape (granulator.rs:686-689).  A memoryless gain in [0, 1] applied to one grain of up to 80:
          // the ~1-ulp sine of the front ends (relative accuracy kept near its zeros: the reduction is exact) and exp2(shape log2 s) with
          // `lg2.approx` / CUDA's exp2f — relative error <= 3e-5 where the window is below 1e-4, <= 1e-6 elsewhere — replace ~180 instructions of the bit-exact ports per
          // grain-sample.
          const float sw = fmaxf(gm::g_sinf_fast(PI_F * clampf(phase, 0.0f, 1.0f)), 0.0f);
          const float window = sw > 0.0f ? exp2f(g.window_shape * __log2f(sw)) : gm::g_powf(sw, g.window_shape);   // lg2.approx: 2^-22 absolute on [0.5, 2], relative elsewhere
          const float rg = g.release_total > 0.0f ? clampf(__fdividef(g.release_samples, g.release_total), 0.0f, 1.0f) : 1.0f;   // release fade: a gain, 2-ulp quotient
          const float smp = gran_sample(buf, blen, g.source_pos);
          part += smp * window * rg * g.velocity * gc;
          g.source_pos += g.speed * g.direction;
          g.age += 1.0f;
          if (g.release_samples > 0.0f) { g.release_samples -= 1.0f; if (g.release_samples <= 0.0f) g.active = 0; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        raw = part;
      }
      // ---- drive + volume (granulator.rs:730-742): lane 0 owns the waveshaper's oversampler state ----
      float y = 0.0f;
      if (lane == 0) {
        s.drive.mix = clampf(s.cur[G_DRIVE], 0.0f, 1.0f);
        y = ws_process(s.drive, raw) * s.cur[G_VOLUME];
      }
      y = __shfl_sync(0xffffffffu, y, 0);
      if (j == lane) mine = y;
      __syncwarp();
    }
    if (lane < nf) out[f0 + lane] = mine;
  }
  __syncwarp();
  {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(&s);
    for (int i = lane; i < GRAN_WORDS; i += 32) L.state[(size_t)i * L.n_pad + sv] = w[i];
  }
}

}  // namespace gd
