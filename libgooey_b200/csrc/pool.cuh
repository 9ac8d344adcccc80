// pool.cuh — host-side state pools, the engine clock table and the per-type launch sequence.
//
// Pool<S>: every instance of one voice type (or every engine's mix state) on one device, stored
// word-interleaved (SoA) with a fixed row pitch (capacity).  Slots are allocated on the host, their
// constructor-built initial states (voices.cuh init functions run on the host through the bit-exact
// gm:: math) are uploaded lazily in bulk.
// TypeRunner<V>: the per-render list of (slot, output row, events) for one type bucket and the
// A -> (B | C pipelined over time chunks) + S launch sequence of kernels.cuh.  Type bucketing keeps
// warps type-homogeneous (no cross-instrument divergence).  choose_back() fixes which kernel plays C for the drums;
// the bass, the granulator and the poly synth have one path each (their warp kernels, or kernel S for LFO-routed
// basses), apart from the serial reference below.
#pragma once
#include <algorithm>
#include <atomic>
#include <map>
#include <type_traits>
#include <mutex>
#include <tuple>
#include "device_rt.h"
#include "wave.cuh"
#include "coop.cuh"
#include "gran_wave.cuh"
#include "bass_wave.cuh"
#include "poly_wave.cuh"
#include "patch.h"

namespace gh {

extern std::atomic<uint64_t> g_launches;

// Per-kernel device time, measured with CUDA events on the stream the kernel is launched on (bench.py's roofline line).
struct KernelStat { uint64_t launches = 0; double ms = 0.0; double voice_frames = 0.0; };
std::map<std::string, KernelStat>& kernel_stats();
std::mutex& kernel_stats_mutex();
// Times launches for kernel_stats(): begin() and end() bracket one launch on its stream with reusable events.  collect()
// runs once the caller has synchronised those streams; it adds the bracketed launches to the table and forgets them.
// clear() forgets them uncounted.
struct KernelTimer {
  struct Rec { cudaEvent_t t0, t1; const char* key; double units; };
  std::vector<Rec> recs;
  size_t n = 0;                          // records bracketed since the last collect() / clear()
  KernelTimer() = default;
  KernelTimer(const KernelTimer&) = delete;
  ~KernelTimer() { for (const Rec& r : recs) { cudaEventDestroy(r.t0); cudaEventDestroy(r.t1); } }
  void begin(cudaStream_t s) {
    if (n == recs.size()) { Rec r{}; GH_CUDA(cudaEventCreate(&r.t0)); GH_CUDA(cudaEventCreate(&r.t1)); recs.push_back(r); }
    GH_CUDA(cudaEventRecord(recs[n].t0, s));
  }
  void end(cudaStream_t s, const char* key, double units) {   // units: voice-frames (or engine-frames) of the launch
    Rec& r = recs[n++];
    r.key = key; r.units = units;
    GH_CUDA(cudaEventRecord(r.t1, s));
  }
  void clear() { n = 0; }
  // after a synchronise: the device time of record i, or -1 when it cannot be read (the error is cleared)
  float elapsed(size_t i) const {
    float ms = 0.0f;
    if (cudaEventElapsedTime(&ms, recs[i].t0, recs[i].t1) == cudaSuccess) return ms;
    cudaGetLastError();
    return -1.0f;
  }
  float ms() const { float sum = 0.0f; for (size_t i = 0; i < n; i++) sum += std::max(elapsed(i), 0.0f); return sum; }
  void collect() {
    std::lock_guard<std::mutex> lk(kernel_stats_mutex());
    for (size_t i = 0; i < n; i++) {
      const float ms = elapsed(i);
      if (ms < 0.0f) continue;
      KernelStat& k = kernel_stats()[recs[i].key];
      k.launches++; k.ms += ms; k.voice_frames += recs[i].units;
    }
    n = 0;
  }
};

__global__ void scatter_words_kernel(uint32_t* __restrict__ dst, long long cap, const uint32_t* __restrict__ src, const uint32_t* __restrict__ slots,
                                     int n, int words) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint32_t s = slots[k];
  for (int w = 0; w < words; w++) dst[(long long)w * cap + s] = src[(long long)w * n + k];
}

template <class S> struct Pool {
  static_assert(sizeof(S) % 4 == 0, "state must be whole 32-bit words");
  static constexpr int W = sizeof(S) / 4;
  DevBuf<uint32_t> d;
  int cap = 0, count = 0;
  std::vector<int> free_list;
  std::vector<std::pair<int, S>> pending;

  int alloc(const S& init) {
    int slot;
    if (!free_list.empty()) { slot = free_list.back(); free_list.pop_back(); } else slot = count++;
    pending.emplace_back(slot, init);
    return slot;
  }
  void release(int slot) {
    for (size_t i = 0; i < pending.size(); i++) if (pending[i].first == slot) { pending.erase(pending.begin() + i); break; }
    free_list.push_back(slot);
  }
  // grow (content preserving) and upload every pending initial state
  void flush(cudaStream_t st) {
    if (count > cap) {
      // Row pitch of the word-interleaved state (and of every ring arena that follows the mix pool's capacity).  Kept an ODD
      // multiple of 32 slots: with a power-of-two pitch the words of one slot (pitch * 4 bytes apart) fall into the same L1 / L2
      // sets and evict each other (measured: 1600 granulators ran 1.8x slower in a pool that had grown to 2048 slots).
      int ncap = std::max(pad32(count), cap * 2);
      if (((ncap / 32) & 1) == 0) ncap += 32;
      DevBuf<uint32_t> nd;
      nd.alloc((size_t)W * ncap);
      GH_CUDA(cudaMemsetAsync(nd.p, 0, (size_t)W * ncap * 4, st));
      if (cap > 0) GH_CUDA(cudaMemcpy2DAsync(nd.p, (size_t)ncap * 4, d.p, (size_t)cap * 4, (size_t)cap * 4, W, cudaMemcpyDeviceToDevice, st));
      GH_CUDA(cudaStreamSynchronize(st));
      std::swap(d.p, nd.p); std::swap(d.n, nd.n);
      cap = ncap;
    }
    if (pending.empty()) return;
    const int n = (int)pending.size();
    std::vector<uint32_t> words((size_t)W * n), slots(n);
    for (int k = 0; k < n; k++) {
      slots[k] = (uint32_t)pending[k].first;
      const uint32_t* w = reinterpret_cast<const uint32_t*>(&pending[k].second);
      for (int i = 0; i < W; i++) words[(size_t)i * n + k] = w[i];
    }
    DevBuf<uint32_t> dw, ds;
    dw.upload(words.data(), words.size(), st);
    ds.upload(slots.data(), slots.size(), st);
    scatter_words_kernel<<<(n + 127) / 128, 128, 0, st>>>(d.p, cap, dw.p, ds.p, n, W);
    g_launches.fetch_add(1);
    GH_CUDA(cudaGetLastError());
    GH_CUDA(cudaStreamSynchronize(st));
    pending.clear();
    pending.shrink_to_fit();
  }
};

inline gd::VoiceEvent make_event(uint32_t frame, uint32_t kind, uint32_t param, float value, uint32_t aux = 0) {
  gd::VoiceEvent e; e.frame = frame; e.kind = (uint16_t)kind; e.param = (uint16_t)param; e.value = value; e.aux = aux;
  return e;
}
// Granulator::set_buffer at `frame`: the buffer's device address (low word in the bits of the value), which kills every grain,
// then its sample rate and length.
inline void gran_buffer_events(std::vector<gd::VoiceEvent>& out, uint32_t frame, const float* buf, float sr, uint32_t len) {
  const uint64_t ptr = (uint64_t)(uintptr_t)buf;
  float lo; uint32_t lo_bits = (uint32_t)ptr; memcpy(&lo, &lo_bits, 4);
  out.push_back(make_event(frame, gd::EV_GRAN_BUFFER, 0, lo, (uint32_t)(ptr >> 32)));
  out.push_back(make_event(frame, gd::EV_SET_AUX, gd::AUX_GRAN_BUFINFO, sr, len));
}

// The engine clock: tt[k] = value of a f64 accumulator after k additions of 1/sr, exactly as the reference's
// `current_time += 1.0 / sample_rate` (bounce.rs:48-53, ffi.rs:1379).  The host keeps one checkpoint every CK additions
// (8 bytes per 1.5 s of audio) and rebuilds any window [k0, k0 + n) from the nearest checkpoint by the same repeated
// addition, so memory does not grow with how long an engine has been streaming.
struct ClockTable {
  static constexpr uint64_t CK = 65536;
  double dt = 0.0;
  std::vector<double> ckpt;   // ckpt[i] = value after i * CK additions
  std::mutex mu;
  void fill(uint64_t k0, size_t n, double* out) {
    std::lock_guard<std::mutex> lk(mu);
    if (ckpt.empty()) ckpt.push_back(0.0);
    const uint64_t need = k0 / CK;
    while (ckpt.size() <= need) { double t = ckpt.back(); for (uint64_t i = 0; i < CK; i++) t += dt; ckpt.push_back(t); }
    double t = ckpt[need];
    for (uint64_t k = need * CK; k < k0; k++) t += dt;
    for (size_t i = 0; i < n; i++) { out[i] = t; t += dt; }
  }
};
// A caller-owned device copy of tt[k0 .. k0 + n): view() returns a pointer `p` such that p[k] is valid for every k of the
// requested range (kernels index the clock with absolute k).  Uploads are ordered on the caller's stream; a window that
// already covers the range is reused (a bounce always asks for [0, frames]).
struct ClockWindow {
  DevBuf<double> d;
  std::vector<double> h;
  uint64_t k0 = 0; size_t n = 0;
  const double* view(ClockTable& T, uint64_t kmin, uint64_t kmax, cudaStream_t st) {
    if (kmin > 0) kmin -= 1;                                   // the poly synth's catch-up reads tt[k - 1]
    if (!(n && kmin >= k0 && kmax < k0 + n)) {
      const size_t want = (size_t)(kmax - kmin + 1);
      const size_t cap = std::max<size_t>((want + 8191) & ~(size_t)8191, 1u << 16);
      if (d.n < cap) { GH_CUDA(cudaStreamSynchronize(st)); d.alloc(cap); }
      h.resize(want);
      T.fill(kmin, want, h.data());
      GH_CUDA(cudaMemcpyAsync(d.p, h.data(), want * sizeof(double), cudaMemcpyHostToDevice, st));
      GH_CUDA(cudaStreamSynchronize(st));                      // h is reused by the next call
      k0 = kmin; n = want;
    }
    return d.p - k0;
  }
};
ClockTable& clock_table(float sr);

// ---- the back ends (kernel C of the A -> (B | C) + S sequence) ----
// launch_back<V>() launches the back end of a bucket and returns its kernel-statistics key.  Which kernel renders a drum
// bucket depends on the voice type and on how many voices of the type one launch holds (choose_back):
//   tom, >= COOP_FROM voices                      coop_kernel<TomC, COOP_NV>   (coop.cuh)
//   kick / snare / hi-hat / tom, fewer voices     wave_kernel<...W>           (wave.cuh)
//   kick / snare / hi-hat, >= SERIAL_FROM voices  back_kernel<V, 32>          (kernels.cuh)
// The other types have one back end each: bass_wave_kernel (slow_kernel<BassV> for LFO-routed basses), poly_wave_kernel
// and gran_wave_kernel.  GOOEY_B200_BACKEND=serial puts every drum on back_kernel and every poly synth on
// slow_kernel<PolyV> (instead of poly_wave_kernel): the per-sample-order references of the parity tests.
enum class Back { Wave, Coop, Serial };
// The cooperative back end issues ~3x fewer instructions per voice-frame but walks a block through barrier-separated phases,
// so a voice's timeline is slower than in the warp-per-voice back end while voices are too few to fill the device with CTAs:
// it takes over from this many voices of one type (measured crossover).
constexpr int COOP_FROM = 4096;
constexpr int COOP_NV = 16;          // voices per cooperative CTA
// From this many voices of one type the per-sample-order back end with one voice per THREAD wins: the warp-per-voice
// back end spends 32 lanes on the replayed recurrences of one voice, which pays only while voices are too few to fill the
// device with threads (measured, 32768 voices x 2 s: tom 234 vs 526 ms, hi-hat 117 vs 193 ms; at 16384: 176 vs 263 and
// 104 vs 97 ms).
constexpr int SERIAL_FROM = 12288;
inline bool serial_backend() { const char* e = getenv("GOOEY_B200_BACKEND"); return e && strcmp(e, "serial") == 0; }
template <class V> inline Back choose_back(int cnt) {
  if (serial_backend()) return Back::Serial;
  if (std::is_same<V, gd::TomV>::value) return cnt >= COOP_FROM ? Back::Coop : Back::Wave;
  return cnt >= SERIAL_FROM ? Back::Serial : Back::Wave;
}
// The scan back end of each drum type and its kernel-statistics key.
template <class V> struct WaveOf;
template <> struct WaveOf<gd::KickV> { using W = gd::wave::KickW; static constexpr const char* name = "wave_kernel<KickW>"; };
template <> struct WaveOf<gd::SnareV> { using W = gd::wave::SnareW; static constexpr const char* name = "wave_kernel<SnareW>"; };
template <> struct WaveOf<gd::HatV> { using W = gd::wave::HatW; static constexpr const char* name = "wave_kernel<HatW>"; };
template <> struct WaveOf<gd::TomV> { using W = gd::wave::TomW; static constexpr const char* name = "wave_kernel<TomW>"; };

inline void coop_launch(int cnt, cudaStream_t s, const gd::VoiceLaunch& L) {
  using SM = gd::coop::Smem<gd::coop::TomC, COOP_NV>;
  auto kernel = gd::coop::coop_kernel<gd::coop::TomC, COOP_NV>;
  func_attr_once((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SM));
  func_attr_once((const void*)kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  kernel<<<(cnt + COOP_NV - 1) / COOP_NV, COOP_NV * 32, sizeof(SM), s>>>(L);
}

// Kernels whose shared-memory carve-out differs cannot share an SM: the L1 / shared split is an SM-wide setting, so a
// back end with 19 KB of scan tables per CTA and one with 3.5 KB would be given disjoint SMs instead of interleaving
// their warps.  Every kernel of the render is therefore pinned to the same (maximum shared) carve-out, once per device.
template <class K> inline void same_carveout(K kernel) {
  func_attr_once((const void*)kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
}
#define GH_LAUNCH(kernel, grid, block, stream, ...) do { same_carveout(kernel); kernel<<<grid, block, 0, stream>>>(__VA_ARGS__); } while (0)

// The per-sample kernel S as a bucket's back end: one-warp CTAs up to 148 * 32 * 4 voices, 128-thread CTAs above.
template <class V> inline void slow_launch(const gd::VoiceLaunch& L, cudaStream_t s) {
  if (L.n <= 148 * 32 * 4) GH_LAUNCH((gd::slow_kernel<V, 32>), (L.n + 31) / 32, 32, s, L);
  else GH_LAUNCH((gd::slow_kernel<V, 128>), (L.n + 127) / 128, 128, s, L);
}
// The drums; the other types specialise it below.
template <class V> inline const char* launch_back(const gd::VoiceLaunch& L, cudaStream_t s) {
  const Back back = choose_back<V>(L.n);
  if (back == Back::Coop) { coop_launch(L.n, s, L); return "coop_kernel<TomC>"; }
  if (back == Back::Wave) {
    GH_LAUNCH((gd::wave::wave_kernel<typename WaveOf<V>::W>), L.n, 32, s, L);   // one voice per one-warp CTA
    return WaveOf<V>::name;
  }
  GH_LAUNCH((gd::back_kernel<V, 32>), (L.n + 31) / 32, 32, s, L);             // one voice per lane, one warp per CTA
  return "back_kernel";
}
template <> inline const char* launch_back<gd::BassV>(const gd::VoiceLaunch& L, cudaStream_t s) {
  if (L.routes) { slow_launch<gd::BassV>(L, s); return "slow_kernel<BassV>"; }   // LFO-routed basses
  GH_LAUNCH((gd::bass_wave_kernel<2>), (L.n + 1) / 2, 64, s, L);                 // one warp per bass voice, lane = frame (bass_wave.cuh)
  return "bass_wave_kernel";
}
template <> inline const char* launch_back<gd::PolyV>(const gd::VoiceLaunch& L, cudaStream_t s) {
  if (serial_backend()) { slow_launch<gd::PolyV>(L, s); return "slow_kernel<PolyV>"; }
  gd::poly_wave_launch(L, s);                                                      // one warp per poly synth, lane = frame (poly_wave.cu)
  return "poly_wave_kernel";
}
template <> inline const char* launch_back<gd::GranV>(const gd::VoiceLaunch& L, cudaStream_t s) {
  GH_LAUNCH((gd::gran_wave_kernel<4>), (L.n + 3) / 4, 128, s, L);                 // one warp per granulator, grains on lanes (gran_wave.cuh)
  return "gran_wave_kernel";
}

// Frames per front/back pipeline stage.
constexpr int CHUNK_FRAMES = 8192;
// One type bucket of one render call.
template <class V> struct TypeRunner {
  using State = typename V::State;
  Pool<State> pool;
  std::vector<uint32_t> slots, rows, ev_begin, span_off;
  std::vector<gd::VoiceEvent> ev_flat;
  std::vector<gd::ModRoute> routes_flat; std::vector<uint32_t> route_begin;       // LFO routes per voice of this launch
  DevBuf<gd::ModRoute> d_routes; DevBuf<uint32_t> d_route_begin;
  const float* mod_planes = nullptr; long long mod_pitch = 0; int mod_frame0 = 0;  // set by the engine path before launch()
  DevBuf<uint32_t> d_slots, d_rows, d_ev_begin, d_span_off, d_n_spans, d_span_cursor;
  DevBuf<gd::VoiceEvent> d_events;
  DevBuf<uint8_t> d_mode, d_spans;
  DevBuf<float> d_planes[2];
  cudaStream_t sB = nullptr, sC = nullptr, sS = nullptr;
  cudaEvent_t evA = nullptr, evB[2] = {nullptr, nullptr}, evC[2] = {nullptr, nullptr}, evDoneC = nullptr, evDoneS = nullptr;
  KernelTimer timer;                     // the back-end launches of the most recent launch (on sC)
  std::vector<cudaEvent_t> evChunk;      // evChunk[i]: frames of chunk i are final in the output (fast-path voices)
  int launched_chunks = 0;               // chunks of the most recent launch (0 = one undivided launch)
  static int chunk_of(int frames) { return std::min(CHUNK_FRAMES, (frames + 31) & ~31); }
  // Makes `s` wait until every voice of this bucket has written frames [i * chunk, (i + 1) * chunk) of the last launch.
  void wait_chunk(cudaStream_t s, int i) {
    if (n() == 0) return;
    if (launched_chunks == 0) { GH_CUDA(cudaStreamWaitEvent(s, evDoneC, 0)); return; }
    GH_CUDA(cudaStreamWaitEvent(s, evDoneS, 0));
    GH_CUDA(cudaStreamWaitEvent(s, evChunk[std::min(i, launched_chunks - 1)], 0));
  }

  int n() const { return (int)slots.size(); }
  // a new voice built from `p` (the reference's `<Voice>::with_config`): its pool slot
  int create(const GooeyVoicePatch& p, float sr) { State s; init_from_patch(s, p, sr); return pool.alloc(s); }
  void reset() { slots.clear(); rows.clear(); ev_flat.clear(); ev_begin.clear(); ev_begin.push_back(0); span_off.clear(); span_off.push_back(0);
                 routes_flat.clear(); route_begin.clear(); route_begin.push_back(0); }
  // events must be ordered by frame and lie inside the call
  void add(uint32_t slot, uint32_t out_row, const std::vector<gd::VoiceEvent>& events, const std::vector<gd::ModRoute>* routes = nullptr) {
    slots.push_back(slot); rows.push_back(out_row);
    if (routes) routes_flat.insert(routes_flat.end(), routes->begin(), routes->end());
    route_begin.push_back((uint32_t)routes_flat.size());
    uint32_t distinct = 0, last = 0xffffffffu;
    for (const auto& e : events) { if (e.frame != last) { distinct++; last = e.frame; } }
    ev_flat.insert(ev_flat.end(), events.begin(), events.end());
    ev_begin.push_back((uint32_t)ev_flat.size());
    span_off.push_back(span_off.back() + distinct + 1);
  }
  void ensure_streams() {
    if (sC) return;
    // Equal stream priorities: ranking the buckets by the length of their chunk chains measured as noise on C2 (the tom
    // chain is slowed by sharing issue slots, not by waiting for them).
    GH_CUDA(cudaStreamCreateWithFlags(&sB, cudaStreamNonBlocking));
    GH_CUDA(cudaStreamCreateWithFlags(&sC, cudaStreamNonBlocking));
    GH_CUDA(cudaStreamCreateWithFlags(&sS, cudaStreamNonBlocking));
    cudaEvent_t* evs[] = {&evA, &evB[0], &evB[1], &evC[0], &evC[1], &evDoneC, &evDoneS};
    for (auto e : evs) GH_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  }
  ~TypeRunner() {
    cudaEvent_t evs[] = {evA, evB[0], evB[1], evC[0], evC[1], evDoneC, evDoneS};
    for (auto e : evs) if (e) cudaEventDestroy(e);
    for (auto e : evChunk) cudaEventDestroy(e);
    if (sB) cudaStreamDestroy(sB);
    if (sC) cudaStreamDestroy(sC);
    if (sS) cudaStreamDestroy(sS);
  }
  // After the launch's streams have been synchronised: add the back-end launches of the last call to the global table.
  void collect_stats() { timer.collect(); }
  // Forks from `parent` (after `start`), runs the bucket on its own streams, joins back into `parent`.
  void launch(cudaStream_t parent, cudaEvent_t start, const gd::RateCtx& rc, const double* tt, int frames, float* out, long long stride) {
    const int cnt = n();
    launched_chunks = 0;
    timer.clear();
    if (cnt == 0 || frames <= 0) return;
    ensure_streams();
    GH_CUDA(cudaStreamWaitEvent(sC, start, 0));
    pool.flush(sC);
    d_slots.upload(slots.data(), slots.size(), sC);
    d_rows.upload(rows.data(), rows.size(), sC);
    if (ev_flat.empty()) ev_flat.push_back(make_event(0xffffffffu, 0xffff, 0, 0.0f));
    d_events.upload(ev_flat.data(), ev_flat.size(), sC);
    d_ev_begin.upload(ev_begin.data(), ev_begin.size(), sC);
    gd::VoiceLaunch L;
    memset(&L, 0, sizeof L);
    L.state = pool.d.p; L.n = cnt; L.n_pad = pool.cap;
    L.slots = d_slots.p; L.rows = d_rows.p; L.row0 = 0;
    L.events = d_events.p; L.ev_begin = d_ev_begin.p; L.tt = tt; L.frames = frames; L.out = out; L.stride = stride; L.rc = rc;
    if (!routes_flat.empty() && mod_planes) {
      d_routes.upload(routes_flat.data(), routes_flat.size(), sC);
      d_route_begin.upload(route_begin.data(), route_begin.size(), sC);
      L.routes = d_routes.p; L.route_begin = d_route_begin.p; L.mod_planes = mod_planes; L.mod_pitch = mod_pitch; L.mod_frame0 = mod_frame0;
    }
    const char* key = nullptr;
    if constexpr (V::FAST) {
      using Span = typename V::Span;
      d_span_off.upload(span_off.data(), span_off.size(), sC);
      d_n_spans.alloc(cnt); d_span_cursor.alloc(cnt); d_mode.alloc(cnt);
      d_spans.alloc((size_t)span_off.back() * sizeof(Span));
      const int chunk = chunk_of(frames);
      const int rows_pad = pad32(cnt);
      const size_t plane_floats = (size_t)rows_pad * chunk;
      d_planes[0].alloc(plane_floats * V::NPL); d_planes[1].alloc(plane_floats * V::NPL);
      L.mode = d_mode.p; L.spans = d_spans.p; L.span_off = d_span_off.p; L.n_spans = d_n_spans.p; L.span_cursor = d_span_cursor.p;
      L.plane_stride = (long long)plane_floats; L.pitch = chunk;
      GH_LAUNCH((gd::plan_kernel<V>), (cnt + 63) / 64, 64, sC, L);
      g_launches.fetch_add(1, std::memory_order_relaxed);
      GH_CUDA(cudaGetLastError());
      GH_CUDA(cudaEventRecord(evA, sC));
      GH_CUDA(cudaStreamWaitEvent(sB, evA, 0));
      GH_CUDA(cudaStreamWaitEvent(sS, evA, 0));
      // general path for the voices A could not plan (whole call, one launch)
      GH_LAUNCH((gd::slow_kernel<V, 32>), (cnt + 31) / 32, 32, sS, L);
      g_launches.fetch_add(1, std::memory_order_relaxed);
      GH_CUDA(cudaGetLastError());
      GH_CUDA(cudaEventRecord(evDoneS, sS));
      int i = 0;
      for (int c0 = 0; c0 < frames; c0 += chunk, i++) {
        const int b = i & 1;
        L.chunk0 = c0; L.chunk_frames = std::min(chunk, frames - c0);
        L.planes = d_planes[b].p;
        if (i >= 2) GH_CUDA(cudaStreamWaitEvent(sB, evC[b], 0));   // plane buffer b is free once C of chunk i-2 is done
        const int bpv = (L.chunk_frames + 255) / 256;
        GH_LAUNCH((gd::front_kernel<V, 256>), (unsigned)((size_t)cnt * bpv), 256, sB, L, bpv);
        GH_CUDA(cudaGetLastError());
        GH_CUDA(cudaEventRecord(evB[b], sB));
        GH_CUDA(cudaStreamWaitEvent(sC, evB[b], 0));
        timer.begin(sC);
        key = launch_back<V>(L, sC);
        GH_CUDA(cudaGetLastError());
        timer.end(sC, key, (double)cnt * L.chunk_frames);
        GH_CUDA(cudaEventRecord(evC[b], sC));
        if ((int)evChunk.size() <= i) { cudaEvent_t e; GH_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); evChunk.push_back(e); }
        GH_CUDA(cudaEventRecord(evChunk[i], sC));
        g_launches.fetch_add(2, std::memory_order_relaxed);
      }
      launched_chunks = i;
    } else {
      timer.begin(sC);
      key = launch_back<V>(L, sC);
      GH_CUDA(cudaGetLastError());
      timer.end(sC, key, (double)cnt * frames);
      g_launches.fetch_add(1, std::memory_order_relaxed);
    }
    GH_CUDA(cudaEventRecord(evDoneC, sC));
    GH_CUDA(cudaStreamWaitEvent(parent, evDoneC, 0));
    if (V::FAST) GH_CUDA(cudaStreamWaitEvent(parent, evDoneS, 0));
    if (getenv("GOOEY_B200_TRACE_TYPES")) {      // diagnostic (serialises the buckets): the back end's device time, drum voices on the per-sample kernel
      GH_CUDA(cudaStreamSynchronize(sC)); GH_CUDA(cudaStreamSynchronize(sS));
      std::string per_sample;
      if constexpr (V::FAST) {
        std::vector<uint8_t> mode(cnt);
        GH_CUDA(cudaMemcpy(mode.data(), d_mode.p, cnt, cudaMemcpyDeviceToHost));
        int slow = 0;
        for (uint8_t m : mode) slow += m != 0;
        per_sample = ", " + std::to_string(slow) + " on the per-sample path";
      }
      fprintf(stderr, "[gooey trace]   %s: %d voices x %d frames, back end %.1f ms%s\n", key, cnt, frames, timer.ms(), per_sample.c_str());
    }
  }
};

// Every voice-type bucket of one device-resident set of voices: one TypeRunner per type of Vs, addressed by the
// instrument id of its voices (V::ID).
template <class... Vs> struct VoiceBankOf {
  std::tuple<TypeRunner<Vs>...> runners;
  template <class F> void each(F f) { (f(std::get<TypeRunner<Vs>>(runners)), ...); }
  // f(the runner of instrument `id`); nothing when no type has that id
  template <class F> void with(uint32_t id, F f) { (void)((id == Vs::ID && (f(std::get<TypeRunner<Vs>>(runners)), true)) || ...); }
  void reset() { each([](auto& r) { r.reset(); }); }
  // returns the pool slot of a new voice built from `p`; -1 = bad instrument
  int create(const GooeyVoicePatch& p, float sr) {
    int slot = -1;
    with(p.instrument, [&](auto& r) { slot = r.create(p, sr); });
    return slot;
  }
  void set_mod(const float* planes, long long pitch, int frame0) {
    each([&](auto& r) { r.mod_planes = planes; r.mod_pitch = pitch; r.mod_frame0 = frame0; });
  }
  void add(uint32_t type, uint32_t slot, uint32_t row, const std::vector<gd::VoiceEvent>& ev, const std::vector<gd::ModRoute>* routes = nullptr) {
    with(type, [&](auto& r) { r.add(slot, row, ev, routes); });
  }
  void release(uint32_t type, int slot) { with(type, [&](auto& r) { r.pool.release(slot); }); }
  void launch(cudaStream_t parent, cudaEvent_t start, const gd::RateCtx& rc, const double* tt, int frames, float* out, long long stride) {
    each([&](auto& r) { r.launch(parent, start, rc, tt, frames, out, stride); });
  }
  // call after the launching stream has been synchronised
  void collect_stats() { each([](auto& r) { r.collect_stats(); }); }
  // frames per output chunk of the last launch (identical for every bucket) and the per-chunk completion fence
  int chunk_frames(int frames) const { return TypeRunner<gd::KickV>::chunk_of(frames); }
  void wait_chunk(cudaStream_t s, int i) { each([&](auto& r) { r.wait_chunk(s, i); }); }
};
using VoiceBank = VoiceBankOf<gd::KickV, gd::SnareV, gd::HatV, gd::TomV, gd::BassV, gd::PolyV, gd::GranV>;

}  // namespace gh
