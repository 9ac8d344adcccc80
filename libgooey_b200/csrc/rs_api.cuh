// rs_api.cuh — batches of Rust-API engines (reference: src/engine/mod.rs Engine, src/bounce.rs).
//
// A Rust-API `Engine` is a bag of named instruments, a list of sequencers that name their target instrument, a master
// gain and a global effect chain that defaults to [SoftLimiter(1.0)] (engine/mod.rs:109-128).  Its mono `tick`
// (engine/mod.rs:400-415) is  Σ instruments  -> x master gain -> effects.  `bounce_to_buffer` (bounce.rs:41-59) resets
// and starts the sequencers, snaps the master gain, and calls tick N times with an f64 clock starting at 0.
// Here thousands of such engines are bounced in one pass: the host resolves every sequencer into trigger events, the
// voice kernels render every instrument of every engine, and rs_mix_kernel does the per-engine sum / master / limiter.
// Engines whose chain holds anything but at most RS_MAX_LIM limiters get 0 limiters there, and rs_chain_kernel
// (rs_chain.cuh) runs their whole chain afterwards.
#pragma once
#include "engine.cuh"
#include "rs_chain.cuh"
#include "../../include/gooey_batch.h"

namespace gd {

struct RsMixLaunch {
  const float* voices; long long voice_stride;   // [voice][frame]
  const uint32_t* first_voice;                   // [n_engines + 1]
  const float* master;                           // [n_engines] snapped master gain
  const float* lim_th; const float* lim_inv;     // [n_engines][MAX_LIM] thresholds in chain order
  const uint32_t* n_lim;                         // [n_engines]
  float* out; long long out_stride; int frames; int n_engines;
};
constexpr int RS_MAX_LIM = 4;
static_assert(GOOEY_RS_MAX_EFFECTS == RS_MAX_FX, "the C ABI's chain length is the kernel's");

// One thread per (engine, 4 frames): the voice rows of an engine are summed in insertion order (the reference iterates a
// HashMap, whose order is unspecified), `+ 0.0` for the empty loop mixer, master gain, limiters.
__global__ void __launch_bounds__(256) rs_mix_kernel(const RsMixLaunch L) {
  const int e = blockIdx.y;
  const int f = (blockIdx.x * 256 + threadIdx.x) * 4;
  if (f >= L.frames) return;
  const uint32_t v0 = L.first_voice[e], v1 = L.first_voice[e + 1];
  const float mg = L.master[e];
  const uint32_t nl = L.n_lim[e];
  float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  const bool vec = f + 4 <= L.frames && (L.voice_stride & 3) == 0;
  for (uint32_t v = v0; v < v1; v++) {
    const float* row = L.voices + (long long)v * L.voice_stride + f;
    if (vec) { const float4 x = *reinterpret_cast<const float4*>(row); acc[0] += x.x; acc[1] += x.y; acc[2] += x.z; acc[3] += x.w; }
    else for (int i = 0; i < 4 && f + i < L.frames; i++) acc[i] += row[i];
  }
#pragma unroll
  for (int i = 0; i < 4; i++) {
    float o = acc[i] + 0.0f;
    o *= mg;
    for (uint32_t k = 0; k < nl; k++) o = gm::g_tanhf(o * L.lim_inv[e * RS_MAX_LIM + k]) * L.lim_th[e * RS_MAX_LIM + k];
    acc[i] = o;
  }
  float* dst = L.out + (long long)e * L.out_stride + f;
  if (f + 4 <= L.frames && (L.out_stride & 3) == 0 && (reinterpret_cast<uintptr_t>(L.out) & 15) == 0) *reinterpret_cast<float4*>(dst) = make_float4(acc[0], acc[1], acc[2], acc[3]);
  else for (int i = 0; i < 4 && f + i < L.frames; i++) dst[i] = acc[i];
}

}  // namespace gd

struct GooeyRsBatch {
  int device = 0; float sr = 44100.0f;
  gd::RateCtx rc;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  struct Inst { std::string name; uint32_t type; uint32_t slot; };
  struct Seq { gh::HostSeq seq; std::string target; };
  struct Fx { uint32_t kind; gd::FxDyn init; };                    // the effect as its constructor left it
  struct Eng {
    float bpm = 120.0f;
    std::vector<Inst> insts;
    std::vector<Seq> seqs;
    float master_cur = 0.25f, master_tgt = 0.25f;                 // SmoothedParam(0.25, 0, 2, sr, 30 ms)
    std::vector<Fx> fx;
    uint32_t fresh = 0;                                           // bit k: position k was constructed since it last reached the state pool
    Eng() { const float one = 1.0f; Fx f; f.kind = gd::FXK_LIMITER; gd::rs_fx_construct(f.init, f.kind, &one, 0.0f); fx.push_back(f); fresh = 1; }   // Engine::new pushes SoftLimiter(1.0)
    bool limiter_only() const { if (fx.size() > (size_t)gd::RS_MAX_LIM) return false; for (const Fx& f : fx) if (f.kind != gd::FXK_LIMITER) return false; return true; }
  };
  std::vector<Eng> engines;
  gh::VoiceBank bank;
  gh::ClockWindow clock;
  gh::DevBuf<float> d_voices, d_out, d_master, d_lim_th, d_lim_inv;
  gh::DevBuf<uint32_t> d_first, d_nlim;
  // global effect chains (rs_chain.cuh): the state pool [engine][position] and one ring arena per position, [word][ring_pitch]
  gd::FxGeom geo;
  gh::DevBuf<gd::FxDyn> d_fx_state, d_fx_fresh;
  gh::DevBuf<float> ring[gd::RS_MAX_FX]; uint32_t ring_words[gd::RS_MAX_FX] = {0}; long long ring_pitch = 0;
  gh::DevBuf<uint32_t> d_chain_rows, d_chain_nfx, d_fx_where, d_ring_clear;
  gh::DevBuf<uint8_t> d_chain_kinds;
  gh::KernelTimer chain_timer;                                    // the last bounce's rs_chain_kernel
  // arena `k` grows to `words` words per engine, keeping what it holds
  void ensure_ring(int k, uint32_t words) {
    if (words <= ring_words[k]) return;
    gh::DevBuf<float> nb;
    nb.alloc((size_t)words * (size_t)ring_pitch);
    GH_CUDA(cudaMemsetAsync(nb.p, 0, (size_t)words * (size_t)ring_pitch * 4, stream));
    if (ring_words[k]) GH_CUDA(cudaMemcpyAsync(nb.p, ring[k].p, (size_t)ring_words[k] * (size_t)ring_pitch * 4, cudaMemcpyDeviceToDevice, stream));
    GH_CUDA(cudaStreamSynchronize(stream));
    std::swap(ring[k].p, nb.p); std::swap(ring[k].n, nb.n);
    ring_words[k] = words;
  }
  ~GooeyRsBatch() {
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    if (stream) cudaStreamDestroy(stream);
  }
};

namespace gh {

// Lays out the chain engines for rs_chain_kernel (warps of one signature, padded with ~0u), grows the ring arenas to
// the kinds each position holds, and moves the effects constructed since the last bounce into the state pool with
// their ring columns zeroed.  Returns the number of warps (0: no engine has a chain beyond limiters).
static uint32_t chain_prepare(GooeyRsBatch* b, const std::map<std::vector<uint8_t>, std::vector<uint32_t>>& chains) {
  if (chains.empty()) return 0;
  cudaStream_t st = b->stream;
  const uint32_t ne = (uint32_t)b->engines.size();
  if (!b->d_fx_state.p) {
    b->ring_pitch = (((long long)ne + 31) / 32) * 32;
    if ((b->ring_pitch / 32) % 2 == 0) b->ring_pitch += 32;        // odd multiple of 32 (DESIGN §3)
    b->d_fx_state.alloc((size_t)ne * gd::RS_MAX_FX);
    b->geo = make_fx_geom(b->sr);
  }
  std::vector<uint32_t> rows, nfx, where;
  std::vector<uint8_t> kinds;
  std::vector<gd::FxDyn> fresh;
  std::vector<uint32_t> need(gd::RS_MAX_FX, 0);
  std::vector<std::vector<uint32_t>> clear(gd::RS_MAX_FX);
  for (const auto& c : chains) {
    const std::vector<uint8_t>& sig = c.first;
    for (size_t k = 0; k < sig.size(); k++) need[k] = std::max(need[k], gd::rs_fx_ring_words(b->geo, sig[k]));
    for (size_t i = 0; i < c.second.size(); i += 32) {
      for (size_t j = 0; j < 32; j++) rows.push_back(i + j < c.second.size() ? c.second[i + j] : ~0u);
      nfx.push_back((uint32_t)sig.size());
      for (int k = 0; k < gd::RS_MAX_FX; k++) kinds.push_back(k < (int)sig.size() ? sig[k] : (uint8_t)gd::FXK_NONE);
    }
    for (uint32_t e : c.second) {
      GooeyRsBatch::Eng& E = b->engines[e];
      for (size_t k = 0; k < E.fx.size(); k++) {
        if (!((E.fresh >> k) & 1u)) continue;
        fresh.push_back(E.fx[k].init);
        where.push_back(e * gd::RS_MAX_FX + (uint32_t)k);
        if (gd::rs_fx_ring_words(b->geo, E.fx[k].kind)) clear[k].push_back(e);
      }
      E.fresh = 0;
    }
  }
  for (int k = 0; k < gd::RS_MAX_FX; k++) b->ensure_ring(k, need[k]);
  for (int k = 0; k < gd::RS_MAX_FX; k++) {
    if (clear[k].empty()) continue;
    b->d_ring_clear.upload(clear[k].data(), clear[k].size(), st);
    const int n = (int)clear[k].size();
    ring_clear_kernel<<<dim3((n + 127) / 128, std::min<uint32_t>(b->ring_words[k], 4096u)), 128, 0, st>>>(b->ring[k].p, b->ring_pitch, b->ring_words[k], b->d_ring_clear.p, n);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    GH_CUDA(cudaGetLastError());
    GH_CUDA(cudaStreamSynchronize(st));     // d_ring_clear is reused by the next position
  }
  if (!fresh.empty()) {
    b->d_fx_fresh.upload(fresh.data(), fresh.size(), st);
    b->d_fx_where.upload(where.data(), where.size(), st);
    const int n = (int)fresh.size();
    gd::rs_fx_init_launch(b->d_fx_state.p, b->d_fx_fresh.p, b->d_fx_where.p, n, st);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    GH_CUDA(cudaGetLastError());
  }
  b->d_chain_rows.upload(rows.data(), rows.size(), st);
  b->d_chain_nfx.upload(nfx.data(), nfx.size(), st);
  b->d_chain_kinds.upload(kinds.data(), kinds.size(), st);
  return (uint32_t)nfx.size();
}

static void rs_bounce_impl(GooeyRsBatch* b, uint32_t frames, float* out_dev, size_t out_stride) {
  use_device(b->device);
  cudaStream_t st = b->stream;
  const uint32_t ne = (uint32_t)b->engines.size();
  const double* tt = b->clock.view(clock_table(b->sr), 0, frames, st);
  b->bank.reset();
  std::vector<uint32_t> first(ne + 1, 0), nlim(ne);
  std::vector<float> master(ne), lth((size_t)ne * gd::RS_MAX_LIM, 1.0f), linv((size_t)ne * gd::RS_MAX_LIM, 1.0f);
  std::vector<SeqFire> fires;
  std::map<std::vector<uint8_t>, std::vector<uint32_t>> chains;   // chain signature -> its engines
  uint32_t row = 0;
  for (uint32_t e = 0; e < ne; e++) {
    GooeyRsBatch::Eng& E = b->engines[e];
    first[e] = row;
    // prepare_for_bounce (engine/mod.rs:464-477): sequencers reset + start, master gain snapped; the effects are left as they are
    E.master_cur = E.master_tgt;
    master[e] = E.master_cur;
    if (E.limiter_only()) {
      nlim[e] = (uint32_t)E.fx.size();
      for (size_t k = 0; k < E.fx.size(); k++) { memcpy(&lth[e * gd::RS_MAX_LIM + k], &E.fx[k].init.w[0], 4); memcpy(&linv[e * gd::RS_MAX_LIM + k], &E.fx[k].init.w[1], 4); }
    } else {
      nlim[e] = 0;
      std::vector<uint8_t> sig;
      for (const auto& f : E.fx) sig.push_back((uint8_t)f.kind);
      chains[sig].push_back(e);
    }
    std::vector<std::vector<gd::VoiceEvent>> ev(E.insts.size());
    for (auto& x : ev) x.push_back(make_event(0, gd::EV_SET_TIME, 0, 0.0f, 0));
    for (auto& s : E.seqs) {
      s.seq.reset(); s.seq.start();
      fires.clear();
      s.seq.run(frames, fires);
      s.seq.stop();
      for (size_t i = 0; i < E.insts.size(); i++) {
        if (E.insts[i].name != s.target) continue;
        for (const SeqFire& f : fires) ev[i].push_back(make_event(f.frame, gd::EV_TRIGGER, 0, f.velocity));
      }
    }
    for (size_t i = 0; i < E.insts.size(); i++) {
      std::stable_sort(ev[i].begin(), ev[i].end(), [](const gd::VoiceEvent& a, const gd::VoiceEvent& c) { return a.frame < c.frame; });
      b->bank.add(E.insts[i].type, E.insts[i].slot, row++, ev[i]);
    }
  }
  first[ne] = row;
  const size_t vstride = ((size_t)frames + 3) & ~(size_t)3;
  b->d_voices.alloc(std::max<size_t>((size_t)row * vstride, 4));
  b->d_first.upload(first.data(), first.size(), st);
  b->d_nlim.upload(nlim.data(), nlim.size(), st);
  b->d_master.upload(master.data(), master.size(), st);
  b->d_lim_th.upload(lth.data(), lth.size(), st);
  b->d_lim_inv.upload(linv.data(), linv.size(), st);
  const uint32_t n_chain_warps = chain_prepare(b, chains);
  GH_CUDA(cudaStreamSynchronize(st));   // the host vectors above are temporaries
  GH_CUDA(cudaEventRecord(b->ev0, st));
  b->bank.launch(st, b->ev0, b->rc, tt, (int)frames, b->d_voices.p, (long long)vstride);
  gd::RsMixLaunch M;
  M.voices = b->d_voices.p; M.voice_stride = (long long)vstride; M.first_voice = b->d_first.p; M.master = b->d_master.p;
  M.lim_th = b->d_lim_th.p; M.lim_inv = b->d_lim_inv.p; M.n_lim = b->d_nlim.p;
  M.out = out_dev; M.out_stride = (long long)out_stride; M.frames = (int)frames; M.n_engines = (int)ne;
  dim3 grid((frames + 1023) / 1024, ne);
  gd::rs_mix_kernel<<<grid, 256, 0, st>>>(M);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  GH_CUDA(cudaGetLastError());
  b->chain_timer.clear();
  if (n_chain_warps) {
    gd::RsChainLaunch C;
    C.out = out_dev; C.out_stride = (long long)out_stride; C.frames = (int)frames;
    C.rows = b->d_chain_rows.p; C.warp_kinds = b->d_chain_kinds.p; C.warp_nfx = b->d_chain_nfx.p;
    C.state = b->d_fx_state.p;
    for (int k = 0; k < gd::RS_MAX_FX; k++) C.ring[k] = b->ring[k].p;
    C.ring_pitch = b->ring_pitch; C.rc = b->rc; C.geo = b->geo;
    size_t n = 0;
    for (const auto& c : chains) n += c.second.size();
    b->chain_timer.begin(st);
    gd::rs_chain_launch(C, n_chain_warps, st);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    GH_CUDA(cudaGetLastError());
    b->chain_timer.end(st, "rs_chain_kernel", (double)n * frames);
  }
  GH_CUDA(cudaEventRecord(b->ev1, st));
}

}  // namespace gh

extern "C" {

int gooey_rs_batch_new(float sample_rate, uint32_t n_engines, int device, GooeyRsBatch** out_batch) {
  GOOEY_TRY
  if (!out_batch) { set_error("null argument"); return GOOEY_E_INVALID; }
  *out_batch = nullptr;
  if (!(sample_rate > 0.0f)) { set_error("sample_rate must be > 0"); return GOOEY_E_INVALID; }
  use_device(device);
  std::unique_ptr<GooeyRsBatch> b(new GooeyRsBatch);
  b->device = device; b->sr = sample_rate; b->rc = gd::make_rate_ctx(sample_rate);
  b->engines.resize(n_engines);
  GH_CUDA(cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking));
  GH_CUDA(cudaEventCreate(&b->ev0));
  GH_CUDA(cudaEventCreate(&b->ev1));
  *out_batch = b.release();
  return GOOEY_E_OK;
  GOOEY_CATCH
}
void gooey_rs_batch_free(GooeyRsBatch* b) {
  if (!b) return;
  cudaSetDevice(b->device);
  cudaDeviceSynchronize();
  delete b;
}
#define RS_ENGINE(b, e) if (!(b) || (e) >= (b)->engines.size()) { set_error("bad batch/engine"); return GOOEY_E_INVALID; } GooeyRsBatch::Eng& E = (b)->engines[e]
int gooey_rs_batch_add_instrument(GooeyRsBatch* b, uint32_t engine, const char* name, const GooeyVoicePatch* patch) {
  GOOEY_TRY
  RS_ENGINE(b, engine);
  if (!name || !patch) { set_error("null argument"); return GOOEY_E_INVALID; }
  use_device(b->device);
  const int slot = b->bank.create(*patch, b->sr);
  if (slot < 0) { set_error("unsupported instrument id in voice patch"); return GOOEY_E_INVALID; }
  // HashMap::insert semantics: a second instrument under the same name replaces the first (engine/mod.rs:190-192)
  for (auto& i : E.insts) if (i.name == name) { b->bank.release(i.type, (int)i.slot); i.type = patch->instrument; i.slot = (uint32_t)slot; return GOOEY_E_OK; }
  E.insts.push_back({name, patch->instrument, (uint32_t)slot});
  return GOOEY_E_OK;
  GOOEY_CATCH
}
int gooey_rs_batch_add_sequencer(GooeyRsBatch* b, uint32_t engine, const char* instrument_name, float bpm, const uint8_t* enabled, const float* velocity,
                                 uint32_t steps) {
  GOOEY_TRY
  RS_ENGINE(b, engine);
  if (!instrument_name || (!enabled && steps)) { set_error("null argument"); return GOOEY_E_INVALID; }
  GooeyRsBatch::Seq s;
  s.seq.init(bpm, b->sr);
  s.seq.pattern.assign(steps, SeqStep());
  for (uint32_t i = 0; i < steps; i++) { s.seq.pattern[i].enabled = enabled[i] != 0; s.seq.pattern[i].velocity = velocity ? gd::clampf(velocity[i], 0.0f, 1.0f) : 1.0f; }
  s.target = instrument_name;
  E.seqs.push_back(std::move(s));
  return GOOEY_E_OK;
  GOOEY_CATCH
}
int gooey_rs_batch_set_bpm(GooeyRsBatch* b, uint32_t engine, float bpm) { GOOEY_TRY RS_ENGINE(b, engine); E.bpm = bpm; return GOOEY_E_OK; GOOEY_CATCH }
float gooey_rs_batch_get_bpm(const GooeyRsBatch* b, uint32_t engine) { return (b && engine < b->engines.size()) ? b->engines[engine].bpm : 120.0f; }
int gooey_rs_batch_set_master_gain(GooeyRsBatch* b, uint32_t engine, float gain) {
  GOOEY_TRY
  RS_ENGINE(b, engine);
  const float c = gd::clampf(gain, 0.0f, 2.0f);
  if (fabsf(E.master_tgt - c) > 1e-8f) E.master_tgt = c;      // SmoothedParam::set_target
  return GOOEY_E_OK;
  GOOEY_CATCH
}
int gooey_rs_batch_clear_global_effects(GooeyRsBatch* b, uint32_t engine) { GOOEY_TRY RS_ENGINE(b, engine); E.fx.clear(); E.fresh = 0; return GOOEY_E_OK; GOOEY_CATCH }
int gooey_rs_batch_add_effect(GooeyRsBatch* b, uint32_t engine, uint32_t effect_id, const float* args, uint32_t n_args) {
  GOOEY_TRY
  RS_ENGINE(b, engine);
  if (effect_id >= 10) { set_error("unknown global effect id"); return GOOEY_E_INVALID; }
  if (n_args != gd::RS_FX_ARGS[effect_id]) { set_error("wrong number of constructor arguments for this global effect"); return GOOEY_E_INVALID; }
  if (!args && n_args) { set_error("null argument"); return GOOEY_E_INVALID; }
  if (E.fx.size() >= (size_t)gd::RS_MAX_FX) { set_error("too many global effects"); return GOOEY_E_INVALID; }
  GooeyRsBatch::Fx f;
  f.kind = effect_id;
  gd::rs_fx_construct(f.init, effect_id, args, b->sr);
  E.fresh |= 1u << E.fx.size();
  E.fx.push_back(f);
  return GOOEY_E_OK;
  GOOEY_CATCH
}
int gooey_rs_batch_add_limiter(GooeyRsBatch* b, uint32_t engine, float threshold) { return gooey_rs_batch_add_effect(b, engine, gd::FXK_LIMITER, &threshold, 1); }
int gooey_rs_batch_bounce_device(GooeyRsBatch* b, uint32_t samples, float* out_dev, size_t stride) {
  GOOEY_TRY
  if (!b || !out_dev || stride < samples) { set_error("bad arguments"); return GOOEY_E_INVALID; }
  if (samples == 0 || b->engines.empty()) return GOOEY_E_OK;
  rs_bounce_impl(b, samples, out_dev, stride);
  GH_CUDA(cudaStreamSynchronize(b->stream));
  GH_CUDA(cudaEventElapsedTime(&gh::g_last_kernel_ms, b->ev0, b->ev1));
  b->chain_timer.collect();
  return GOOEY_E_OK;
  GOOEY_CATCH
}
int gooey_rs_batch_bounce(GooeyRsBatch* b, uint32_t samples, float* out_host) {
  GOOEY_TRY
  if (!b || !out_host) { set_error("bad arguments"); return GOOEY_E_INVALID; }
  if (samples == 0 || b->engines.empty()) return GOOEY_E_OK;
  use_device(b->device);
  const size_t stride = ((size_t)samples + 3) & ~(size_t)3;
  b->d_out.alloc(b->engines.size() * stride);
  rs_bounce_impl(b, samples, b->d_out.p, stride);
  GH_CUDA(cudaMemcpy2DAsync(out_host, (size_t)samples * 4, b->d_out.p, stride * 4, (size_t)samples * 4, b->engines.size(), cudaMemcpyDeviceToHost, b->stream));
  GH_CUDA(cudaStreamSynchronize(b->stream));
  GH_CUDA(cudaEventElapsedTime(&gh::g_last_kernel_ms, b->ev0, b->ev1));
  b->chain_timer.collect();
  return GOOEY_E_OK;
  GOOEY_CATCH
}
#undef RS_ENGINE

// ---- WAV output (bounce.rs:80-133, ffi.rs:7942-7980): mono PCM, `(s * scale).round() as iN` (round half away from zero,
// saturating cast), 16- or 24-bit little endian in a canonical 44-byte RIFF header (what hound writes for PCM). ----
int gooey_b200_write_wav(const char* utf8_path, const float* samples, uint32_t n, uint32_t sample_rate, uint32_t bit_depth) {
  GOOEY_TRY
  if (!utf8_path || (!samples && n)) { set_error("null argument"); return GOOEY_E_INVALID; }
  if (bit_depth != 16 && bit_depth != 24) { set_error("Unsupported bit depth. Use 16 or 24."); return GOOEY_E_INVALID; }
  const uint32_t bps = bit_depth / 8;
  const uint64_t data_bytes = (uint64_t)n * bps;
  if (data_bytes + 36 > 0xffffffffull) { set_error("WAV too large"); return GOOEY_E_INVALID; }
  FILE* f = fopen(utf8_path, "wb");
  if (!f) { set_error("Failed to create WAV"); return GOOEY_E_INVALID; }
  std::vector<uint8_t> buf;
  buf.reserve(44 + (size_t)data_bytes);
  auto u32 = [&](uint32_t v) { for (int i = 0; i < 4; i++) buf.push_back((uint8_t)(v >> (8 * i))); };
  auto u16 = [&](uint32_t v) { buf.push_back((uint8_t)v); buf.push_back((uint8_t)(v >> 8)); };
  buf.insert(buf.end(), {'R', 'I', 'F', 'F'}); u32((uint32_t)(36 + data_bytes)); buf.insert(buf.end(), {'W', 'A', 'V', 'E', 'f', 'm', 't', ' '});
  u32(16); u16(1); u16(1); u32(sample_rate); u32(sample_rate * bps); u16(bps); u16(bit_depth);
  buf.insert(buf.end(), {'d', 'a', 't', 'a'}); u32((uint32_t)data_bytes);
  const float scale = bit_depth == 16 ? 32767.0f : 8388607.0f;
  for (uint32_t i = 0; i < n; i++) {
    const float r = roundf(samples[i] * scale);          // f32::round: half away from zero
    int32_t q;                                           // `as i16` / `as i32`: saturating, NaN -> 0
    if (std::isnan(r)) q = 0;
    else if (bit_depth == 16) q = r >= 32767.0f ? 32767 : (r <= -32768.0f ? -32768 : (int32_t)r);
    else q = r >= 2147483648.0f ? 2147483647 : (r <= -2147483648.0f ? (int32_t)0x80000000u : (int32_t)r);   // hound then keeps the low 24 bits
    for (uint32_t k = 0; k < bps; k++) buf.push_back((uint8_t)((uint32_t)q >> (8 * k)));
  }
  const bool ok = fwrite(buf.data(), 1, buf.size(), f) == buf.size();
  const bool closed = fclose(f) == 0;
  if (!ok || !closed) { set_error("Failed to write sample"); return GOOEY_E_INVALID; }
  return GOOEY_E_OK;
  GOOEY_CATCH
}
// 32-bit float WAV (the format of ffi.rs:8030-8048 / tests/loop_render_wav.rs: WAVE_FORMAT_IEEE_FLOAT, `channels` interleaved)
int gooey_b200_write_wav_f32(const char* utf8_path, const float* interleaved, uint32_t frames, uint32_t channels, uint32_t sample_rate) {
  if (!utf8_path || (!interleaved && frames) || channels == 0 || channels > 2) { set_error("bad arguments"); return GOOEY_E_INVALID; }
  const uint64_t data_bytes = (uint64_t)frames * channels * 4;
  if (data_bytes + 36 > 0xffffffffull) { set_error("WAV too large"); return GOOEY_E_INVALID; }
  FILE* f = fopen(utf8_path, "wb");
  if (!f) { set_error("Failed to create WAV"); return GOOEY_E_INVALID; }
  uint8_t h[44];
  auto u32 = [&](int o, uint32_t v) { for (int i = 0; i < 4; i++) h[o + i] = (uint8_t)(v >> (8 * i)); };
  auto u16 = [&](int o, uint32_t v) { h[o] = (uint8_t)v; h[o + 1] = (uint8_t)(v >> 8); };
  memcpy(h, "RIFF", 4); u32(4, (uint32_t)(36 + data_bytes)); memcpy(h + 8, "WAVEfmt ", 8);
  u32(16, 16); u16(20, 3); u16(22, channels); u32(24, sample_rate); u32(28, sample_rate * channels * 4); u16(32, channels * 4); u16(34, 32);
  memcpy(h + 36, "data", 4); u32(40, (uint32_t)data_bytes);
  const size_t n = (size_t)frames * channels;
  const bool ok = fwrite(h, 1, 44, f) == 44 && fwrite(interleaved, 4, n, f) == n;      // little-endian host
  const bool closed = fclose(f) == 0;
  if (!ok || !closed) { set_error("Failed to write sample"); return GOOEY_E_INVALID; }
  return GOOEY_E_OK;
}
// 16-bit mono WAV from samples that are already PCM (the device-quantised drain)
static int write_wav_pcm16(const char* utf8_path, const int16_t* pcm, uint32_t n, uint32_t sample_rate) {
  const uint64_t data_bytes = (uint64_t)n * 2;
  if (data_bytes + 36 > 0xffffffffull) { set_error("WAV too large"); return GOOEY_E_INVALID; }
  FILE* f = fopen(utf8_path, "wb");
  if (!f) { set_error("Failed to create WAV"); return GOOEY_E_INVALID; }
  uint8_t h[44];
  auto u32 = [&](int o, uint32_t v) { for (int i = 0; i < 4; i++) h[o + i] = (uint8_t)(v >> (8 * i)); };
  auto u16 = [&](int o, uint32_t v) { h[o] = (uint8_t)v; h[o + 1] = (uint8_t)(v >> 8); };
  memcpy(h, "RIFF", 4); u32(4, (uint32_t)(36 + data_bytes)); memcpy(h + 8, "WAVEfmt ", 8);
  u32(16, 16); u16(20, 1); u16(22, 1); u32(24, sample_rate); u32(28, sample_rate * 2); u16(32, 2); u16(34, 16);
  memcpy(h + 36, "data", 4); u32(40, (uint32_t)data_bytes);
  const bool ok = fwrite(h, 1, 44, f) == 44 && fwrite(pcm, 2, n, f) == n;      // little-endian host (x86-64 / aarch64)
  const bool closed = fclose(f) == 0;
  if (!ok || !closed) { set_error("Failed to write sample"); return GOOEY_E_INVALID; }
  return GOOEY_E_OK;
}
int gooey_batch_bounce_to_wav(GooeyEngine* const* engines, uint32_t n, uint32_t bars, const char* const* utf8_paths) {
  if (!engines || !utf8_paths) { set_error("null argument"); return GOOEY_E_INVALID; }
  for (uint32_t i = 0; i < n; i++) if (!engines[i] || !utf8_paths[i]) { set_error("null engine / path in batch"); return GOOEY_E_INVALID; }
  // engines whose tempo gives a different length are bounced as separate groups
  std::map<uint32_t, std::vector<uint32_t>> groups;
  for (uint32_t i = 0; i < n; i++) groups[gh::bounce_frames(engines[i], bars)].push_back(i);
  for (auto& g : groups) {
    const uint32_t frames = g.first;
    std::vector<GooeyEngine*> E;
    for (uint32_t i : g.second) E.push_back(engines[i]);
    std::vector<int16_t> pcm((size_t)E.size() * std::max<uint32_t>(frames, 1));
    if (frames > 0) {
      const int rc = gooey_batch_bounce_pcm16(E.data(), (uint32_t)E.size(), bars, pcm.data(), frames, nullptr);
      if (rc != GOOEY_E_OK) return rc;
    }
    for (size_t k = 0; k < E.size(); k++) {
      const int rc = write_wav_pcm16(utf8_paths[g.second[k]], pcm.data() + k * frames, frames, (uint32_t)gd::f32_to_u64_sat(E[k]->sr));
      if (rc != GOOEY_E_OK) return rc;
    }
  }
  return GOOEY_E_OK;
}
bool gooey_engine_bounce_to_wav(GooeyEngine* e, uint32_t bars, const char* utf8_path) {   // ffi.rs:7942-7980
  if (!e || !utf8_path) return false;
  uint32_t n = 0;
  float* buf = gooey_engine_bounce_to_buffer(e, bars, &n);
  if (!buf) return false;
  const int rc = gooey_b200_write_wav(utf8_path, buf, n, (uint32_t)gd::f32_to_u64_sat(e->sr), 16);
  gooey_engine_free_buffer(buf, n);
  return rc == GOOEY_E_OK;
}

}  // extern "C"
