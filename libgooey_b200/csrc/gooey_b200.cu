// gooey_b200.cu — libgooey_b200.so: the C ABI (include/gooey_batch.h, include/gooey.h)
// over the sm_100a kernels.  The kernels are header templates (kernels.cuh); this file instantiates them and owns the
// host side.  The Rust-API effect chain's kernels and the poly synth's warp-per-voice kernel are compiled apart, in
// rs_chain.cu and poly_wave.cu.
#include <mutex>
#include <memory>
#include "pool.cuh"
#include "halfband_design.h"
#include "rs_chain.cuh"
#include "poly_wave.cuh"

namespace gh {

std::string& last_error() { static thread_local std::string e; return e; }
std::atomic<uint64_t> g_launches{0};
static float g_last_kernel_ms = 0.0f;
std::map<std::string, KernelStat>& kernel_stats() { static std::map<std::string, KernelStat> m; return m; }
std::mutex& kernel_stats_mutex() { static std::mutex m; return m; }

ClockTable& clock_table(float sr) {
  static std::mutex mu;
  static std::map<uint32_t, ClockTable*> tables;
  std::lock_guard<std::mutex> lk(mu);
  uint32_t key; memcpy(&key, &sr, 4);
  auto it = tables.find(key);
  if (it == tables.end()) {
    ClockTable* t = new ClockTable();
    t->dt = 1.0 / (double)sr;
    it = tables.emplace(key, t).first;
  }
  return *it->second;
}

// One hardware work queue per stream: the render uses up to 3 streams per voice type plus a copy stream, and with the
// default of 8 connections independent launches alias onto the same queue and serialise.  Read by the driver when the
// context is created, so it is set when the library is loaded (never overriding the host's own choice).
static const int g_conn_env = setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);

// ---- device bring-up --------------------------------------------------------------------------
static std::mutex g_dev_mutex;
static std::vector<char> g_dev_ready;

static int device_count() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

// Select `device` and make sure its constant memory holds the half-band coefficients.
static void use_device(int device) {
  int n = device_count();
  if (n <= 0) throw CudaError("no CUDA device visible: libgooey_b200 has no CPU fallback");
  if (device < 0 || device >= n) throw CudaError("device index out of range");
  GH_CUDA(cudaSetDevice(device));
  std::lock_guard<std::mutex> lk(g_dev_mutex);
  if ((int)g_dev_ready.size() < n) g_dev_ready.resize(n, 0);
  if (!g_dev_ready[device]) {
    float hb[8];
    gd::design_halfband8(hb);
    GH_CUDA(cudaMemcpyToSymbol(gd::c_hb, hb, sizeof hb));
    gd::rs_chain_set_halfband(hb);
    {
      static float inv_sq[gd::INV_SQ_N];
      for (int k = 0; k < gd::INV_SQ_N; k++) { volatile float fi = (float)(2 * k + 1); volatile float sq = fi * fi; inv_sq[k] = 1.0f / sq; }
      GH_CUDA(cudaMemcpyToSymbol(gd::c_inv_sq, inv_sq, sizeof inv_sq));
    }
    double mf[128];   // music/note.rs:81-83 midi_to_freq in f64, with the platform libm
    for (int n = 0; n < 128; n++) mf[n] = 440.0 * pow(2.0, ((double)n - 69.0) / 12.0);
    GH_CUDA(cudaMemcpyToSymbol(gd::c_midi_freq, mf, sizeof mf));
    gd::poly_wave_set_midi_freq(mf);
    g_dev_ready[device] = 1;
  }
}

}  // namespace gh

using namespace gh;

// =================================================================================================
// Voice batch
// =================================================================================================
namespace gh {
// A granulator's source buffer as the host hands it to the device: shared by every voice that plays it.
struct GranSource { std::shared_ptr<DevBuf<float>> buf; uint32_t len = 0; float sr = 0.0f; };
}  // namespace gh

struct GooeyVoiceBatch {
  int device = 0;
  float sr = 44100.0f;
  gd::RateCtx rc;
  cudaStream_t stream = nullptr, copy_stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  uint32_t n = 0;
  uint32_t k = 0;                        // engine clock index of the next frame (shared by every voice of the batch)
  gh::ClockWindow clock;
  std::vector<uint8_t> vtype;
  std::vector<uint32_t> vslot;
  std::vector<std::vector<gd::VoiceEvent>> pending;   // per voice, frames relative to the next render
  // Granulator sources per voice.  A buffer stays alive while the device state points at it (gran_live) or a queued
  // EV_GRAN_BUFFER names it (gran_queued, frames relative to the next render, in call order); gran_latest is the buffer
  // of the most recent set_buffer / share_buffer call, which share_buffer hands on.
  std::vector<gh::GranSource> gran_live, gran_latest;
  std::vector<std::vector<std::pair<uint32_t, gh::GranSource>>> gran_queued;
  std::vector<gh::GranSource> gran_retired;           // replaced during the last render: freed when the next one starts
  VoiceBank bank;
  DevBuf<float> d_out;
  DevBuf<int16_t> d_pcm;
  ~GooeyVoiceBatch() {
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    if (stream) cudaStreamDestroy(stream);
    if (copy_stream) cudaStreamDestroy(copy_stream);
  }
};

namespace gh {

static void voice_batch_render_impl(GooeyVoiceBatch* b, uint32_t frames, float* out_dev, size_t stride) {
  use_device(b->device);
  cudaStream_t st = b->stream;
  if ((uint64_t)b->k + frames >= 0xffffffffull) throw std::runtime_error("engine clock index overflow");
  const double* tt = b->clock.view(clock_table(b->sr), b->k, (uint64_t)b->k + frames, st);
  b->gran_retired.clear();                           // every render call has synchronised its stream before returning
  b->bank.reset();
  std::vector<gd::VoiceEvent> now, later;
  for (uint32_t v = 0; v < b->n; v++) {
    auto& ev = b->pending[v];
    std::stable_sort(ev.begin(), ev.end(), [](const gd::VoiceEvent& a, const gd::VoiceEvent& c) { return a.frame < c.frame; });
    now.clear(); later.clear();
    for (auto& e : ev) { if (e.frame < frames) now.push_back(e); else { e.frame -= frames; later.push_back(e); } }
    b->bank.add(b->vtype[v], b->vslot[v], v, now);
    ev = later;
    if (!b->gran_queued.empty() && !b->gran_queued[v].empty()) {   // sources whose EV_GRAN_BUFFER this call applies
      auto& q = b->gran_queued[v];
      std::stable_sort(q.begin(), q.end(), [](const std::pair<uint32_t, GranSource>& a, const std::pair<uint32_t, GranSource>& c) { return a.first < c.first; });
      std::vector<std::pair<uint32_t, GranSource>> keep;
      for (auto& e : q) {
        if (e.first >= frames) { keep.emplace_back(e.first - frames, e.second); continue; }
        if (b->gran_live[v].buf) b->gran_retired.push_back(b->gran_live[v]);   // still read before the event's frame
        b->gran_live[v] = e.second;
      }
      q.swap(keep);
    }
  }
  GH_CUDA(cudaEventRecord(b->ev0, st));
  b->bank.launch(st, b->ev0, b->rc, tt, (int)frames, out_dev, (long long)stride);
  GH_CUDA(cudaEventRecord(b->ev1, st));
  b->k += frames;
}

}  // namespace gh

#define GOOEY_TRY try {
#define GOOEY_CATCH                                                              \
  } catch (const gh::CudaError& e) { gh::set_error(e.what());                    \
    return std::string(e.what()).find("no CUDA device") != std::string::npos ? GOOEY_E_NO_DEVICE : GOOEY_E_CUDA; \
  } catch (const std::exception& e) { gh::set_error(e.what()); return GOOEY_E_INVALID; }

extern "C" {

const char* gooey_b200_last_error(void) { return gh::last_error().c_str(); }
int gooey_b200_device_count(void) { return gh::device_count(); }
uint64_t gooey_b200_launch_count(void) { return gh::g_launches.load(); }
float gooey_b200_last_kernel_ms(void) { return gh::g_last_kernel_ms; }
int gooey_b200_kernel_stat(const char* kernel, uint64_t* launches, double* total_ms, double* voice_frames) {
  if (!kernel) return GOOEY_E_INVALID;
  std::lock_guard<std::mutex> lk(gh::kernel_stats_mutex());
  auto it = gh::kernel_stats().find(kernel);
  gh::KernelStat k = it == gh::kernel_stats().end() ? gh::KernelStat() : it->second;
  if (launches) *launches = k.launches;
  if (total_ms) *total_ms = k.ms;
  if (voice_frames) *voice_frames = k.voice_frames;
  return GOOEY_E_OK;
}
const char* gooey_b200_kernel_stat_names(void) {
  static thread_local std::string names;
  std::lock_guard<std::mutex> lk(gh::kernel_stats_mutex());
  names.clear();
  for (const auto& kv : gh::kernel_stats()) { if (!names.empty()) names += ';'; names += kv.first; }
  return names.c_str();
}
void gooey_b200_kernel_stats_reset(void) { std::lock_guard<std::mutex> lk(gh::kernel_stats_mutex()); gh::kernel_stats().clear(); }

int gooey_voice_batch_new(float sample_rate, uint32_t n_voices, const GooeyVoicePatch* patches, int device, GooeyVoiceBatch** out_batch) {
  GOOEY_TRY
  if (!out_batch || (!patches && n_voices)) { set_error("null argument"); return GOOEY_E_INVALID; }
  *out_batch = nullptr;
  if (!(sample_rate > 0.0f)) { set_error("sample_rate must be > 0"); return GOOEY_E_INVALID; }
  use_device(device);
  std::unique_ptr<GooeyVoiceBatch> b(new GooeyVoiceBatch);
  b->device = device; b->sr = sample_rate; b->n = n_voices;
  b->rc = gd::make_rate_ctx(sample_rate);
  GH_CUDA(cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking));
  GH_CUDA(cudaStreamCreateWithFlags(&b->copy_stream, cudaStreamNonBlocking));
  GH_CUDA(cudaEventCreate(&b->ev0));
  GH_CUDA(cudaEventCreate(&b->ev1));
  b->vtype.resize(n_voices); b->vslot.resize(n_voices); b->pending.resize(n_voices);
  b->gran_live.resize(n_voices); b->gran_latest.resize(n_voices); b->gran_queued.resize(n_voices);
  for (uint32_t v = 0; v < n_voices; v++) {
    int slot = b->bank.create(patches[v], sample_rate);
    if (slot < 0) { set_error("unsupported instrument id in voice patch"); return GOOEY_E_INVALID; }
    b->vtype[v] = (uint8_t)patches[v].instrument;
    b->vslot[v] = (uint32_t)slot;
  }
  *out_batch = b.release();
  return GOOEY_E_OK;
  GOOEY_CATCH
}

void gooey_voice_batch_free(GooeyVoiceBatch* b) {
  if (!b) return;
  cudaSetDevice(b->device);
  cudaDeviceSynchronize();
  delete b;
}

int gooey_voice_batch_trigger(GooeyVoiceBatch* b, uint32_t voice, uint32_t frame, float velocity) {
  GOOEY_TRY
  if (!b || voice >= b->n) { set_error("bad batch/voice"); return GOOEY_E_INVALID; }
  b->pending[voice].push_back(make_event(frame, gd::EV_TRIGGER, 0, velocity));
  return GOOEY_E_OK;
  GOOEY_CATCH
}

int gooey_voice_batch_trigger_all(GooeyVoiceBatch* b, uint32_t frame, const float* velocities) {
  GOOEY_TRY
  if (!b) { set_error("null batch"); return GOOEY_E_INVALID; }
  for (uint32_t v = 0; v < b->n; v++) b->pending[v].push_back(make_event(frame, gd::EV_TRIGGER, 0, velocities ? velocities[v] : 1.0f));
  return GOOEY_E_OK;
  GOOEY_CATCH
}

int gooey_voice_batch_set_param(GooeyVoiceBatch* b, uint32_t voice, uint32_t frame, uint32_t param, float value, int snap) {
  GOOEY_TRY
  if (!b || voice >= b->n) { set_error("bad batch/voice"); return GOOEY_E_INVALID; }
  bool known = ffi_param_to_events(b->vtype[voice], param, value,
                                   [&](uint32_t kind, uint32_t p, float v) { b->pending[voice].push_back(make_event(frame, kind, p, v)); });
  if (known && snap) b->pending[voice].push_back(make_event(frame, gd::EV_SNAP, 0, 0.0f));
  return GOOEY_E_OK;
  GOOEY_CATCH
}

// ---- poly synth and granulator voices: the events of PolySynth::trigger_note / release_all and Granulator::set_buffer /
// set_seed.  A refused call queues nothing.
static int voice_of_kind(GooeyVoiceBatch* b, uint32_t voice, uint32_t kind, const char* what) {
  if (!b || voice >= b->n) { set_error("bad batch/voice"); return GOOEY_E_INVALID; }
  if (b->vtype[voice] != kind) {
    set_error(std::string(what) + ": voice " + std::to_string(voice) + " is not a " + (kind == GOOEY_B200_VOICE_POLY ? "poly synth" : "granulator"));
    return GOOEY_E_INVALID;
  }
  return GOOEY_E_OK;
}
static void gran_queue(GooeyVoiceBatch* b, uint32_t voice, uint32_t frame, const gh::GranSource& src) {
  gran_buffer_events(b->pending[voice], frame, src.buf->p, src.sr, src.len);
  b->gran_queued[voice].emplace_back(frame, src);
  b->gran_latest[voice] = src;
}

int gooey_voice_batch_note_on(GooeyVoiceBatch* b, uint32_t voice, uint32_t frame, uint32_t note, float velocity) {
  GOOEY_TRY
  if (int rc = voice_of_kind(b, voice, GOOEY_B200_VOICE_POLY, "note_on")) return rc;
  if (note > 127) { set_error("note_on: note " + std::to_string(note) + " is above 127"); return GOOEY_E_INVALID; }
  b->pending[voice].push_back(make_event(frame, gd::EV_POLY_NOTE, note, velocity));   // velocity as trigger_note takes it: unclamped
  return GOOEY_E_OK;
  GOOEY_CATCH
}

int gooey_voice_batch_release(GooeyVoiceBatch* b, uint32_t voice, uint32_t frame) {
  GOOEY_TRY
  if (int rc = voice_of_kind(b, voice, GOOEY_B200_VOICE_POLY, "release")) return rc;
  b->pending[voice].push_back(make_event(frame, gd::EV_POLY_RELEASE, 0, 0.0f));
  return GOOEY_E_OK;
  GOOEY_CATCH
}

int gooey_voice_batch_set_buffer(GooeyVoiceBatch* b, uint32_t voice, uint32_t frame, const float* samples, uint32_t len, float sample_rate) {
  GOOEY_TRY
  if (int rc = voice_of_kind(b, voice, GOOEY_B200_VOICE_GRANULATOR, "set_buffer")) return rc;
  if (!samples || len == 0) { set_error("set_buffer: empty buffer"); return GOOEY_E_INVALID; }
  if (!std::isfinite(sample_rate) || !(sample_rate > 0.0f)) { set_error("set_buffer: sample_rate must be finite and > 0"); return GOOEY_E_INVALID; }   // SampleBuffer::from_mono
  for (uint32_t i = 0; i < len; i++)
    if (!std::isfinite(samples[i])) { set_error("set_buffer: sample " + std::to_string(i) + " is not finite"); return GOOEY_E_INVALID; }
  use_device(b->device);
  gh::GranSource src;
  src.buf = std::make_shared<DevBuf<float>>();
  src.buf->alloc(len);
  GH_CUDA(cudaMemcpy(src.buf->p, samples, (size_t)len * 4, cudaMemcpyHostToDevice));
  src.len = len; src.sr = sample_rate;
  gran_queue(b, voice, frame, src);
  return GOOEY_E_OK;
  GOOEY_CATCH
}

int gooey_voice_batch_share_buffer(GooeyVoiceBatch* b, uint32_t dst_voice, uint32_t frame, uint32_t src_voice) {
  GOOEY_TRY
  if (int rc = voice_of_kind(b, dst_voice, GOOEY_B200_VOICE_GRANULATOR, "share_buffer")) return rc;
  if (int rc = voice_of_kind(b, src_voice, GOOEY_B200_VOICE_GRANULATOR, "share_buffer")) return rc;
  if (!b->gran_latest[src_voice].buf) { set_error("share_buffer: voice " + std::to_string(src_voice) + " holds no buffer"); return GOOEY_E_INVALID; }
  const gh::GranSource src = b->gran_latest[src_voice];
  gran_queue(b, dst_voice, frame, src);
  return GOOEY_E_OK;
  GOOEY_CATCH
}

int gooey_voice_batch_set_seed(GooeyVoiceBatch* b, uint32_t voice, uint32_t frame, uint32_t seed) {
  GOOEY_TRY
  if (int rc = voice_of_kind(b, voice, GOOEY_B200_VOICE_GRANULATOR, "set_seed")) return rc;
  b->pending[voice].push_back(make_event(frame, gd::EV_GRAN_SEED, 0, 0.0f, seed));
  return GOOEY_E_OK;
  GOOEY_CATCH
}

int gooey_voice_batch_render_device(GooeyVoiceBatch* b, uint32_t frames, float* out_dev, size_t stride) {
  GOOEY_TRY
  if (!b || !out_dev || stride < frames) { set_error("bad arguments"); return GOOEY_E_INVALID; }
  voice_batch_render_impl(b, frames, out_dev, stride);
  GH_CUDA(cudaStreamSynchronize(b->stream));
  GH_CUDA(cudaEventElapsedTime(&gh::g_last_kernel_ms, b->ev0, b->ev1));
  b->bank.collect_stats();
  return GOOEY_E_OK;
  GOOEY_CATCH
}

int gooey_voice_batch_render(GooeyVoiceBatch* b, uint32_t frames, float* out_host) {
  GOOEY_TRY
  if (!b || !out_host) { set_error("bad arguments"); return GOOEY_E_INVALID; }
  use_device(b->device);
  const size_t stride = (frames + 3) & ~(size_t)3;
  b->d_out.alloc((size_t)b->n * stride);
  voice_batch_render_impl(b, frames, b->d_out.p, stride);
  // drain chunk by chunk while later chunks are still being rendered (overlaps with compute when out_host is pinned)
  const uint32_t chunk = (uint32_t)b->bank.chunk_frames((int)frames);
  int ci = 0;
  for (uint32_t c0 = 0; c0 < frames; c0 += chunk, ci++) {
    const uint32_t nf = std::min(chunk, frames - c0);
    b->bank.wait_chunk(b->copy_stream, ci);
    GH_CUDA(cudaMemcpy2DAsync(out_host + c0, (size_t)frames * 4, b->d_out.p + c0, stride * 4, (size_t)nf * 4, b->n, cudaMemcpyDeviceToHost, b->copy_stream));
  }
  GH_CUDA(cudaStreamSynchronize(b->copy_stream));
  GH_CUDA(cudaStreamSynchronize(b->stream));
  GH_CUDA(cudaEventElapsedTime(&gh::g_last_kernel_ms, b->ev0, b->ev1));
  b->bank.collect_stats();
  return GOOEY_E_OK;
  GOOEY_CATCH
}

}  // extern "C"

#include "engine_api.cuh"
#include "rs_api.cuh"
#include "loops_api.cuh"
#include <sys/syscall.h>
#include <unistd.h>

extern "C" {

// 16-bit PCM of every voice (what bounce_to_wav stores, bounce.rs:105-113): rendered as f32 on the device, quantised there
// chunk by chunk and drained as int16 — half the bytes of gooey_voice_batch_render over PCIe and into host memory.
int gooey_voice_batch_render_pcm16(GooeyVoiceBatch* b, uint32_t frames, int16_t* out_host) {
  GOOEY_TRY
  if (!b || !out_host) { set_error("bad arguments"); return GOOEY_E_INVALID; }
  use_device(b->device);
  const size_t stride = (frames + 3) & ~(size_t)3;
  b->d_out.alloc((size_t)b->n * stride);
  b->d_pcm.alloc((size_t)b->n * stride);
  voice_batch_render_impl(b, frames, b->d_out.p, stride);
  const uint32_t chunk = (uint32_t)b->bank.chunk_frames((int)frames);
  int ci = 0;
  for (uint32_t c0 = 0; c0 < frames; c0 += chunk, ci++) {
    const uint32_t nf = std::min(chunk, frames - c0);
    b->bank.wait_chunk(b->copy_stream, ci);
    gd::quantize_pcm16_kernel<<<dim3((nf + 1023) / 1024, b->n), 256, 0, b->copy_stream>>>(b->d_out.p, (long long)stride, b->d_pcm.p, (long long)stride, (int)c0, (int)nf);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    GH_CUDA(cudaGetLastError());
    GH_CUDA(cudaMemcpy2DAsync(out_host + c0, (size_t)frames * 2, b->d_pcm.p + c0, stride * 2, (size_t)nf * 2, b->n, cudaMemcpyDeviceToHost, b->copy_stream));
  }
  GH_CUDA(cudaStreamSynchronize(b->copy_stream));
  GH_CUDA(cudaStreamSynchronize(b->stream));
  GH_CUDA(cudaEventElapsedTime(&gh::g_last_kernel_ms, b->ev0, b->ev1));
  b->bank.collect_stats();
  return GOOEY_E_OK;
  GOOEY_CATCH
}

// Pinned host memory for drains, placed on the NUMA node the device hangs off (read from sysfs through the device's PCI bus
// id; no libnuma: the memory policy is set with the raw syscall for the duration of the allocation and restored afterwards).
// With eight ranks draining at once, buffers that all sit on one node bound the whole box (profiles/README.md, round 1).
void* gooey_b200_host_alloc(size_t bytes, int device, int* out_numa_node) {
  if (out_numa_node) *out_numa_node = -1;
  if (bytes == 0) return nullptr;
  try { use_device(device); } catch (const std::exception& ex) { set_error(ex.what()); return nullptr; }
  int node = -1;
  char bus[32] = {0};
  if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) == cudaSuccess) {
    for (char* c = bus; *c; c++) *c = (char)tolower(*c);
    const std::string path = std::string("/sys/bus/pci/devices/") + bus + "/numa_node";
    if (FILE* f = fopen(path.c_str(), "r")) { if (fscanf(f, "%d", &node) != 1) node = -1; fclose(f); }
  } else cudaGetLastError();
  bool bound = false;
#ifdef SYS_set_mempolicy
  if (node >= 0 && node < 1024) {
    unsigned long mask[16] = {0};
    mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
    bound = syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, (unsigned long)(sizeof mask * 8)) == 0;
  }
#endif
  void* p = nullptr;
  const cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocPortable);
  if (e == cudaSuccess) memset(p, 0, bytes);           // first touch under the policy
  if (e == cudaSuccess) {
    // First DMA into freshly pinned pages is several times slower than later passes (measured with eight ranks draining into new
    // 5.8 GB blocks: 20 GB/s aggregate against 94 GB/s into blocks that had been written before — IOMMU / page-table warm-up on
    // the host side), so the allocator makes that first pass itself: zeros from a small device block over the whole range.
    void* d = nullptr;
    const size_t chunk = (size_t)64 << 20;
    if (cudaMalloc(&d, std::min(chunk, bytes)) == cudaSuccess) {
      cudaMemset(d, 0, std::min(chunk, bytes));
      for (size_t off = 0; off < bytes; off += chunk)
        cudaMemcpyAsync((char*)p + off, d, std::min(chunk, bytes - off), cudaMemcpyDeviceToHost, 0);
      cudaDeviceSynchronize();
      cudaFree(d);
    }
    cudaGetLastError();
  }
#ifdef SYS_set_mempolicy
  if (bound) syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0ul);
#endif
  if (e != cudaSuccess) { cudaGetLastError(); set_error("cudaHostAlloc failed"); return nullptr; }
  if (out_numa_node) *out_numa_node = bound ? node : -1;
  return p;
}
void gooey_b200_host_free(void* p) { if (p) cudaFreeHost(p); }

}  // extern "C"

// =================================================================================================
// Self-test hooks (tests/test_gmath_gpu.py): evaluate the gm:: routines on the device so the test can
// compare them bit-for-bit with the host libm the reference links.
// =================================================================================================
namespace gh {
__global__ void math_selftest_kernel(int kind, const float* x, const float* y, float* out, uint32_t n) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float r;
  switch (kind) {
    case 0: r = gm::g_powf(x[i], y[i]); break;
    case 1: r = gm::g_sinf(x[i]); break;
    case 2: r = gm::g_cosf(x[i]); break;
    case 3: r = gm::g_expf(x[i]); break;
    case 4: r = gd::hash_noise((uint64_t)x[i]); break;
    case 5: r = gd::max_curve(x[i], y[i]); break;
    case 6: r = gm::g_tanhf(x[i]); break;
    case 7: r = gm::g_tanf(x[i]); break;
    case 8: r = gm::g_expm1f(x[i]); break;
    case 9: r = gm::g_sinf_fast(x[i]); break;                                  // the front end's ~1-ulp sine
    case 10: r = gm::g_div_by(x[i], y[i], 1.0f / y[i]); break;                  // x / y through the hoisted reciprocal: must equal the IEEE quotient
    default: r = 0.0f;
  }
  out[i] = r;
}
}  // namespace gh

extern "C" int gooey_b200_selftest_math(int kind, const float* x_host, const float* y_host, float* out_host, uint32_t n, int device) {
  GOOEY_TRY
  use_device(device);
  DevBuf<float> dx, dy, dout;
  dx.upload(x_host, n, 0);
  dy.upload(y_host ? y_host : x_host, n, 0);
  dout.alloc(n);
  gh::math_selftest_kernel<<<(n + 255) / 256, 256>>>(kind, dx.p, dy.p, dout.p, n);
  g_launches.fetch_add(1);
  GH_CUDA(cudaGetLastError());
  GH_CUDA(cudaMemcpy(out_host, dout.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
  return GOOEY_E_OK;
  GOOEY_CATCH
}
