// tests/rs_chain_host.cpp — TEST INFRASTRUCTURE ONLY (never loaded by the product).  The global effect chain of a Rust-API
// `Engine` (engine/mod.rs:400-412: `for effect in global_effects: x = effect.process(x)`) restated on the oracle's own effect
// classes (oracle/effects.hpp, oracle/prims.hpp), built with the oracle's compiler flags, for tests/rs_effects_oracle.py.
// The chain only follows the engine's mono sum, so folding a dry bounce through it sample by sample is what the engine's
// tick computes.
#include <memory>
#include <vector>
#include "../oracle/effects.hpp"

using namespace orc;

namespace {
// one effect by FFI effect id, from its constructor arguments after the sample rate, in the reference's order
struct MonoFx {
  std::unique_ptr<StereoEffect> fx; std::unique_ptr<Waveshaper> ws; std::unique_ptr<FeedbackWaveshaper> fb; std::unique_ptr<SoftLimiter> lim;
  float process(float in) { return fx ? fx->process(in) : ws ? ws->process(in) : fb ? fb->process(in) : lim->process(in); }
};
bool build(MonoFx& m, uint32_t kind, float sr, const float* c) {
  switch (kind) {
    case 0: m.fx.reset(new LowpassFilterEffect(sr, c[0], c[1])); return true;
    case 1: m.fx.reset(new DelayEffect(sr, (uint32_t)c[0], c[1], c[2], c[3], c[4])); return true;
    case 2: m.fx.reset(new TubeSaturation(sr, c[0], c[1], c[2])); return true;
    case 3: m.fx.reset(new TubeCompressor(sr, c[0], c[1], c[2], c[3], c[4])); return true;
    case 4: m.fx.reset(new TiltFilterEffect(sr)); return true;
    case 5: m.lim.reset(new SoftLimiter(c[0])); return true;
    case 6: m.fx.reset(new SpringReverbEffect(sr, c[0], c[1], c[2])); return true;
    case 7: m.ws.reset(new Waveshaper(c[0], c[1])); return true;
    case 8: m.fb.reset(new FeedbackWaveshaper(sr, c[0], c[1], c[2], c[3])); return true;
    case 9: m.fx.reset(new PlateReverbEffect(sr, c[0], c[1], c[2])); return true;
    default: return false;
  }
}
struct Chain { float sr; std::vector<std::unique_ptr<MonoFx>> fx; };
}  // namespace

extern "C" {
void* rs_chain_new(float sr) { return new Chain{sr, {}}; }
void rs_chain_free(void* h) { delete (Chain*)h; }
void rs_chain_clear(void* h) { ((Chain*)h)->fx.clear(); }
int rs_chain_add(void* h, uint32_t kind, const float* args) {
  Chain* ch = (Chain*)h;
  auto m = std::make_unique<MonoFx>();
  if (!build(*m, kind, ch->sr, args)) return -1;
  ch->fx.push_back(std::move(m));
  return 0;
}
void rs_chain_process(void* h, const float* in, float* out, uint32_t n) {
  Chain* ch = (Chain*)h;
  for (uint32_t i = 0; i < n; i++) {
    float x = in[i];
    for (auto& m : ch->fx) x = m->process(x);
    out[i] = x;
  }
}
}  // extern "C"
