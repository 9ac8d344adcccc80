// rs_chain.cuh — the global effect chain of Rust-API engines (reference: src/engine/mod.rs:400-412, src/effects/*.rs).
//
// `Engine::tick` runs `for effect in global_effects: x = effect.process(x)` on the mono mix.  `process` is the channel-0
// path of each effect, except that the compressor is its own side-chain, the plate has its own mono mix
// (plate_reverb.rs `process`) and the stand-alone waveshapers are single instances.  The per-channel device functions of
// mix.cuh are reused on channel 0; only the mono plate mix and the limiter are written here.
//
// rs_mix_kernel writes Σ instruments x master for the engines of this kernel (their limiter count is 0 there), and
// rs_chain_kernel runs the chain in place on those output rows.  One thread per engine; the host orders engines so that
// each warp shares one chain signature (the kinds in order), so the per-kind dispatch is warp-uniform.  Effect state
// (one FxDyn per chain position) persists in a device pool across bounces; delay / spring / plate lines and the
// oversampler histories live in one ring arena per chain position, laid out [word][engine] (mix.cuh, DESIGN §3).
#pragma once
#include "mix.cuh"

namespace gd {

constexpr int RS_MAX_FX = 8;
// constructor arguments after the sample rate, by FFI effect id (orc_fx_new order)
constexpr uint32_t RS_FX_ARGS[10] = {2, 5, 3, 5, 0, 1, 3, 2, 4, 3};

// Builds effect `kind` from its constructor arguments at sample rate `sr`, with fresh state.  The limiter keeps its
// threshold and reciprocal in the first two words (the arithmetic of rs_mix_kernel and limiter.rs).
inline void rs_fx_construct(FxDyn& f, uint32_t kind, const float* a, float sr) {
  for (int i = 0; i < 40; i++) f.w[i] = 0;
  switch (kind) {
    case FXK_LOWPASS: lp_init(f.lp, a[0], a[1]); break;
    case FXK_DELAY: delay_init(f.delay, (uint32_t)f32_to_u64_sat(a[0]), a[1], a[2], a[3], a[4]); break;
    case FXK_SATURATION: sat_init(f.sat, a[0], a[1], a[2]); break;
    case FXK_COMPRESSOR: comp_init(f.comp, a[0], a[1], a[2], a[3], a[4]); break;
    case FXK_TILT: tilt_init(f.tilt, sr); break;
    case FXK_LIMITER: { const float th = fmaxf(a[0], 0.001f), inv = 1.0f / th; memcpy(&f.w[0], &th, 4); memcpy(&f.w[1], &inv, 4); } break;
    case FXK_SPRING: spring_init(f.spring, a[0], a[1], a[2]); break;
    case FXK_WAVESHAPER: for (int c = 0; c < 2; c++) { f.ws.drive[c] = clampf(a[0], 1.0f, 10.0f); f.ws.mix[c] = clampf(a[1], 0.0f, 1.0f); } f.ws.shared = 1; break;
    case FXK_FBWS: for (int c = 0; c < 2; c++) fbsmall_init(f.fbws.s[c], sr, a[0], a[1], a[2], a[3]); f.fbws.shared = 1; break;
    case FXK_PLATE: plate_init(f.plate, a[0], a[1], a[2]); break;
    default: break;
  }
}
// ring words one engine needs for the channel-0 path of `kind`
inline uint32_t rs_fx_ring_words(const FxGeom& g, uint32_t kind) {
  switch (kind) {
    case FXK_DELAY: return g.delay_len;
    case FXK_SPRING: return g.spring_off[6];
    case FXK_PLATE: return g.ring_words[3];
    case FXK_SATURATION: case FXK_COMPRESSOR: case FXK_WAVESHAPER: case FXK_FBWS: return OS_WORDS;
    default: return 0;
  }
}

struct RsChainLaunch {
  float* out; long long out_stride; int frames;
  const uint32_t* rows;           // [n_warps * 32] engine of each thread (= its output row, pool column and ring column); ~0u = padding
  const uint8_t* warp_kinds;      // [n_warps][RS_MAX_FX] the chain signature of each warp
  const uint32_t* warp_nfx;       // [n_warps]
  FxDyn* state;                   // [engine][RS_MAX_FX]
  float* ring[RS_MAX_FX]; long long ring_pitch;
  RateCtx rc; FxGeom geo;
};

// rs_chain.cu, a translation unit of its own, so that its call sites cannot change how the compiler inlines into the
// other kernels.  Each module has its own copy of the half-band coefficients.
void rs_chain_launch(const RsChainLaunch& L, uint32_t n_warps, cudaStream_t st);
void rs_fx_init_launch(FxDyn* state, const FxDyn* fresh, const uint32_t* where, int n, cudaStream_t st);
void rs_chain_set_halfband(const float hb[8]);

}  // namespace gd
