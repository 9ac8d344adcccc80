// rs_chain.cu — the kernels of rs_chain.cuh and their launchers.
#define GOOEY_OWN_KERNELS_TU
#include "device_rt.h"
#include "rs_chain.cuh"

namespace gd {

__device__ __forceinline__ float rs_fx_mono(FxDyn& f, uint32_t kind, const RingRef& r, const FxGeom& g, float x, const RateCtx& rc) {
  switch (kind) {
    case FXK_LOWPASS: return lowpass_one(f.lp, 0, x, rc);
    case FXK_DELAY: {   // delay.rs `process` = the left channel of process_stereo without ping-pong
      const float in = isfinite(x) ? x : 0.0f;
      const DelayPrep p = delay_prep(f.delay, 0, r, g.delay_len, rc);
      const float s1 = r.at(p.r1), s2 = r.at(p.r2);
      const DelayStep s = delay_filter(f.delay, 0, p, s1, s2, rc);
      return delay_write(f.delay, 0, r, g.delay_len, in, in, s, s.filtered);
    }
    case FXK_SATURATION: return sat_one(f.sat, 0, r, x, rc);
    case FXK_COMPRESSOR: return comp_one(f.comp, 0, r, x, x, rc);
    case FXK_TILT: return tilt_one(f.tilt, 0, x, rc);
    case FXK_LIMITER: return gm::g_tanhf(x * __uint_as_float(f.w[1])) * __uint_as_float(f.w[0]);
    case FXK_SPRING: {
      float dl[6];
#pragma unroll
      for (int i = 0; i < 6; i++) dl[i] = r.at(g.spring_off[i] + f.spring.ch[0].idx[i]);
      return spring_one(f.spring, 0, r, g, x, rc, dl);
    }
    case FXK_WAVESHAPER: return wsfx_one(f.ws, 0, r, x);
    case FXK_FBWS: return fbwsfx_one(f.fbws, 0, r, x);
    case FXK_PLATE: {   // plate_reverb.rs `process`: the tank's two outputs averaged, one mix
      const float in = isfinite(x) ? x : 0.0f;
      float wl, wr, mix;
      plate_tank(f.plate, r, g, in, wl, wr, mix, rc);
      const float o = in * (1.0f - mix) + 0.5f * (wl + wr) * mix;
      return isfinite(o) ? o : in;
    }
    default: return x;
  }
}

// grid = n_warps, 32 threads; dynamic shared memory RS_CHAIN_SMEM (the FxDyn states are indexed by a run-time chain
// position, which would put them in local memory).
constexpr size_t RS_CHAIN_SMEM = 32 * RS_MAX_FX * sizeof(FxDyn);
__global__ void __launch_bounds__(32) rs_chain_kernel(const RsChainLaunch L) {
  __shared__ float tile[TILE * 33];
  extern __shared__ __align__(16) unsigned char rs_chain_smem[];
  FxDyn* dyn = reinterpret_cast<FxDyn*>(rs_chain_smem) + threadIdx.x * RS_MAX_FX;
  const int lane = threadIdx.x;
  const uint32_t* rows = L.rows + blockIdx.x * 32;
  const uint32_t e = rows[lane];
  const bool valid = e != ~0u;
  const uint32_t row_mask = __ballot_sync(0xffffffffu, valid);
  const uint32_t nfx = L.warp_nfx[blockIdx.x];
  const uint8_t* kinds = L.warp_kinds + blockIdx.x * RS_MAX_FX;
  if (valid)
    for (uint32_t k = 0; k < nfx; k++) dyn[k] = L.state[(size_t)e * RS_MAX_FX + k];
  for (int f0 = 0; f0 < L.frames; f0 += TILE) {
    const int nf = min(TILE, L.frames - f0);
    for (int r = 0; r < 32; r++)
      if (((row_mask >> r) & 1u) && lane < nf) tile[r * 33 + lane] = L.out[(long long)rows[r] * L.out_stride + f0 + lane];
    __syncwarp();
    if (valid) {
      for (int j = 0; j < nf; j++) {
        float x = tile[lane * 33 + j];
#pragma unroll 1
        for (uint32_t k = 0; k < nfx; k++) x = rs_fx_mono(dyn[k], kinds[k], RingRef{L.ring[k], L.ring_pitch, (int)e}, L.geo, x, L.rc);
        tile[lane * 33 + j] = x;
      }
    }
    __syncwarp();
    store_tile_voice_major(tile, L.out, L.out_stride, 0, rows, row_mask, f0, nf, lane);
    __syncwarp();
  }
  if (valid)
    for (uint32_t k = 0; k < nfx; k++) L.state[(size_t)e * RS_MAX_FX + k] = dyn[k];
}

// Writes freshly constructed effects into the state pool: one thread per (engine, position) entry.
__global__ void rs_fx_init_kernel(FxDyn* __restrict__ state, const FxDyn* __restrict__ fresh, const uint32_t* __restrict__ where, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) state[where[i]] = fresh[i];
}

void rs_chain_launch(const RsChainLaunch& L, uint32_t n_warps, cudaStream_t st) { rs_chain_kernel<<<n_warps, 32, RS_CHAIN_SMEM, st>>>(L); }
void rs_fx_init_launch(FxDyn* state, const FxDyn* fresh, const uint32_t* where, int n, cudaStream_t st) { rs_fx_init_kernel<<<(n + 127) / 128, 128, 0, st>>>(state, fresh, where, n); }
void rs_chain_set_halfband(const float hb[8]) {
  GH_CUDA(cudaMemcpyToSymbol(c_hb, hb, 8 * sizeof(float)));
}

}  // namespace gd
