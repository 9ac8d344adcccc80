// poly_wave.cuh — host interface of the poly synth's warp-per-voice back end (poly_wave.cu).
//
// poly_wave_kernel renders one PolySynth per warp, lane = frame inside blocks of up to 32 frames, on the same state layout
// as slow_kernel<PolyV> and bit-identical to it, so the two may alternate from one render call to the next.  It is compiled
// in a translation unit of its own behind the launcher below (as rs_chain.cu is), so that its call sites cannot change how
// the compiler inlines into the other kernels.  That unit has its own copies of the __constant__ tables: c_midi_freq
// must be uploaded into it per device (the gm:: tables it reaches are static initialisers and need no upload).
#pragma once
#include "kernels.cuh"

namespace gd {

// grid = ceil(n / POLY_WAVE_WARPS) CTAs of POLY_WAVE_WARPS warps, one voice per warp
constexpr int POLY_WAVE_WARPS = 2;
void poly_wave_launch(const VoiceLaunch& L, cudaStream_t st);
void poly_wave_set_midi_freq(const double mf[128]);

}  // namespace gd
