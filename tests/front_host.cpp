// tests/front_host.cpp — TEST INFRASTRUCTURE ONLY (never loaded by the product).  Host build of the MaxCurve envelope the
// hi-hat and tom front ends evaluate (libgooey_b200/csrc/dsp.cuh compiled by g++), for tests/test_front_cpu.py.
#include <cstdint>
#include "../libgooey_b200/csrc/dsp.cuh"

using namespace gd;

extern "C" {
// Two-segment MaxCurve envelope (seg6 = (target, ms, curve) x 2) triggered at 0 and sampled at times[]: hoisted = 0 ticks it
// through maxenv_value (the per-sample path), 1 evaluates every time from the trigger snapshot with the segment constants
// the planner derives once per span (the front end's path).
int front_maxenv(const float* seg6, const double* times, float* out, uint32_t n, int hoisted) {
  MaxEnv2 e;
  maxenv_init(e, seg6[0], seg6[1], seg6[2], seg6[3], seg6[4], seg6[5]);
  maxenv_trigger(e, 0.0);
  const MaxEnv2 snap = e;
  const MaxEnvK k = maxenv_k(snap);
  for (uint32_t i = 0; i < n; i++) out[i] = hoisted ? maxenv_value_pure(snap, k, times[i]) : maxenv_value(e, times[i]);
  return 0;
}
}  // extern "C"
