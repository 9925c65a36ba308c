// steph.cpp -- CPU build of the per-step time constants of poseestimationkf_b200/csrc/ekf_math.cuh (StepH).
//
// TEST TOOL ONLY: the packed kernel of a batch of recordings forms StepH<f32x2> from two lanes with different dt; each
// lane must round as the scalar kernels' StepH<float> of its own dt.  Compiled by tests/test_batch_recordings_cpu.py
// with the flags of tests/hostsim/innovation.py (-ffp-contract=off: only the explicit fma_ calls fuse).
#include <cstdint>
#include "../../poseestimationkf_b200/csrc/ekf_math.cuh"

using namespace pkf;

// out[0..3n): h, h^2, -h/6 of StepH<float>(h0[i]) and StepH<float>(h1[i]) interleaved as lanes x, y;
// out[6n..12n): the same from StepH<f32x2>(f32x2(h0[i], h1[i])).
extern "C" int hostsim_steph(int64_t n, const float* h0, const float* h1, float* out) {
  for (int64_t i = 0; i < n; ++i) {
    const StepH<float> a(h0[i]), b(h1[i]);
    const StepH<f32x2> p(f32x2(h0[i], h1[i]));
    float* s = out + 6 * i;
    float* v = out + 6 * n + 6 * i;
    s[0] = a.h; s[1] = b.h; s[2] = a.hh; s[3] = b.hh; s[4] = a.mh6; s[5] = b.mh6;
    v[0] = p.h.x; v[1] = p.h.y; v[2] = p.hh.x; v[3] = p.hh.y; v[4] = p.mh6.x; v[5] = p.mh6.y;
  }
  return 0;
}
