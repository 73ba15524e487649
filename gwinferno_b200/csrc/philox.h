// Philox4x32-10 (Salmon et al., SC'11) and the 53-bit uniform built from two of its words: the counter-based generator of
// the device-side synthetic injections (synth.cu) and of the posterior-predictive draws (sample_draw.cuh).  Host + device;
// gwinferno_b200/synthetic.py: philox4x32_10 is the bit-exact NumPy twin.
#pragma once
#include <cstdint>

#include "gwi_internal.h"

namespace gwi {

struct U4 {
  uint32_t x, y, z, w;
};

GWI_HD inline U4 philox4x32_10(U4 c, uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)M0 * c.x, p1 = (uint64_t)M1 * c.z;
    U4 n;
    n.x = (uint32_t)(p1 >> 32) ^ c.y ^ k0;
    n.y = (uint32_t)p1;
    n.z = (uint32_t)(p0 >> 32) ^ c.w ^ k1;
    n.w = (uint32_t)p0;
    c = n;
    k0 += W0;
    k1 += W1;
  }
  return c;
}

// 53-bit uniform in [0, 1) from two 32-bit words (what numpy's next_double does with a 64-bit word)
GWI_HD inline double u01(uint32_t hi, uint32_t lo) { return (double)((((uint64_t)hi << 32) | lo) >> 11) * (1.0 / 9007199254740992.0); }

}  // namespace gwi
