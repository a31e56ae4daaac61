// Host build of csrc/philox.cuh: the Random123 known-answer vectors of Philox4x32-10 and the end points of the
// uniform mapping.  Prints "kat<i> w0 w1 w2 w3" (hex) and "u0 <value>" / "u1 <value>" (%a, exact).
#include <stdio.h>

#include "philox.cuh"

using namespace babe;

int main() {
  const uint32_t kat[3][6] = {{0u, 0u, 0u, 0u, 0u, 0u},
                              {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu},
                              {0x243f6a88u, 0x85a308d3u, 0x13198a2eu, 0x03707344u, 0xa4093822u, 0x299f31d0u}};
  for (int i = 0; i < 3; ++i) {
    const Philox4 o = philox4x32_10(kat[i][0], kat[i][1], kat[i][2], kat[i][3], kat[i][4], kat[i][5]);
    printf("kat%d %08x %08x %08x %08x\n", i, o.x[0], o.x[1], o.x[2], o.x[3]);
  }
  printf("u0 %a\n", (double)philox_uniform(0u));
  printf("u1 %a\n", (double)philox_uniform(0xffffffffu));
  return 0;
}
