/* TEST INFRASTRUCTURE ONLY.  tests/cpp/jit_host_shim.h plus the intrinsics that the generated source of function-grammar
 * programs uses (op_sqrt, op_abs; mcb_trig.h itself needs none under g++). */
#include "jit_host_shim.h"
static inline float __uint_as_float(unsigned u) { float f; std::memcpy(&f, &u, 4); return f; }
static inline float __fsqrt_rn(float a) { return std::sqrt(a); }
