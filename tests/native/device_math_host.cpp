// Host build of the product's device math primitives (csrc/fit_math.cuh, csrc/gppd_device.cuh)
// so that the CPU test-suite can hold them to high-precision references without a GPU.
// g++ -O2 -ffp-contract=off -I/usr/local/cuda/include: every explicit fma / _rn operation is
// the same IEEE operation as on the device; sincos() / hypot() / atan2() are the C library's.
// sqrt4 (inline PTX) exists on the device only (device_math.cu).
#include "cuda_host_shim.h"
#include "fit_math.cuh"

struct Stage {
    template <class T> const T *in(const T *p, long long) { return p; }
    template <class T> T *out(T *p, long long) { return p; }
    template <class F> int run(const F &f, long long n) {
        for (long long i = 0; i < n; ++i) f(i);
        return 0;
    }
};

#include "device_math_entries.h"
