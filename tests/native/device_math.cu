// Device build of the product's device math primitives (csrc/fit_math.cuh,
// csrc/gppd_device.cuh), one kernel launch per entry point, built twice by
// tests/test_device_math.py with the library's flags: -fmad=true (as stream_kernels.cu,
// harm_*.cu) and -fmad=false (as fit_kernels.cu).  Each call copies its host arrays in
// with cudaMemcpy, runs the element function once per element, copies the results out and
// frees everything before it returns.
#include <vector>

#include "fit_math.cuh"

template <class F> __global__ void k_each(F f, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) f(i);
}

struct Stage {
    struct Out {
        void *host, *dev;
        size_t bytes;
    };
    std::vector<void *> bufs;
    std::vector<Out> outs;
    cudaError_t err = cudaSuccess;

    void *alloc(size_t bytes) {
        void *d = nullptr;
        if (err == cudaSuccess) err = cudaMalloc(&d, bytes ? bytes : 1);
        if (d) bufs.push_back(d);
        return d;
    }
    template <class T> const T *in(const T *p, long long n) {
        T *d = static_cast<T *>(alloc(n * sizeof(T)));
        if (err == cudaSuccess && n) err = cudaMemcpy(d, p, n * sizeof(T), cudaMemcpyHostToDevice);
        return d;
    }
    template <class T> T *out(T *p, long long n) {
        T *d = static_cast<T *>(alloc(n * sizeof(T)));
        outs.push_back({p, d, n * sizeof(T)});
        return d;
    }
    template <class F> int run(const F &f, long long n) {
        if (err == cudaSuccess && n > 0) {
            k_each<<<(unsigned)((n + 255) / 256), 256>>>(f, n);
            err = cudaGetLastError();
        }
        if (err == cudaSuccess) err = cudaDeviceSynchronize();
        for (const Out &o : outs)
            if (err == cudaSuccess && o.bytes) err = cudaMemcpy(o.host, o.dev, o.bytes, cudaMemcpyDeviceToHost);
        return (int)err;
    }
    ~Stage() {
        for (void *d : bufs) cudaFree(d);
    }
};

#include "device_math_entries.h"

namespace dm {
// r[4 j + k] from the quad h[4 j .. 4 j + 3] (one range check for the four values)
struct Sqrt4Op {
    const double *h;
    double *r;
    __device__ void operator()(long long j) const {
        const double hq[4] = {h[4 * j], h[4 * j + 1], h[4 * j + 2], h[4 * j + 3]};
        double rq[4];
        gppd::sqrt4(hq, rq);
        for (int k = 0; k < 4; ++k) r[4 * j + k] = rq[k];
    }
};
struct SqrtOp {
    const double *h;
    double *r;
    __device__ void operator()(long long i) const { r[i] = sqrt(h[i]); }
};
}  // namespace dm

extern "C" {
// n: a multiple of 4
int dm_sqrt4(const double *h, double *r, long long n) {
    Stage st;
    return st.run(dm::Sqrt4Op{st.in(h, n), st.out(r, n)}, n / 4);
}
int dm_sqrt(const double *h, double *r, long long n) {
    Stage st;
    return st.run(dm::SqrtOp{st.in(h, n), st.out(r, n)}, n);
}
}
