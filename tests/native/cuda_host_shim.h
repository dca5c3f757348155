// Host stand-ins for the CUDA intrinsics the product's device headers use, so that
// g++ can compile those headers unchanged.  Every one is the exact IEEE operation or
// bit move the intrinsic names (__dmul_rn / __dadd_rn are one correctly rounded
// multiply / add, __fma_rn one fused multiply-add); compile with -ffp-contract=off so
// that g++ does not fuse the other products and sums either (nvcc -fmad=false).
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>
#include <cuda_runtime.h>  // double2 / float2 and the __device__ family (empty for g++)

using std::atan2;
using std::fabs;
using std::fma;
using std::hypot;
using std::rint;
using std::sqrt;

static inline long long __double_as_longlong(double x) {
    long long u;
    std::memcpy(&u, &x, 8);
    return u;
}
static inline double __longlong_as_double(long long u) {
    double x;
    std::memcpy(&x, &u, 8);
    return x;
}
static inline int __double2hiint(double x) { return (int)((unsigned long long)__double_as_longlong(x) >> 32); }
static inline int __double2loint(double x) { return (int)(uint32_t)__double_as_longlong(x); }
static inline double __hiloint2double(int hi, int lo) {
    return __longlong_as_double((long long)(((unsigned long long)(uint32_t)hi << 32) | (uint32_t)lo));
}
static inline float __uint_as_float(uint32_t u) {
    float f;
    std::memcpy(&f, &u, 4);
    return f;
}
static inline uint32_t __float_as_uint(float f) {
    uint32_t u;
    std::memcpy(&u, &f, 4);
    return u;
}
static inline double __dmul_rn(double a, double b) { return a * b; }
static inline double __dadd_rn(double a, double b) { return a + b; }
static inline double __fma_rn(double a, double b, double c) { return std::fma(a, b, c); }
template <class T> static inline T __ldg(const T *p) { return *p; }
// byte i of the result = byte (s >> 4 i) & 7 of the eight bytes {y, x} (x the low four)
static inline uint32_t __byte_perm(uint32_t x, uint32_t y, uint32_t s) {
    const uint64_t v = ((uint64_t)y << 32) | x;
    uint32_t r = 0;
    for (int i = 0; i < 4; ++i) r |= (uint32_t)((v >> (8 * ((s >> (4 * i)) & 7))) & 0xff) << (8 * i);
    return r;
}
