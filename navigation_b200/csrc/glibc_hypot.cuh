// glibc_hypot.cuh -- hypot(x, y) as glibc 2.35 and later computes it (sysdeps/ieee754/dbl-64/e_hypot.c, the
// `hypot@@GLIBC_2.35` symbol of x86-64, an ordinary function rather than an ifunc, built without FMA), for the host
// and the device alike.  glibc's hypot is not correctly rounded, so CUDA's hypot (or any correctly rounded one) does
// not give the host's bits; this restatement does, with plain IEEE operations: a scaled square root, then one
// correction step.  The device side spells every operation as a round-to-nearest intrinsic, so neither FMA
// contraction nor -prec-div / -prec-sqrt can change it.
//
// Self-contained: it also compiles as plain C++ (g++ -O2 -ffp-contract=off), where glibc_hypot_matches_libm()
// compares it with the running libm's hypot on a fixed list of pairs -- among them pairs where glibc 2.35+ is not
// correctly rounded, the cutoffs of the scaled paths and the non-finite cases.  Callers that need the device to give
// the host's hypot (the TrajectoryPlanner's device fleet step) check it once per process.
#pragma once

#include <cmath>
#include <cstdint>
#include <cstring>

#ifdef __CUDACC__
#define GLIBC_HYPOT_HD __host__ __device__
#else
#define GLIBC_HYPOT_HD
#endif

namespace glibc_hypot_detail {

#ifdef __CUDA_ARCH__
__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double div(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ double sqrt_rn(double a) { return __dsqrt_rn(a); }
__device__ __forceinline__ uint64_t bits(double a) { return (uint64_t)__double_as_longlong(a); }
#else
inline double add(double a, double b) { return a + b; }
inline double sub(double a, double b) { return a - b; }
inline double mul(double a, double b) { return a * b; }
inline double div(double a, double b) { return a / b; }
inline double sqrt_rn(double a) { return std::sqrt(a); }
inline uint64_t bits(double a) {
  uint64_t u;
  std::memcpy(&u, &a, sizeof(u));
  return u;
}
#endif

// e_hypot.c's kernel: ax >= ay >= 0, scaled so that neither squaring ax, ay nor (ax - ay) overflows or underflows
GLIBC_HYPOT_HD inline double kernel(double ax, double ay) {
  double h = sqrt_rn(add(mul(ax, ax), mul(ay, ay)));
  double t1, t2;
  if (h <= mul(2.0, ay)) {
    const double d = sub(h, ay);
    t1 = mul(ax, sub(mul(2.0, d), ax));
    t2 = mul(sub(d, mul(2.0, sub(ax, ay))), d);
  } else {
    const double d = sub(h, ax);
    t1 = mul(mul(2.0, d), sub(ax, mul(2.0, ay)));
    t2 = add(mul(sub(mul(4.0, d), ay), ay), mul(d, d));
  }
  return sub(h, div(add(t1, t2), mul(2.0, h)));
}

GLIBC_HYPOT_HD inline bool is_nan(double a) { return (bits(a) & 0x7fffffffffffffffull) > 0x7ff0000000000000ull; }
GLIBC_HYPOT_HD inline bool is_inf(double a) { return (bits(a) & 0x7fffffffffffffffull) == 0x7ff0000000000000ull; }
GLIBC_HYPOT_HD inline bool is_signaling(double a) { return is_nan(a) && !(bits(a) & 0x0008000000000000ull); }

}  // namespace glibc_hypot_detail

GLIBC_HYPOT_HD inline double glibc_hypot(double x, double y) {
  namespace d = glibc_hypot_detail;
  // (the cutoffs and scale factors of the x86-64 build: ay below 0x1p-459 takes the scaled-up path)
  const double kLarge = 0x1p+511, kTiny = 0x1p-459, kEps = 0x1p-54;
  if (d::is_nan(x) || d::is_nan(y) || d::is_inf(x) || d::is_inf(y)) {
    // an infinity wins over a quiet NaN; otherwise a NaN (x + y, as glibc returns it)
    if ((d::is_inf(x) || d::is_inf(y)) && !d::is_signaling(x) && !d::is_signaling(y)) return HUGE_VAL;
    return d::add(x, y);
  }
  x = std::fabs(x);
  y = std::fabs(y);
  const double ax = x < y ? y : x, ay = x < y ? x : y;
  if (ax > kLarge) {  // scale down, so that the squares do not overflow
    if (ay <= d::mul(ax, kEps)) return d::add(ax, ay);
    return d::mul(d::kernel(d::mul(ax, 0x1p-600), d::mul(ay, 0x1p-600)), 0x1p+600);
  }
  if (ay < kTiny) {  // scale up, so that the squares do not underflow
    if (ax >= d::mul(ay, 0x1p+54)) return d::add(ax, ay);
    return d::mul(d::kernel(d::mul(ax, 0x1p+600), d::mul(ay, 0x1p+600)), 0x1p-600);
  }
  if (ay <= d::mul(ax, kEps)) return d::add(ax, ay);
  return d::kernel(ax, ay);
}

// Host only: whether the running libm's hypot gives glibc_hypot's bits on a fixed list of pairs (NaNs compare as
// NaNs): pairs where glibc 2.35+ is not correctly rounded, integers, equal arguments, zeros, subnormals, both sides of
// the scaled paths' cutoffs, and the non-finite cases.  False on a libm that computes hypot another way (an older glibc, musl),
// whose hypot the device then does not reproduce.
inline bool glibc_hypot_matches_libm() {
  static const double kPairs[][2] = {
      // glibc 2.35+ is not correctly rounded on these: its result is one ulp from the correctly rounded value
      {0x1.04450df36734ep-16, 0x1.acf53b2ffb10dp-17}, {0x1.c4db9eded536bp-23, 0x1.4d86bf3a5c646p-24},
      {0x1.1a28b00147f97p-6, 0x1.06ca521f092bfp-6}, {0x1.416c54673015dp+8, 0x1.2044136192fe4p+8},
      {0x1.134f1be2b91e9p+13, 0x1.8746f3319ed61p+12}, {0x1.663fbf8417898p-2, 0x1.863cb52dd2d88p-3},
      {0x1.dfbd69bf39fe9p+11, 0x1.0c8f47e57868cp+9}, {0x1.18bd8e5dfd705p-7, 0x1.05e5c3d615a44p-7},
      {3.0, 4.0}, {5.0, 12.0}, {1.0, 1.0}, {0.1, 0.1}, {0.3, -0.4}, {-2.5, 0.0}, {0.0, -0.0}, {0.0, 0.0},
      {1e-300, 1e-300}, {4.9406564584124654e-324, 4.9406564584124654e-324}, {2.2250738585072009e-308, 1e-310},
      {0x1p+511, 0x1p+511}, {0x1.0000000000001p+511, 0x1p+510}, {0x1p+1023, 0x1p+1023}, {1.7976931348623157e308, 1.0},
      {0x1p-459, 0x1p-459}, {0x1.fffffffffffffp-460, 0x1p-400}, {0x1.26957477f64eap-511, 0x1.26957477f64eap-511},
      {0x1p-400, 0x1p-455}, {0x1p-400, 0x1p-453},
      {1.0, 0x1p-54}, {1.0, 0x1.0000000000001p-54}, {1e4, 1e-9}, {1e4, 1.3e-12},
      {HUGE_VAL, NAN}, {NAN, -HUGE_VAL}, {NAN, 1.0}, {2.0, NAN}, {-HUGE_VAL, 3.0}, {NAN, NAN}};
  for (const auto& p : kPairs) {
    // (read through volatile, so that the compiler cannot fold std::hypot into its own, correctly rounded, constant)
    volatile double vx = p[0], vy = p[1];
    const double x = vx, y = vy;
    const double want = std::hypot(x, y), got = glibc_hypot(x, y);
    if (std::isnan(want) != std::isnan(got)) return false;
    if (!std::isnan(want) && glibc_hypot_detail::bits(want) != glibc_hypot_detail::bits(got)) return false;
  }
  return true;
}

#undef GLIBC_HYPOT_HD
