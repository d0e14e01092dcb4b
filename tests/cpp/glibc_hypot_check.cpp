// glibc_hypot (navigation_b200/csrc/glibc_hypot.cuh) against the running libm's hypot, bit for bit, on a seeded set
// of pairs: random magnitudes over the whole exponent range, nearby magnitudes, integers, equal arguments, one argument
// zero, subnormals, both sides of the 0x1p+511 and 0x1p-459 cutoffs and of the 0x1p-54 ratio, and every +-inf / NaN
// combination.
// Prints "pairs <n> mismatches <m> probe <0|1>" and, for the first few mismatches, the pair.
// Build: g++ -O2 -ffp-contract=off -std=c++17 glibc_hypot_check.cpp -lm
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <limits>

#include "../../navigation_b200/csrc/glibc_hypot.cuh"

namespace {

uint64_t g_state = 0x9e3779b97f4a7c15ull;
uint64_t next_u64() {  // xorshift64*
  g_state ^= g_state >> 12;
  g_state ^= g_state << 25;
  g_state ^= g_state >> 27;
  return g_state * 0x2545f4914f6cdd1dull;
}
double uniform() { return (next_u64() >> 11) * 0x1p-53; }
double from_bits(uint64_t u) {
  double d;
  std::memcpy(&d, &u, sizeof(d));
  return d;
}
double sign() { return (next_u64() & 1) ? -1.0 : 1.0; }

long g_pairs = 0, g_mismatches = 0;
void check(double x, double y) {
  for (int k = 0; k < 2; ++k) {  // both argument orders
    const double a = k ? y : x, b = k ? x : y;
    const double want = std::hypot(a, b), got = glibc_hypot(a, b);
    ++g_pairs;
    const bool same =
        std::isnan(want) ? std::isnan(got) : glibc_hypot_detail::bits(want) == glibc_hypot_detail::bits(got);
    if (!same && g_mismatches++ < 10) std::printf("mismatch %a %a: libm %a, glibc_hypot %a\n", a, b, want, got);
  }
}

}  // namespace

int main() {
  const double inf = HUGE_VAL, qnan = std::numeric_limits<double>::quiet_NaN();
  const double snan = std::numeric_limits<double>::signaling_NaN();
  const double specials[] = {0.0, -0.0, 1.0, -3.5, 0x1p-1074, 0x1p-1022, 1.7976931348623157e308, inf, -inf, qnan,
                             -qnan, snan};
  for (double a : specials)
    for (double b : specials) check(a, b);
  // 2 x 1.5e6: any finite bit patterns (every exponent, subnormals included)
  for (int i = 0; i < 1500000; ++i) check(from_bits(next_u64() & 0x7fefffffffffffffull) * sign(),
                                          from_bits(next_u64() & 0x7fefffffffffffffull) * sign());
  // 2 x 2e6: log-uniform magnitudes over the whole exponent range, independently and within 2^-60 .. 2^60 of each other
  for (int i = 0; i < 1000000; ++i) {
    const double x = std::ldexp(1.0 + uniform(), (int)(next_u64() % 2098) - 1074);
    check(x * sign(), std::ldexp(1.0 + uniform(), (int)(next_u64() % 2098) - 1074) * sign());
    check(x * sign(), x * std::ldexp(1.0 + uniform(), (int)(next_u64() % 121) - 60));
  }
  // 2 x 2e6: the planner's range, 1e-9 .. 2e4, independent and with nearby magnitudes
  for (int i = 0; i < 1000000; ++i) {
    const double lo = std::log(1e-9), hi = std::log(2e4);
    const double x = std::exp(lo + uniform() * (hi - lo));
    check(x * sign(), std::exp(lo + uniform() * (hi - lo)) * sign());
    check(x, x * (0.05 + 0.95 * uniform()));
  }
  // 2 x 5e5: integers; equal arguments; one argument zero
  for (int i = 0; i < 500000; ++i) {
    check((double)(int64_t)(next_u64() % 100000), (double)(int64_t)(next_u64() % 100000));
    const double x = std::ldexp(1.0 + uniform(), (int)(next_u64() % 2098) - 1074);
    check(x, -x);
    check(i % 2 ? 0.0 : -0.0, x);
  }
  // 3 x 2 x 5e5 around each cutoff: ax near 0x1p+511, ay near 0x1p-459 and 0x1p-511, ay / ax near 0x1p-54, both
  // neighbours included
  for (int i = 0; i < 500000; ++i) {
    const double big = std::ldexp(1.0, 511), tiny = std::ldexp(1.0, i % 2 ? -459 : -511);
    const double near_big = from_bits(glibc_hypot_detail::bits(big) + (int64_t)(next_u64() % 9) - 4);
    const double near_tiny = from_bits(glibc_hypot_detail::bits(tiny) + (int64_t)(next_u64() % 9) - 4);
    check(near_big, near_big * std::ldexp(1.0 + uniform(), -(int)(next_u64() % 70)));
    check(near_tiny, near_tiny * std::ldexp(1.0 + uniform(), (int)(next_u64() % 70)));
    const double x = std::ldexp(1.0 + uniform(), (int)(next_u64() % 1400) - 700);
    const double r = from_bits(glibc_hypot_detail::bits(std::ldexp(1.0, -54)) + (int64_t)(next_u64() % 9) - 4);
    check(x, x * r * (1.0 + (double)((int64_t)(next_u64() % 5) - 2) * 0x1p-52));
  }
  std::printf("pairs %ld mismatches %ld probe %d\n", g_pairs, g_mismatches, glibc_hypot_matches_libm() ? 1 : 0);
  return 0;
}
