// moog_seg_cross.cuh -- range tests on a quotient fl(n / d) decided without the division, for the
// per-pair paths of moog_step.cu: segments_intersect (the outline test) and unit_ratio (the
// crossing test of the directed search).  Kept in a header of its own so that a test can compare
// the decision with the division on operands no scene produces.
#pragma once
#include <math.h>

namespace moog {

// |x| in [2^(lo - 1023), 2^(hi - 1023)) for biased exponents lo < hi <= 2047, read from the exponent
// field of the high word; +-0, subnormals below 2^(lo - 1023), inf and NaN fail
__device__ __forceinline__ bool exp_field_in(double x, unsigned lo, unsigned hi) {
  const unsigned h = (unsigned)__double2hiint(x) & 0x7fffffffu;
  return h - (lo << 20) < ((hi - lo) << 20);
}

// matplotlib's range tests of one segment parameter u = fl(n / den) (src/_path.h, segments_intersect):
//   lower:  u > 0 || isclose_(u, 0)      upper:  u < 1 || isclose_(u, 1)
// with isclose_(a, b) = |a - b| <= max(1e-10 max(|a|, |b|), 1e-13).  For finite u they read
//   lower  <=>  u >= -1e-13                                  (|u| <= 1e-10 |u| only for u == 0)
//   upper  <=>  u < 1, or u in [1, 2] and u - 1 <= fl(1e-10 u)   (u - 1 exact there; for u > 2,
//               fl(u - 1) >= u / 2 > fl(1e-10 u))
// (the literals are the doubles nearest 1e-10 and 1e-13), while u = +-inf passes both (inf <= inf)
// and NaN fails both.
//
// Let N = n sign(den), D = |den| (exact), so u = fl(N / D).  Rounding is monotone and fixes the powers
// of two, so a bound N / D <= 2^k (or >=) carries over to u, and multiplying D by a power of two is
// exact in the regime below:
//   lower true   when N >= -2^-44 D:  u >= -2^-44 > -1e-13 (2^-44 = 5.7e-14)
//   lower false  when N <= -2^-43 D:  u <= -2^-43 < -1e-13 (2^-43 = 1.14e-13)
// With r = fl(N - D):  N <= D gives r <= 0;  D < N <= 2D makes r = N - D exactly (Sterbenz);
// N > 2D gives r >= fl(D) = D.  So
//   upper true   when r <= 2^-34 D:   u <= 1 + 2^-34, and u - 1 <= 2^-34 = 5.8e-11 < 1e-10 <= fl(1e-10 u)
//   upper false  when r >= 2^-33 D:   u >= 1 + 2^-33; on [1 + 2^-33, 2], u - 1 - 1e-10 u (1 + 2^-53)
//                                     grows with u and is > 0 at its left end (2^-33 = 1.16e-10);
//                                     past 2 see above
// Between those margins (-2^-43 D < N < -2^-44 D, or 2^-34 D < r < 2^-33 D) the decision is left to
// the division.  Regime: n == 0 or |n| in [2^-959, 2^961), and |den| in [2^-44, 2^1024).  Then |u| <
// 2^1005 never overflows, the scaled D stay normal, and r is exact or decided by its sign as above.
// Outside it (|den| < 2^-44 included, where u can overflow to the +-inf that passes both tests), and
// for +-inf and NaN operands, `exact` is false and the caller divides.
__device__ __forceinline__ bool seg_param_in_unit(double n, double den, bool &exact) {
  const double N = den < 0.0 ? -n : n, D = fabs(den);
  const double r = N - D;
  const bool lo_in = N >= -0x1p-44 * D, lo_out = N <= -0x1p-43 * D;
  const bool hi_in = r <= 0x1p-34 * D, hi_out = r >= 0x1p-33 * D;
  exact = (exp_field_in(n, 64u, 1984u) || n == 0.0) && exp_field_in(den, 979u, 2047u) && (lo_in || lo_out) &&
          (hi_in || hi_out);
  return lo_in && hi_in;
}

// (fl(n / d) >= 0 && fl(n / d) <= 1) without the division, for the crossing test of
// sprite.py:171-175.  Rounding to nearest is monotone and 0 and 1 are representable, so for
// finite operands whose quotient neither overflows nor underflows
//   fl(n/d) <= 1  <=>  n/d <= 1   (the smallest quotient above 1, (d + ulp)/d, is > 1 + 2^-53
//                                  and rounds to 1 + 2^-52)
//   fl(n/d) >= 0  <=>  n/d >= 0 or n == -0.0  (-0.0 >= 0 is true)
// and d == 0 gives +-inf or NaN, false either way.  `exact` is false when the operands are
// outside that regime -- |n| in [2^-959, 2^961) or n == 0, and |d| in [2^-959, 2^33) or d == 0,
// inside [1e-290, 1e290] and [1e-290, 1e10]; NaN / inf fail -- and the caller then divides.
__device__ __forceinline__ bool unit_ratio(double n, double d, bool &exact) {
  exact = (exp_field_in(n, 64u, 1984u) || n == 0.0) && (exp_field_in(d, 64u, 1056u) || d == 0.0);
  return d > 0.0 ? (n >= 0.0 && n <= d) : (d < 0.0 && n <= 0.0 && n >= d);
}

}  // namespace moog
