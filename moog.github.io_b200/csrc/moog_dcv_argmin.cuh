// moog_dcv_argmin.cuh -- stage B of the directed collision search (moog_step.cu,
// directed_collision_vectors_impl): np.argmin over the edges of every contained vertex
// (collisions.py:150-180), taken over the list of crossing (vertex, edge) pairs 32 pairs at a time.
// The list is in ascending (vertex, edge) order, so the pairs of one vertex are one segment of it,
// and a segment may go on from one pass into the next.  Kept in a header of its own so that a test
// can run it on lists no scene produces.
#pragma once
#include <math.h>

namespace moog {

// np.argmin order of |1 - A|: a NaN beats everything, then the smaller value (|1 - A| >= 0, so its
// bit pattern orders like the value); ties go to the smaller index.  Every key is at most
// dcv_argmin_key(-inf) = bits(+inf) + 1, the key of an edge that does not cross.
__device__ __forceinline__ unsigned long long dcv_argmin_key(double A) {
  const double ab = fabs(1.0 - A);
  return isnan(ab) ? 0ull : (unsigned long long)__double_as_longlong(ab) + 1ull;
}

// the running winner of the segment that the previous pass ended in (t = its vertex, -1: none)
struct DcvCarry {
  int t = -1, ed = 0;
  unsigned long long key = 0;
  double a = 0;
};

// One pass, lane = pair: `act` (false past the last pair), vertex t, edge ed, cross_a A;
// t_after = vertex of the first pair of the next pass (255 when there is none).  Returns true on
// the lane that holds the last pair of a vertex's segment, with the vertex's winning edge and its
// cross_a in w_ed / w_a: np.argmin of the vertex's row, where every edge that does not cross holds
// -inf.  Updates `c` for the next pass.
__device__ __forceinline__ bool dcv_argmin_pass(bool act, int t, int ed, double A, int t_after, int lane,
                                                DcvCarry &c, int &w_ed, double &w_a) {
  const unsigned FULLW = 0xffffffffu;
  const unsigned long long KEY_INF = (unsigned long long)__double_as_longlong(INFINITY) + 1ull;
  unsigned long long key = act ? dcv_argmin_key(A) : ~0ull;
  // segments: the pairs of one vertex (idle lanes: one segment of their own)
  const int sv = act ? t : 255;
  const int sv_prev = __shfl_up_sync(FULLW, sv, 1), sv_next = __shfl_down_sync(FULLW, sv, 1);
  const unsigned heads = __ballot_sync(FULLW, lane == 0 || sv_prev != sv);
  const bool last = sv != (lane == 31 ? t_after : sv_next);
  const int seg0 = 31 - __clz(heads & ((2u << lane) - 1u));
  // a prefix minimum inside the segments, the earlier pair winning ties, over as many doubling
  // steps as the longest segment of the pass needs -- the one that goes on into the next pass
  // (lane 31's) included: its minimum so far is carried
  const int span = __reduce_max_sync(FULLW, act && (last || lane == 31) ? lane - seg0 + 1 : 0);
  int wl = lane;
#pragma unroll 1
  for (int d = 1; d < span; d <<= 1) {
    const unsigned long long okey = __shfl_up_sync(FULLW, key, d);
    const int owl = __shfl_up_sync(FULLW, wl, d);
    if (lane - d >= seg0 && !(key < okey)) { key = okey; wl = owl; }
  }
  w_ed = __shfl_sync(FULLW, ed, wl);
  w_a = __shfl_sync(FULLW, A, wl);
  if (sv == c.t && !(key < c.key)) { key = c.key; w_ed = c.ed; w_a = c.a; }  // the carried pairs came first
  if (t_after != 255) {
    c.t = __shfl_sync(FULLW, sv, 31);
    c.key = __shfl_sync(FULLW, key, 31);
    c.ed = __shfl_sync(FULLW, w_ed, 31);
    c.a = __shfl_sync(FULLW, w_a, 31);
  }
  // a minimum of bits(+inf) + 1 is edge 0's key too, and edge 0 comes first: its cross_a is +-inf
  // when it crosses, -inf when it does not
  if (key == KEY_INF) {
    if (w_ed != 0) w_a = -INFINITY;
    w_ed = 0;
  }
  return act && last;
}

}  // namespace moog
