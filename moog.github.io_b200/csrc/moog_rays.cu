// moog_rays.cu -- RaySensor (moog/observers/pil_renderer.py): range-finder rays from an agent sprite to the
// first outline they cross, out[N][n_rays][2] float32 (include/moog_b200.h moog_ray_sensor).
//
// A launch of its own behind the step, like moog_observe_kernel.  One CTA per env, one thread per ray.
//   1. The target edges (every edge of every live slot of the target layers but the agent's, in slot
//      order) are numbered by a scan of the slots' vertex counts.
//   2. Even-odd test of the origin against every target slot: the last slot that holds the origin reads
//      t = 0 on every ray, so the edges of that slot and of the slots before it cannot change a reading
//      and are never walked.
//   3. The remaining edges are staged tile by tile in shared memory as e = b - a, w = a - o and w x e
//      (the parts of the hit formulas that do not depend on the ray); every ray walks each tile in
//      edge order and keeps the smallest t, a tie going to the later edge.
// The hit test divides only for edges that pass exact division-free rejections (ray_maybe_hits), so
// the readings are those of the formulas evaluated as written for every edge.
#include <math.h>

#include "moog_common.cuh"

namespace moog {
namespace {

constexpr int kRayTile = 128;  // edges staged per pass (7.3 KB of shared memory in all, so that many one-warp CTAs share an SM)

__device__ __forceinline__ bool ray_maybe_hits(double D, double U, double T, double best) {
  // false only when RN(U / D) is outside [0, 1], RN(T / D) < 0 or RN(T / D) > best, the quotients the
  // hit test below evaluates (U, T, D: u's and t's numerators and the denominator, signs normalised so
  // that D > 0).  Every rejection needs |quotient| well away from the limit it fails, checked by
  // scaling with powers of two (exact) and by differences that are exact (Sterbenz) whenever they
  // decide; NaNs fail every comparison and pass on to the division.  D outside [2^-900, 2^900] (no
  // scaling below can over- or underflow then) and best below 2^-1000 are left to the division.
  if (!(D >= 0x1p-900 && D <= 0x1p900)) return true;
  if (U < 0.0 && -U * 0x1p1000 > D) return false;                  // u < 0, not a -0 underflow
  if (U > D && (U - D) * 0x1p30 > D) return false;                 // u > 1 + 2^-30
  if (T < 0.0 && -T * 0x1p1000 > D) return false;                  // t < 0, not a -0 underflow
  if (best >= 0x1p-1000) {
    const double B = best * D;                                     // rounded, normal: relative error 2^-53
    if (B >= 0x1p-900 && T > B && (T - B) * 0x1p30 > B) return false;   // t > best (1 + 2^-31)
  }
  return true;
}

__global__ void __launch_bounds__(256) moog_ray_sensor_kernel(RayArgs a) {
  __shared__ double s_ex[kRayTile], s_ey[kRayTile], s_wx[kRayTile], s_wy[kRayTile], s_tn[kRayTile];
  __shared__ int16_t s_slot[kRayTile];
  __shared__ int s_first[MOOG_MAX_SLOTS + 1];  // first target edge of each slot (exclusive scan of nv)
  __shared__ int s_odd[MOOG_MAX_SLOTS];        // crossings of the even-odd test, mod 2
  __shared__ int s_inside;                     // last target slot that holds the origin, or -1
  const int n = blockIdx.x, t = threadIdx.x, T = blockDim.x;
  const int S = a.S, R = a.n_rays;
  const ProgramView pv = view_of(a.blob);
  const double *dyn = a.st.dyn + (size_t)n * MOOG_DYN_FIELDS * S;
  const int32_t *meta = a.st.meta + (size_t)n * MOOG_META_FIELDS * S;
  const int32_t *cnt = a.st.cnt + (size_t)n * MOOG_MAX_LAYERS;
  const double2 *vtx = (const double2 *)(a.st.vtx + (size_t)n * a.VT * 2);
  float2 *out = (float2 *)(a.out + (size_t)n * R * 2);
  const int agent = a.layer_off[a.agent_layer] + a.agent_index;
  if (a.agent_index >= cnt[a.agent_layer]) {   // no origin: every ray reads "no hit"
    for (int r = t; r < R; r += T) out[r] = make_float2(1.f, -1.f);
    return;
  }
  const double ox = dyn[MOOG_D_X * S + agent], oy = dyn[MOOG_D_Y * S + agent];

  // 1. edges per slot (0 unless a live target other than the agent), scanned by warp 0
  if (t < 32) {
    int carry = 0;
    for (int base = 0; base < S; base += 32) {
      const int s = base + t;
      int e = 0;
      if (s < S) {
        int layer = 0;
        for (int l = 1; l < a.L; ++l) layer += s >= a.layer_off[l];
        const bool live = s - a.layer_off[layer] < cnt[layer];
        if (live && ((a.layers >> layer) & 1u) && s != agent) e = max(meta[MOOG_M_NV * S + s], 0);
      }
      int incl = e;
#pragma unroll
      for (int k = 1; k < 32; k <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, k);
        if (t >= k) incl += v;
      }
      if (s < S) s_first[s] = carry + incl - e;
      carry += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (t == 0) { s_first[S] = carry; s_inside = -1; }
  }
  for (int s = t; s < S; s += T) s_odd[s] = 0;
  __syncthreads();
  const int E = s_first[S];

  // the slot of target edge k: the last slot whose first edge is <= k (and that owns an edge)
  auto slot_of = [&](int k) {
    int lo = 0, hi = S - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (s_first[mid] <= k) lo = mid; else hi = mid - 1;
    }
    return lo;
  };
  auto edge_ends = [&](int k, int s, double2 &p, double2 &q) {
    const int j = k - s_first[s], nv = s_first[s + 1] - s_first[s], v = pv.voff[s];
    p = vtx[v + j];
    q = vtx[v + (j + 1 < nv ? j + 1 : 0)];
  };

  // 2. even-odd rule: edges with (a.y > o.y) != (b.y > o.y) and o.x < a.x + (o.y - a.y)(b.x - a.x) / (b.y - a.y)
  for (int k = t; k < E; k += T) {
    const int s = slot_of(k);
    double2 p, q;
    edge_ends(k, s, p, q);
    if ((p.y > oy) != (q.y > oy) && ox < p.x + (oy - p.y) * (q.x - p.x) / (q.y - p.y)) atomicXor(&s_odd[s], 1);
  }
  __syncthreads();
  for (int s = t; s < S; s += T)
    if (s_odd[s]) atomicMax(&s_inside, s);
  __syncthreads();
  const int inside = s_inside;

  // 3. the rays
  double dx = 0.0, dy = 0.0;
  if (t < R) { dx = a.dirs[2 * t]; dy = a.dirs[2 * t + 1]; }
  double best = inside >= 0 ? 0.0 : a.max_range;
  int hit = inside;
  for (int base = inside >= 0 ? s_first[inside + 1] : 0; base < E; base += kRayTile) {
    const int m = min(kRayTile, E - base);
    __syncthreads();   // the previous tile is no longer read
    for (int i = t; i < m; i += T) {
      const int s = slot_of(base + i);
      double2 p, q;
      edge_ends(base + i, s, p, q);
      const double ex = q.x - p.x, ey = q.y - p.y, wx = p.x - ox, wy = p.y - oy;
      s_ex[i] = ex; s_ey[i] = ey; s_wx[i] = wx; s_wy[i] = wy;
      s_tn[i] = wx * ey - wy * ex;
      s_slot[i] = (int16_t)s;
    }
    __syncthreads();
    if (t < R) {
      for (int i = 0; i < m; ++i) {
        const double ex = s_ex[i], ey = s_ey[i], wx = s_wx[i], wy = s_wy[i], tn = s_tn[i];
        const double den = dx * ey - dy * ex;   // d x e
        const double un = wx * dy - wy * dx;    // w x d
        const bool neg = den < 0.0;
        if (den != 0.0 && ray_maybe_hits(neg ? -den : den, neg ? -un : un, neg ? -tn : tn, best)) {
          const double tt = tn / den, u = un / den;
          if (u >= 0.0 && u <= 1.0 && tt >= 0.0 && tt <= best) {
            best = tt;
            hit = s_slot[i];
          }
        }
      }
    }
  }
  if (t < R)
    out[t] = hit >= 0 ? make_float2(__double2float_rn(best / a.max_range), (float)hit) : make_float2(1.f, -1.f);
}

}  // namespace

cudaError_t launch_ray_sensor(const RayArgs &a, cudaStream_t stream, int *n_launches) {
  const int threads = (a.n_rays + 31) / 32 * 32;
  moog_ray_sensor_kernel<<<a.n_envs, threads, 0, stream>>>(a);
  if (n_launches) *n_launches += 1;
  return cudaGetLastError();
}

}  // namespace moog
