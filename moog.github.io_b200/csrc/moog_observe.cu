// moog_observe.cu -- RawState (moog/observers/raw_state.py:17-19) of N envs as float32 tensors:
// out[N][S][MOOG_OBS_COLS], layout in include/moog_b200_program.h (MOOG_OBS_*).
//
// A launch of its own behind the step rather than a phase of the step kernel: the step kernel is bound
// by its instruction footprint (DESIGN.md section 3.1), and this pass needs none of its shared state.
//
// One warp per env, lane = slot, 32 slots per pass.  Each lane loads the 14 record rows of its slot
// (unit stride across the warp, live slots only), converts them and writes its 64-byte output row into
// a padded shared-memory tile; the warp then stores the tile's 32 x 64 contiguous bytes with 16-byte
// stores, 512 contiguous bytes per warp store, so that writes into pinned host memory cross PCIe in
// whole lines.
#include "moog_common.cuh"

namespace moog {
namespace {

constexpr int kObsWarps = 4;                 // envs per CTA
constexpr int kObsRow = MOOG_OBS_COLS + 4;   // floats per tile row: 80 bytes keeps the float4 stores of
                                             // eight consecutive lanes on distinct banks

static_assert(MOOG_OBS_COLS == 16, "the tile moves one slot as four float4");

__global__ void __launch_bounds__(32 * kObsWarps) moog_observe_kernel(ObserveArgs a) {
  __shared__ __align__(16) float tile[kObsWarps][32 * kObsRow];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int n = blockIdx.x * kObsWarps + w;
  if (n >= a.n_envs) return;
  const int S = a.S;
  const double *dyn = a.st.dyn + (size_t)n * MOOG_DYN_FIELDS * S;
  const double *stat = a.st.stat + (size_t)n * MOOG_STAT_FIELDS * S;
  const int32_t *meta = a.st.meta + (size_t)n * MOOG_META_FIELDS * S;
  const int cnt_l = lane < a.L ? a.st.cnt[(size_t)n * MOOG_MAX_LAYERS + lane] : 0;
  float4 *dst = (float4 *)(a.out + (size_t)n * S * MOOG_OBS_COLS);
  float *row = &tile[w][lane * kObsRow];
  for (int base = 0; base < S; base += 32) {
    const int s = base + lane;
    int layer = 0;
    for (int l = 1; l < a.L; ++l) layer += s >= a.layer_off[l];
    const int cnt = __shfl_sync(0xffffffffu, cnt_l, layer);  // every lane: the mask names the whole warp
    const bool live = s < S && s - a.layer_off[layer] < cnt;
    float v[MOOG_OBS_COLS];
#pragma unroll
    for (int c = 0; c < MOOG_OBS_COLS; ++c) v[c] = 0.f;
    if (live) {
      v[MOOG_OBS_X] = __double2float_rn(dyn[MOOG_D_X * S + s]);
      v[MOOG_OBS_Y] = __double2float_rn(dyn[MOOG_D_Y * S + s]);
      v[MOOG_OBS_SHAPE] = (float)meta[MOOG_M_SHAPE * S + s];
      v[MOOG_OBS_ANGLE] = __double2float_rn(dyn[MOOG_D_ANG * S + s]);
      v[MOOG_OBS_SCALE] = __double2float_rn(stat[MOOG_S_SCALE * S + s]);
      v[MOOG_OBS_ASPECT] = __double2float_rn(stat[MOOG_S_ASPECT * S + s]);
      v[MOOG_OBS_C0] = __double2float_rn(stat[MOOG_S_C0 * S + s]);
      v[MOOG_OBS_C1] = __double2float_rn(stat[MOOG_S_C1 * S + s]);
      v[MOOG_OBS_C2] = __double2float_rn(stat[MOOG_S_C2 * S + s]);
      v[MOOG_OBS_OPACITY] = __double2float_rn(stat[MOOG_S_OPACITY * S + s]);
      v[MOOG_OBS_X_VEL] = __double2float_rn(dyn[MOOG_D_VX * S + s]);
      v[MOOG_OBS_Y_VEL] = __double2float_rn(dyn[MOOG_D_VY * S + s]);
      v[MOOG_OBS_ANGLE_VEL] = __double2float_rn(dyn[MOOG_D_ANGVEL * S + s]);
      v[MOOG_OBS_MASS] = __double2float_rn(stat[MOOG_S_MASS * S + s]);
      v[MOOG_OBS_ALIVE] = 1.f;
    }
    v[MOOG_OBS_LAYER] = (float)layer;
#pragma unroll
    for (int q = 0; q < MOOG_OBS_COLS / 4; ++q)
      *(float4 *)&row[4 * q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    __syncwarp();
    // this pass's slots [base, base + m) are the float4s [4 * base, 4 * (base + m)) of the env block
    const int nq = 4 * min(32, S - base);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = 32 * k + lane;
      if (i < nq) dst[4 * base + i] = *(const float4 *)&tile[w][(i >> 2) * kObsRow + 4 * (i & 3)];
    }
    __syncwarp();
  }
}

}  // namespace

cudaError_t launch_observe(const ObserveArgs &a, cudaStream_t stream, int *n_launches) {
  const int blocks = (a.n_envs + kObsWarps - 1) / kObsWarps;
  moog_observe_kernel<<<blocks, 32 * kObsWarps, 0, stream>>>(a);
  if (n_launches) *n_launches += 1;
  return cudaGetLastError();
}

}  // namespace moog
