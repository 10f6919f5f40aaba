// moog_common.cuh -- shared declarations of the libmoog_b200 translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "../../include/moog_b200.h"

namespace moog {

// Parsed view of a program blob (pointers may be host or device).
struct ProgramView {
  const int32_t *hdr;
  const moog_op *ops;
  const int32_t *ipool;
  const moog_ex *expr;
  const int32_t *voff;
  const double *dpool;
};

__host__ __device__ inline ProgramView view_of(const void *blob) {
  ProgramView v;
  v.hdr = (const int32_t *)blob;
  v.ops = (const moog_op *)(v.hdr + MOOG_HDR_WORDS);
  v.ipool = (const int32_t *)(v.ops + v.hdr[MOOG_H_N_OPS]);
  int npool = (v.hdr[MOOG_H_N_IPOOL] + 1) & ~1;
  v.expr = (const moog_ex *)(v.ipool + npool);
  v.voff = v.ipool + v.hdr[MOOG_H_VOFF];
  v.dpool = (const double *)(v.expr + v.hdr[MOOG_H_N_EXPR]);
  return v;
}

enum StepMode { MODE_ENV_STEP = 0, MODE_PHYSICS = 1, MODE_POST_RESET = 2, MODE_OVERLAP = 3 };

struct StepArgs {
  const void *blob;  // device copy of the program
  const uint16_t *vmap;  // [VT] cached vertex -> slot << 8 | index within the slot's outline (255: beyond 254)
  moog_state st;
  int n_envs;
  int mode;
  int S, L, K, VT, NF, CMW;  // program dimensions (filled in by launch_step from the header)
  int dcv_tile;              // contained vertices per pass of the directed search (launch_step)
  const int *order;          // [n_envs] env handled by CTA i, or nullptr = identity
  int *cost;                 // [n_envs] SM cycles >> 6 this call cost each env, or nullptr
  int *done;                 // nullptr or [1 + n_envs], zeroed: count, then env + 1 in finishing order
  int *sm_active;            // nullptr or [256], zeroed: envs being stepped on each SM right now
  int trace;                 // MOOG_TRACE_TIMES=1: io.counters[n][6..7] = globaltimer at start / finish
  moog_step_io io;
  // io.frames when the step kernel draws them itself (StepPlan::fuse), else nullptr, and the
  // shared-memory offset of the renderer's buffers behind the part of the env record it reads
  uint8_t *frames;
  int render_off;
  moog_state pool;  // valid iff io.pool != nullptr
  // MODE_OVERLAP
  int layer_a, layer_b;
  uint8_t *overlap_out;
};

struct RenderArgs {
  const void *blob;
  int view_off;         // int32 word of the blob where the view's MOOG_VIEW_WORDS settings start
  moog_state st;
  int n_envs;
  uint8_t *frames;
  long long *trace;     // MOOG_TRACE_TIMES=1: the step's counters; [n][4..5] = globaltimer at render start / end
  const int *resample;  // anti_aliasing > 1: device copy of resample_tables()
  int ksize_h, ksize_v;
};

struct ObserveArgs {
  moog_state st;
  float *out;  // [n_envs][S][MOOG_OBS_COLS]
  int n_envs, S, L;
  int layer_off[MOOG_MAX_LAYERS + 1];
};

struct RayArgs {
  const void *blob;     // device copy of the program (its voff table)
  moog_state st;
  float *out;           // [n_envs][n_rays][2]
  const double *dirs;   // [n_rays][2]
  double max_range;
  int n_envs, S, L, VT, n_rays;
  int agent_layer, agent_index;
  unsigned layers;      // bit l: layer l holds targets
  int layer_off[MOOG_MAX_LAYERS + 1];
};

// Launch options of one program (moog_program_set_option / the MOOG_* environment variables, which
// are read ONCE, when the program is created).  -1 / 0 = decided by the library.
struct LaunchOptions {
  int helper = -1;            // "helper": second warp per env for one direction of _get_collision_vectors
  int ctas_per_sm = 0;        // "ctas_per_sm": envs resident per SM (the shared-memory request is padded to cap it)
  int trace_times = 0;        // "trace_times": per-env globaltimer stamps in io.counters (diagnostic)
  int seed = 0;               // "seed": the draws of moog_env_post_reset (which has no io.seed of its own)
};
LaunchOptions launch_options_from_env();
bool set_launch_option(LaunchOptions &o, const char *name, int value);

// host-side launchers (defined in the .cu files)
constexpr int kMaxForceOps = 32;
int env_smem_bytes(const int32_t *hdr, bool helper = true);
int candidate_matrix_words(const void *host_blob);
// How a step call launches its batch (plan_step is the one place that decides it).
struct StepPlan {
  bool ordered;    // envs dispatched longest-first by the costs of the previous call (launch_order)
  int resident;    // envs resident per SM the shared-memory request is padded to (0: as many as fit)
  bool helper;     // every env's CTA gets a second warp for one direction of _get_collision_vectors
  size_t smem;     // dynamic shared memory of one step CTA
  bool fuse;       // the step kernel draws io.frames itself, its canvas at render_off
  int render_off;
  bool tail;       // io.frames drawn by the persistent tail render kernel behind the step (StepArgs::done)
};
// mode: StepMode; frames: io.frames wanted (MODE_ENV_STEP); sms: multiprocessors of the device
StepPlan plan_step(const int32_t *host_hdr, int mode, int n_envs, bool frames, int sms, const LaunchOptions &opt);
cudaError_t launch_step(const StepArgs &a, const int32_t *host_hdr, const StepPlan &plan, cudaStream_t stream,
                        int *n_launches);
cudaError_t launch_order(const int *cost, int *order, int n, cudaStream_t stream, int *n_launches);
int resample_tables(int H, int W, int OH, int OW, std::vector<int> &table, int *ksize_h, int *ksize_v);
int lanczos_ksize(int in_size, int out_size);
// How the render kernels draw a view (the one place that decides it; moog_render_plan exposes it).
// rows: canvas rows drawn at once -- the whole canvas, a band (anti_aliasing 1) or a chunk
// (anti_aliasing > 1, streamed through the Lanczos resize); ring: rows of the horizontally resampled
// ring (anti_aliasing > 1); P threads per canvas row, T per env; env_bytes: shared memory per env.
// ok == false: no band / chunk fits one CTA's shared memory.
struct RenderPlan { bool ok; int rows, ring, P, T, env_bytes; };
RenderPlan render_plan(const int32_t *host_hdr, const int32_t *host_view);
// done: nullptr, or the finished-env list of the step kernel launched just before on `stream`
// (StepArgs::done, with StepArgs::sm_active behind it): the persistent tail render kernel is then
// launched with programmatic stream serialization, starts while the last envs are still being
// stepped and draws the envs in finishing order.
// plan: render_plan of the view (the program keeps one per view); host_view: the host copy of the
// words at a.view_off (the view's settings)
cudaError_t launch_render(const RenderArgs &a, const RenderPlan &plan, const int32_t *host_view, cudaStream_t stream,
                          int *n_launches, int *done = nullptr, int n_done = 0);
// moog_render_mask: a.view_off locates the mask row, a.frames is the int16 [n_envs][H][W] destination;
// plan: render_plan of the mask row (anti_aliasing 1: its bands are an anti_aliasing 1 frame's)
cudaError_t launch_mask(const RenderArgs &a, const RenderPlan &plan, cudaStream_t stream, int *n_launches);
// moog_observe_sprites (moog_observe.cu): one warp per env
cudaError_t launch_observe(const ObserveArgs &a, cudaStream_t stream, int *n_launches);
// moog_ray_sensor (moog_rays.cu): one CTA per env, one thread per ray
cudaError_t launch_ray_sensor(const RayArgs &a, cudaStream_t stream, int *n_launches);
// ints behind the finished list that launch_render's tail kernel uses: a ticket counter and the
// per-SM count of envs being stepped
constexpr int kTailExtraInts = 1 + 256;

}  // namespace moog
