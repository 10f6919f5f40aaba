/*
 * moog_b200.h -- C ABI of libmoog_b200.so, the B200-native batched
 * implementation of MOOG's Environment.step hot path.
 *
 * MOOG has no FFI of its own: its boundary is the Python component API
 * (moog/environment.py:28-35 Environment(state_initializer, physics, task,
 * action_space, observers, game_rules)).  The host package compiles those
 * component objects into a flat "program" blob (include/moog_b200_program.h)
 * and drives the entry points below, each of which replaces one stretch of the
 * reference's per-env Python loop for N envs at once.  All `moog_state` pointers
 * and all array arguments are DEVICE pointers owned by the caller (torch
 * tensors in the Python host); the library never allocates or frees them.
 * Every call enqueues kernels on `stream` (a cudaStream_t passed as void*) and
 * returns without synchronising.
 *
 * Return value: 0 on success, a negative MOOG_E_* code on a configuration /
 * launch error (moog_strerror gives the text).  Data-dependent reference
 * exceptions (ValueError of collisions.py:323-326, tether_physics.py:192-196)
 * are not return codes: they set bits in the env's envi[MOOG_EI_ERR] word and
 * the host raises them lazily.
 */
#ifndef MOOG_B200_H_
#define MOOG_B200_H_

#include <stddef.h>
#include <stdint.h>

#include "moog_b200_program.h"

#ifdef __cplusplus
extern "C" {
#endif

#define MOOG_E_INVAL (-1)    /* bad argument / malformed program blob          */
#define MOOG_E_CUDA (-2)     /* a CUDA runtime call failed (see moog_last_cuda_error) */
#define MOOG_E_TOO_BIG (-3)  /* one env record does not fit in shared memory   */
#define MOOG_E_UNSUPPORTED (-4)

#define MOOG_N_COUNTERS 8

typedef struct moog_program moog_program;

/* Device pointers to the SoA state record of N envs (layout: moog_b200_program.h). */
typedef struct {
  double *dyn;   /* [N][MOOG_DYN_FIELDS][S]  */
  double *stat;  /* [N][MOOG_STAT_FIELDS][S] */
  int32_t *meta; /* [N][MOOG_META_FIELDS][S] */
  int32_t *cnt;  /* [N][MOOG_MAX_LAYERS]     */
  int32_t *envi; /* [N][MOOG_ENVI_WORDS]     */
  double *envf;  /* [N][hdr[MOOG_H_N_ENVF]]  */
  double *vtx;   /* [N][VT][2]               */
} moog_state;

/* Optional inputs / outputs of moog_env_step (any pointer may be NULL). */
typedef struct {
  const double *actions;    /* [N][action_dim]; NULL = zeros (joystick.py:45, grid.py:52)       */
  const double *noise;      /* [N][K][noise_dim] uniforms in [0,1) behind RandomForce
                               (random_force.py:22-26); NULL = device Philox stream             */
  const double *rule_noise; /* [N][rule_noise_dim] uniforms behind ModifySprites(sample_one)
                               (modify_sprites.py:48-49); NULL = device Philox stream           */
  const moog_state *pool;   /* initial states an env that terminated on the previous call is
                               re-initialised from (environment.py:100-101 -> reset());
                               NULL = terminated envs keep stepping (no auto-reset)             */
  int32_t pool_size;
  const int32_t *reset_index; /* [N] pool entry to use, NULL = hash(seed, env, episode)         */
  uint64_t seed;
  float *reward;       /* [N]  TimeStep.reward   (NaN on a FIRST step: dm_env's None)           */
  int32_t *step_type;  /* [N]  MOOG_STEP_FIRST / MID / LAST                                     */
  float *discount;     /* [N]  1 mid, 0 last, NaN first                                         */
  int64_t *counters;   /* [N][MOOG_N_COUNTERS]: overlaps_sprite calls, calls that returned True,
                          resolved collisions, order-sensitive hash of the True (slot_a, slot_b)
                          events, SM cycles the env's warp spent in the kernel, 3 spare          */
  double *stats;       /* [4]  += sum reward, sum finished-episode length, finished episodes,
                          env-steps; the only quantity ever reduced across GPUs                 */
  int32_t sample_resets; /* non-zero (and the program has MOOG_Z_* ops): an env that resets takes
                            pool entry 0 as its template and draws its generated sprites afresh on
                            the device (Philox keyed by seed, env, episode) instead of copying a
                            whole pool entry                                                       */
  uint8_t *frames;     /* [N][H][W][3] or NULL: PILRenderer.__call__ (pil_renderer.py:88-120) of the state
                          every env is left in, as moog_render would draw it after this call.  When the
                          canvas fits next to the env record in shared memory the step kernel draws it
                          itself, env by env as they finish, otherwise the render kernel follows.  Any
                          device-accessible address: HBM, or pinned host memory (cudaHostAlloc /
                          cudaHostRegister under unified addressing) for frames the host reads          */
} moog_step_io;

/* Checks a program blob without touching the GPU: every section start / count, pool index, layer id,
 * expression start and sampler table an op refers to lies inside the blob (moog_program_create runs it
 * first).  0, or MOOG_E_INVAL.  (No reference counterpart: the reference passes Python objects.) */
int moog_program_validate(const void *blob, size_t nbytes);

/* Upload a compiled program (host pointer to the blob).  Replaces nothing in the
 * reference: it is the device-side image of the component objects passed to
 * Environment.__init__ (moog/environment.py:28-68). */
int moog_program_create(const void *blob, size_t nbytes, moog_program **out);
void moog_program_destroy(moog_program *p);

/* Bytes of shared memory one env record occupies inside the step kernel. */
int moog_program_env_smem_bytes(const moog_program *p);

/* Environment.step for N envs (moog/environment.py:98-126): game rules ->
 * action space -> Physics.step (K substeps of forces, Collision, correctives,
 * Euler integration: moog/physics/physics.py:88-117, abstract_physics.py:39-42)
 * -> step_count += 1 -> task.reward.  Envs whose previous step terminated are
 * re-initialised from `pool` and run the post-reset sequence of
 * environment.py:82-96 instead (their action is ignored, step_type = FIRST). */
int moog_env_step(moog_program *p, const moog_state *st, int n_envs, const moog_step_io *io,
                  void *stream);

/* The part of Environment.reset after the state initializer ran
 * (moog/environment.py:88-96): task / action-space reset, every rule reset and
 * stepped once, step_count = 0. */
int moog_env_post_reset(moog_program *p, const moog_state *st, int n_envs, const double *rule_noise,
                        void *stream);

/* AbstractPhysics.step alone (moog/physics/abstract_physics.py:39-42). */
int moog_physics_step(moog_program *p, const moog_state *st, int n_envs, const double *noise,
                      int64_t *counters, void *stream);

/* Sprite.overlaps_sprite (moog/sprite.py:462-484) for every (i, j) of two
 * layers of every env: out[N][cap_a][cap_b] uint8 (contact_rules.py:15-35). */
int moog_overlap_pairs(moog_program *p, const moog_state *st, int n_envs, int layer_a, int layer_b,
                       uint8_t *out, void *stream);

/* PILRenderer.__call__ (moog/observers/pil_renderer.py:88-120) for N envs:
 * frames[N][H][W][3] uint8, row 0 = top. */
int moog_render(moog_program *p, const moog_state *st, int n_envs, uint8_t *frames, void *stream);

/* moog_render for view `view` of a config with several PILRenderer observers (views: moog_b200_program.h
 * MOOG_H_VIEWS): frames[N][H_view][W_view][3] uint8 with that renderer's settings; view 0 is what
 * moog_render draws.  A launch of its own on `stream`, like moog_observe_sprites: call it after
 * moog_env_step (whose io.frames is view 0) to draw the other views of the state that call left.  `frames`
 * is any device-accessible address aligned to 16 bytes: HBM, or pinned host memory.  MOOG_E_INVAL for a
 * NULL program / state / frames, n_envs < 0, a misaligned frames, a program without a renderer or a view
 * outside [0, 1 + hdr[MOOG_H_N_VIEWS]). */
int moog_render_view(moog_program *p, const moog_state *st, int n_envs, int view, uint8_t *frames, void *stream);

/* How the render kernel draws view `view` of a program blob, without touching the GPU (like
 * moog_program_validate, which it runs first).  The canvas (anti_aliasing x the image size) is drawn
 * *chunk_rows rows at a time: the whole canvas, a band (anti_aliasing 1) or a chunk streamed through
 * the Lanczos resize (anti_aliasing > 1); *smem_bytes of shared memory per env.  Either pointer may
 * be NULL.  0; MOOG_E_INVAL for a malformed blob, a program without a renderer or a view outside
 * [0, 1 + hdr[MOOG_H_N_VIEWS]); MOOG_E_UNSUPPORTED for a view no chunk size can hold in one CTA's
 * shared memory (moog_render, moog_render_view and moog_env_step with io.frames refuse it the same way,
 * before launching anything). */
int moog_render_plan(const void *blob, size_t nbytes, int view, int *chunk_rows, int *smem_bytes);

/* SpriteMask `mask` of N envs (no reference counterpart; moog_b200_program.h MOOG_H_MASKS): out[N][H][W] int16,
 * row 0 = top as in the frames, each pixel the slot of the last sprite in draw order whose Pillow polygon
 * fill covers it (the fill the frames use, at the mask's image size and polygon modifier; sprites whose
 * ink alpha byte is 0 are left out), -1 where none does.  A launch of its own on `stream`, like
 * moog_render_view: call it after moog_env_step to draw the masks of the state that call left.  `out` is
 * any device-accessible address aligned to 16 bytes: HBM, or pinned host memory.  MOOG_E_INVAL for a NULL
 * program / state / out, n_envs < 0, a misaligned out or a mask outside [0, hdr[MOOG_H_N_MASKS]);
 * MOOG_E_UNSUPPORTED for a mask no band holds (moog_mask_plan). */
int moog_render_mask(moog_program *p, const moog_state *st, int n_envs, int mask, int16_t *out, void *stream);

/* How the mask kernel draws mask `mask` of a program blob, without touching the GPU (like
 * moog_render_plan): *band_rows rows at a time, *smem_bytes of shared memory per env; either pointer
 * may be NULL.  0; MOOG_E_INVAL for a malformed blob or a mask outside [0, hdr[MOOG_H_N_MASKS]);
 * MOOG_E_UNSUPPORTED for a mask no band can hold in one CTA's shared memory (TorusGeometry over outlines
 * as large as cleanup's). */
int moog_mask_plan(const void *blob, size_t nbytes, int mask, int *band_rows, int *smem_bytes);

/* RawState.__call__ (moog/observers/raw_state.py:17-19) for N envs: every sprite slot's state as
 * out[N][S][MOOG_OBS_COLS] float32 (layout and columns: moog_b200_program.h MOOG_OBS_*).  A launch of its
 * own on `stream`, so call it after moog_env_step to observe the state that call left.  `out` is any
 * device-accessible address aligned to 16 bytes: HBM, or pinned host memory as for moog_step_io.frames.
 * MOOG_E_INVAL for a NULL program / state / out, n_envs < 0 or a misaligned out; n_envs == 0 launches
 * nothing. */
int moog_observe_sprites(moog_program *p, const moog_state *st, int n_envs, float *out, void *stream);

/* One RaySensor (no reference counterpart; moog/observers/pil_renderer.py RaySensor): n_rays rays from the
 * position of slot layer_off[agent_layer] + agent_index.  Target slots: the live slots of the layers whose
 * bit is set in `layers`, except the agent's own.  dirs is a DEVICE pointer to [n_rays][2] float64
 * directions (cos phi_k, sin phi_k), computed by the host. */
typedef struct {
  int32_t agent_layer;
  int32_t agent_index;
  uint32_t layers;     /* bit l: layer l holds targets */
  int32_t n_rays;      /* 1 .. 256 */
  double max_range;    /* finite, > 0 */
  const double *dirs;  /* [n_rays][2], 8-byte aligned */
} moog_ray_spec;

/* RaySensor readings of N envs: out[N][n_rays][2] float32.  For ray k with direction d from origin o, every
 * edge (a, b) of a target slot's closed outline (its MOOG_M_NV cached world vertices, vertex j joined to
 * vertex (j + 1) mod nv) is tested in float64, formulas as written: e = b - a, w = a - o, den = d x e,
 * t = (w x e) / den, u = (w x d) / den, a hit when den != 0, 0 <= u <= 1 and t >= 0 (a x b = a.x b.y - a.y b.x).
 * A slot whose outline holds o by the even-odd rule (edges with (a.y > o.y) != (b.y > o.y) and
 * o.x < a.x + (o.y - a.y)(b.x - a.x) / (b.y - a.y)) reads t = 0.  The reading is (float(t / max_range), slot)
 * for the smallest t <= max_range over the target slots, a tie going to the later slot, and (1, -1) when
 * there is none or the agent layer holds no sprite at agent_index.  No wrapping under TorusGeometry.  A
 * launch of its own on `stream`, like moog_observe_sprites: call it after moog_env_step.  `out` is any
 * device-accessible address aligned to 16 bytes: HBM, or pinned host memory.  MOOG_E_INVAL for a NULL
 * program / state / spec / dirs / out, n_envs < 0, n_rays outside [1, 256], a max_range that is not finite
 * and > 0, an agent layer, an agent index < 0 or a target layer outside the program, a misaligned out or
 * dirs; nothing is launched then, nor for n_envs == 0. */
int moog_ray_sensor(moog_program *p, const moog_state *st, int n_envs, const moog_ray_spec *spec, float *out,
                    void *stream);

/* Host-side (CPU) polygon predicates for the HOST Sprite class only: the state
 * initializer's rejection sampling calls Sprite.overlaps_sprite /
 * contains_points (moog/state_initialization/sprite_generators.py:69-105,
 * moog/sprite.py:442-484) while it builds episodes.  Closed outlines
 * ([n][2] doubles, last vertex == first), matplotlib Path semantics.  Never
 * used by the step. */
int moog_host_paths_overlap(const double *a, int na, const double *b, int nb);
void moog_host_points_in_path(const double *pts, int np, const double *path, int nv, uint8_t *out);

const char *moog_strerror(int code);
const char *moog_last_cuda_error(void);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t moog_launch_count(void);
/* How moog_env_step launches a batch of n_envs on the current device: envs resident per SM
 * (0 = as many as fit), warps per env (2 = owner + helper warp), dynamic shared memory per
 * env in bytes.  The step is bound by its longest-running env; see DESIGN.md section 3.1. */
int moog_step_launch_info(const moog_program *p, int n_envs, int *resident_envs_per_sm, int *warps_per_env,
                          int *smem_bytes_per_env);

/* 1 when moog_env_step with io->frames draws the frames of a batch of n_envs inside the step
 * kernel (the canvas fits next to the env record without costing residency), 0 when the render
 * kernel follows the step kernel. */
int moog_step_draws_frames(const moog_program *p, int n_envs);

/* Launch options of a program (tuning / tests; the reference has no counterpart).  The MOOG_*
 * environment variables of the same names (MOOG_HELPER, MOOG_CTAS_PER_SM, MOOG_TRACE_TIMES) are
 * read once, when the program is created; this call changes one option of a live program: name in
 * {"helper", "ctas_per_sm", "trace_times", "seed"}, any other name is MOOG_E_INVAL.  "helper" 0 / 1:
 * the helper warp off / on, "ctas_per_sm": envs resident per SM for the step kernel; value -1
 * (helper) or 0 (ctas_per_sm) hands the decision back to the library.  "trace_times" 1: globaltimer
 * stamps of every env's step and render in io->counters (diagnostic).  None of the launch options
 * changes results; "seed" is the io.seed that moog_env_post_reset (which takes no moog_step_io) keys
 * the draws of its rules pass with (CreateSprites, random conditions). */
int moog_program_set_option(moog_program *p, const char *name, int value);

#ifdef __cplusplus
}
#endif
#endif /* MOOG_B200_H_ */
