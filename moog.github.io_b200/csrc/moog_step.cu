// moog_step.cu -- one-warp-per-env kernel for MOOG's Environment.step.
//
// Reference path (moog/environment.py:98-126): game rules -> action space ->
// Physics.step (K substeps: forces in itertools.product order, the rotational
// Collision, corrective physics, Euler integration) -> task reward.
//
// Execution model.  One warp owns one env.  The env's whole state record
// (positions, velocities, the cached world vertices, ...) is staged in shared
// memory for the duration of the step and written back once, so HBM sees one
// read and one write of the record per env-step.  Control flow is warp-uniform:
// every decision is taken on values all 32 lanes agree on (shared-memory reads,
// ballots, shuffled reductions).  Lanes are spent on the inner dimensions the
// reference loops over serially inside numpy / matplotlib:
//   * lane = second sprite of a layer pair      (broad phase, abstract_force loops)
//   * lane = polygon edge / vertex              (Path.intersects_path, contains_points,
//                                                segment_crossing_coefficients)
//   * lane = cached vertex                      (position / angle setters)
// The ORDER in which sprite pairs are visited is the reference's (physics.py:92-108):
// a Collision mutates positions and velocities the next pair sees, so pairs are
// never reordered -- the broad phase of the pairs (i, j0..j31) is evaluated in
// one shot and re-evaluated after every resolved contact of sprite i.
//
// Arithmetic is float64 with the reference's operation order (compiled with
// -fmad=false; fma() appears only where numpy's BLAS kernels fuse, see
// oracle/moog_oracle.c), because contact decisions and argmin / argmax ties are
// decided by the last bit.
#include <math.h>
#include <stdlib.h>

#include "moog_common.cuh"
#include "moog_dcv_argmin.cuh"
#include "moog_render_dev.cuh"
#include "moog_seg_cross.cuh"

namespace moog {

#define FULL 0xffffffffu
#define MAXV MOOG_MAX_VERTS
#define EPS_INTERP 1e-8 /* moog/sprite.py:35 */
#define EPS_COLL 1e-2   /* moog/physics/collisions.py:46 */

// Padding of the bounding boxes used to skip work whose result is provably
// "no intersection" (see DESIGN.md, "exact culling").
#define AABB_PAD 1e-7
#define SHORT_EDGE2 1e-8

#define SLF_SHORT_EDGE 1  // slot flag: some edge is shorter than 1e-4 -> serial matplotlib path
#define SLF_NONFINITE 2   // some cached vertex coordinate is NaN / inf -> no culling at all
#define SLF_ALLNAN 4      // every cached vertex coordinate is NaN -> overlaps nothing
// Some edge is vertical up to rounding but not exactly (0 < |dx| <= STEEP_DX).  matplotlib's
// segments_intersect calls two nearly parallel, nearly collinear segments intersecting when their
// X-INTERVALS overlap (unless x1 == x2 == x3 exactly, then the y-intervals decide): for such an edge
// the x-interval is a few ulps wide and the rule fires for segments that are far apart in y.  A
// collinearity tolerance of 1e-13 / |edge| bridges a gap of at most 1e-13 / |dx| along the line, so
// edges with |dx| > STEEP_DX stay inside the boxes' padding; a slot that has a steeper one gets a
// box that covers every y (culling on x stays exact) and the serial matplotlib path.
#define SLF_STEEP 8
#define SLF_MASK 15
#define STEEP_DX 1e-5

enum { KIND_WEAK = 0, KIND_F32 = 1, KIND_F64 = 2 };

struct SmemLayout {
  int rec, dyn, stat, aabb, aabb0, nskin, tmp, vtx, envf, ctr, meta, sflag, voff, cnt, envi, cmoff, cmask, nearp, hdr, scratch, xchg, mbar, plist, win_a, win_e, tile, vmap, total;
};

#define MOOG_MAX_FORCE_OPS 32
/* contained vertices per pass of _directed_collision_vectors: one pass covers any outline when the
   step is bound by its longest env (few envs per SM, shared memory to spare); the small tile keeps
   the record small when the batch is large and residency is what counts */
#define DCV_TILE_MAX 32
#define DCV_TILE_MIN 8
#define DCV_U 2 /* vertices (x edges) per trip of stage A1 of the directed search */
#define NEAR_SKIN 0.02
#define NEAR_CAP 512  /* near-list entries; more near pairs than this -> every pair is tested */

__host__ __device__ inline SmemLayout smem_layout(int S, int VT, int NF, int CMW, int warps, int tile) {
  SmemLayout L;
  int o = 0;
  L.rec = o;   o += 224;  // EnvRec (static_assert below)
  L.dyn = o;   o += 8 * MOOG_DYN_FIELDS * S;
  L.stat = o;  o += 8 * MOOG_STAT_FIELDS * S;
  L.aabb = o;  o += 8 * 4 * S;
  L.vtx = o;   o += 16 * VT;     // 16-byte aligned: everything before it is a multiple of 16
  L.envf = o;  o += 8 * NF;
  L.ctr = o;   o += 8 * 12;
  L.meta = o;  o += 4 * MOOG_META_FIELDS * S;
  L.sflag = o; o += 4 * S;
  L.aabb0 = o; o += 4 * 4 * S;  // float: box snapshot of the near list
  L.nskin = o; o += 4 * S;      // float: drift allowance per slot
  L.voff = o;  o += 4 * (S + 1);
  L.cnt = o;   o += 4 * MOOG_MAX_LAYERS;
  L.envi = o;  o += 4 * MOOG_ENVI_WORDS;
  L.cmoff = o; o += 4 * MOOG_MAX_FORCE_OPS;
  L.cmask = o; o += 4 * (CMW > 0 ? CMW : 1);
  L.nearp = o; o += CMW > 0 ? 4 * NEAR_CAP : 4;
  L.hdr = o;   o += 4 * MOOG_HDR_WORDS;
  L.scratch = o; o += 64 * warps;  // one per warp (owner, helper)
  o = (o + 15) & ~15;
  L.xchg = o;  o += 128;                  // main <-> helper: request words, the helper's CVec
  L.mbar = o;  o += 16;                   // mbarrier of the bulk (TMA) loads of the record
  L.tile = tile;
  L.plist = o; o += CMW > 0 ? 2 * 32 * tile * warps : 8;  // crossing (vertex, edge) pairs, per warp
  o = (o + 15) & ~15;
  // per warp, the directed search's winner of each contained vertex (up to 32): its edge's cross_a and the edge
  L.win_a = o; o += CMW > 0 ? 8 * 32 * warps : 0;
  L.win_e = o; o += CMW > 0 ? 32 * warps : 0;
  L.tmp = o;   o += 8 * 3 * S;  // (16-byte aligned) tether scratch (3 fields) / per-slot translations of the Euler pass
  L.vmap = o;  o += VT;  // cached vertex -> slot (integrate_all)
  L.total = (o + 15) & ~15;
  return L;
}

int env_smem_bytes(const int32_t *hdr, bool helper) {
  return smem_layout(hdr[MOOG_H_N_SLOTS], hdr[MOOG_H_N_VTX] > 0 ? hdr[MOOG_H_N_VTX] : 1, hdr[MOOG_H_N_ENVF],
                     hdr[MOOG_H_CMASK_WORDS], helper ? 2 : 1, helper ? DCV_TILE_MAX : DCV_TILE_MIN).total;
}

// words of the candidate matrices of all collision ops (see MOOG_H_CMASK_WORDS)
int candidate_matrix_words(const void *host_blob) {
  ProgramView pv = view_of(host_blob);
  int words = 0;
  for (int f = 0; f < pv.hdr[MOOG_H_N_FORCES]; ++f) {
    const moog_op *op = pv.ops + pv.hdr[MOOG_H_FORCES] + f;
    if (op->kind != MOOG_F_COLLISION) continue;
    int ca = pv.hdr[MOOG_H_LAYER_OFF + op->i[0] + 1] - pv.hdr[MOOG_H_LAYER_OFF + op->i[0]];
    int cb = pv.hdr[MOOG_H_LAYER_OFF + op->i[1] + 1] - pv.hdr[MOOG_H_LAYER_OFF + op->i[1]];
    words += ca * ((cb + 31) / 32);
  }
  return words;
}

struct Env {
  // shared memory
  double *dyn, *stat, *aabb, *tmp, *envf;
  float *aabb0, *nskin;
  double2 *vtx;
  int *meta, *sflag, *voff, *cnt, *envi, *cmoff;
  unsigned *cmask, *nearp;
  unsigned char *scratch;
  double *win_a;
  unsigned char *win_e;
  unsigned char *xchg;
  unsigned short *plist;
  int dcv_tile;
  unsigned long long *mbar;
  // program (global memory, read-only)
  const int32_t *hdr;
  const moog_op *ops;
  const int32_t *ipool;
  const moog_ex *expr;
  const uint8_t *vmap;       // program constant: cached vertex -> slot
  const double *dpool;       // shape records / reset-sampler parameters of the blob
  int S, L, K, VT, lane;
  const double *noise;       // [K][noise_dim] of this env or nullptr
  const double *rule_noise;  // [rule_noise_dim] of this env or nullptr
  uint64_t seed;
  int env_id;
  // Mutable per-env bookkeeping lives in shared memory (lane 0 updates it), so
  // that this struct is immutable after set-up and stays in registers: passed
  // by const reference through the inlined hot path and BY VALUE to the rare
  // out-of-line paths, its address never escapes.
  //   ctr[0..7] = counters (moog_step_io::counters), ctr[8] = current substep
  long long *ctr;
};

// The env's view record at the start of the CTA's shared memory: out-of-line
// device functions rebuild their `Env` from it (a few broadcast LDS) instead
// of receiving ~50 registers through the stack.
struct EnvRec {
  SmemLayout lay;
  int S, L, K, VT, env_id, pad;
  const moog_op *ops;
  const int32_t *ipool;
  const moog_ex *expr;
  const double *noise, *rule_noise;
  const uint16_t *vmap;      // (global memory; staged into shared memory as one byte per vertex)
  const double *dpool;
  uint64_t seed;
};
static_assert(sizeof(EnvRec) <= 224, "EnvRec must fit its shared-memory slot");

__device__ __forceinline__ Env env_view() {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned char *base = smem_raw;
  const EnvRec *r = (const EnvRec *)base;
  Env e;
  e.dyn = (double *)(base + r->lay.dyn);
  e.stat = (double *)(base + r->lay.stat);
  e.aabb = (double *)(base + r->lay.aabb);
  e.aabb0 = (float *)(base + r->lay.aabb0);
  e.nskin = (float *)(base + r->lay.nskin);
  e.tmp = (double *)(base + r->lay.tmp);
  e.vtx = (double2 *)(base + r->lay.vtx);
  e.envf = (double *)(base + r->lay.envf);
  e.ctr = (long long *)(base + r->lay.ctr);
  e.meta = (int *)(base + r->lay.meta);
  e.sflag = (int *)(base + r->lay.sflag);
  e.voff = (int *)(base + r->lay.voff);
  e.cnt = (int *)(base + r->lay.cnt);
  e.envi = (int *)(base + r->lay.envi);
  e.cmoff = (int *)(base + r->lay.cmoff);
  e.cmask = (unsigned *)(base + r->lay.cmask);
  e.nearp = (unsigned *)(base + r->lay.nearp);
  e.hdr = (const int32_t *)(base + r->lay.hdr);
  const int warp = threadIdx.x >> 5;
  e.scratch = base + r->lay.scratch + 64 * warp;
  e.win_a = (double *)(base + r->lay.win_a) + 32 * warp;
  e.win_e = base + r->lay.win_e + 32 * warp;
  e.xchg = base + r->lay.xchg;
  e.plist = (unsigned short *)(base + r->lay.plist) + 32 * r->lay.tile * warp;
  e.dcv_tile = r->lay.tile;
  e.mbar = (unsigned long long *)(base + r->lay.mbar);
  e.ops = r->ops; e.ipool = r->ipool; e.expr = r->expr;
  e.vmap = r->vmap ? (const uint8_t *)(base + r->lay.vmap) : nullptr;
  e.dpool = r->dpool;
  e.S = r->S; e.L = r->L; e.K = r->K; e.VT = r->VT;
  e.lane = threadIdx.x & 31;
  e.noise = r->noise; e.rule_noise = r->rule_noise;
  e.seed = r->seed;
  e.env_id = r->env_id;
  return e;
}

#if defined(MOOG_PROFILE_PHASES) || defined(MOOG_PROFILE_DCV) || defined(MOOG_PROFILE_GCV) || defined(MOOG_PROFILE_INTEG)
#define PROF_RESOLVE(e, t1)
#elif defined(MOOG_CYCLE_COUNTERS)
#define PROF_RESOLVE(e, t1) ctr_add(e, CT_CYC_RESOLVE, clock64() - (t1))
#else
#define PROF_RESOLVE(e, t1)
#endif

enum { CT_CALLS = 0, CT_TRUE, CT_COLL, CT_HASH, CT_CYCLES, CT_NARROW, CT_CYC_NARROW, CT_CYC_RESOLVE, CT_SUBSTEP,
       CT_NEAR /* near-list length; -1 overflowed, -2 not built yet */ };
__device__ __forceinline__ void ctr_add(const Env &e, int k, long long v) {
  if (e.lane == 0) e.ctr[k] += v;
}

#define DYN(e, f, s) ((e).dyn[(f) * (e).S + (s)])
#define STAT(e, f, s) ((e).stat[(f) * (e).S + (s)])
#define META(e, f, s) ((e).meta[(f) * (e).S + (s)])
// bounding box of slot s: [xmin, ymin, xmax + AABB_PAD, ymax + AABB_PAD], interleaved per slot.
// The maxima are stored padded so that the broad phase is four compares; the
// pad only has to be conservative (>> accumulated rounding), never exact.
#define BOX(e, f, s) ((e).aabb[4 * (s) + (f)])
#define TMP(e, f, s) ((e).tmp[(f) * (e).S + (s)])
#define LOFF(e, l) ((e).hdr[MOOG_H_LAYER_OFF + (l)])

__device__ __forceinline__ void wsync() { __syncwarp(); }
// scalar store by one lane; callers wsync() before anybody reads it back
__device__ __forceinline__ void put(const Env &e, double *p, double v) {
  if (e.lane == 0) *p = v;
}
__device__ __forceinline__ void puti(const Env &e, int *p, int v) {
  if (e.lane == 0) *p = v;
}

__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(FULL, v, src); }
__device__ __forceinline__ double shflx_d(double v, int m) { return __shfl_xor_sync(FULL, v, m); }

// ---------------------------------------------------------------------------
// counter-based RNG (Philox4x32-10) for RandomForce / sample_one when the
// caller supplies no noise tensor
// ---------------------------------------------------------------------------
__device__ inline double philox_uniform(uint64_t seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  uint64_t bits = ((uint64_t)c0 << 21) ^ (uint64_t)(c1 >> 11);  // 53 bits
  return (double)(bits & ((1ull << 53) - 1)) * (1.0 / 9007199254740992.0);
}

// ---------------------------------------------------------------------------
// numpy arithmetic conventions (see oracle/moog_oracle.c for the derivation)
// ---------------------------------------------------------------------------
__device__ __forceinline__ double norm_ax(double x, double y) { return sqrt(x * x + y * y); }
__device__ __forceinline__ double dot2(double ax, double ay, double bx, double by) { return fma(ay, by, ax * bx); }
__device__ __forceinline__ double norm1(double x, double y) { return sqrt(dot2(x, y, x, y)); }
// a / b where a is often exactly zero (DownGravity's x component): a zero numerator
// takes the fp64 division's slow path, so produce its signed-zero result directly
__device__ __forceinline__ double div_z(double a, double b) {
  if (a == 0.0 && b != 0.0 && isfinite(b)) return (signbit(a) != signbit(b)) ? -0.0 : 0.0;
  return a / b;
}
__device__ __forceinline__ double f32r(double x) { return (double)(float)x; }
__device__ __forceinline__ double f32mul(double a, double b) { return (double)__fmul_rn((float)a, (float)b); }
__device__ __forceinline__ double f32add(double a, double b) { return (double)__fadd_rn((float)a, (float)b); }
__device__ __forceinline__ double f32sub(double a, double b) { return (double)__fsub_rn((float)a, (float)b); }
__device__ __forceinline__ double f32div(double a, double b) { return (double)__fdiv_rn((float)a, (float)b); }

__device__ __forceinline__ bool vel32(const Env &e, int s) { return (META(e, MOOG_M_FLAGS, s) & MOOG_SF_VEL32) != 0; }
__device__ __forceinline__ int angvel_kind(const Env &e, int s) { return (META(e, MOOG_M_FLAGS, s) >> MOOG_SF_ANGVEL_SHIFT) & 3; }
__device__ __forceinline__ int ang_kind(const Env &e, int s) { return (META(e, MOOG_M_FLAGS, s) >> MOOG_SF_ANG_SHIFT) & 3; }
__device__ __forceinline__ void set_angvel_kind(const Env &e, int s, int k) {
  puti(e, &META(e, MOOG_M_FLAGS, s), (META(e, MOOG_M_FLAGS, s) & ~(3 << MOOG_SF_ANGVEL_SHIFT)) | (k << MOOG_SF_ANGVEL_SHIFT));
  wsync();
}

__device__ __forceinline__ int valias(const Env &e, int s) {
  return (META(e, MOOG_M_FLAGS, s) >> MOOG_SF_VALIAS_SHIFT) & MOOG_SF_VALIAS_MASK;
}
// `sprite.velocity += dv` (float64 dv; a float32 velocity array keeps its dtype).
// The ndarray may be shared with other sprites (MOOG_SF_VALIAS_SHIFT in
// moog_b200_program.h): the in-place add then shows in all of them.
__device__ inline void add_velocity(const Env &e, int s, double dvx, double dvy) {
  double vx = DYN(e, MOOG_D_VX, s) + dvx, vy = DYN(e, MOOG_D_VY, s) + dvy;
  if (vel32(e, s)) {
    vx = f32r(vx);
    vy = f32r(vy);
  }
  const int id = valias(e, s);
  wsync();
  if (id) {
    for (int t = e.lane; t < e.S; t += 32)
      if (valias(e, t) == id) {
        DYN(e, MOOG_D_VX, t) = vx;
        DYN(e, MOOG_D_VY, t) = vy;
      }
  } else {
    put(e, &DYN(e, MOOG_D_VX, s), vx);
    put(e, &DYN(e, MOOG_D_VY, s), vy);
  }
  wsync();
}
// `sprite.velocity = value` replaces the array by a new float64 one
__device__ inline void assign_velocity(const Env &e, int s, double vx, double vy) {
  int fl = META(e, MOOG_M_FLAGS, s) & ~(MOOG_SF_VEL32 | (MOOG_SF_VALIAS_MASK << MOOG_SF_VALIAS_SHIFT));
  wsync();
  put(e, &DYN(e, MOOG_D_VX, s), vx);
  put(e, &DYN(e, MOOG_D_VY, s), vy);
  puti(e, &META(e, MOOG_M_FLAGS, s), fl);
  wsync();
}
// a fresh alias id for an array object that several sprites are about to share
__device__ inline int new_valias(const Env &e) {
  int id = e.envi[MOOG_EI_VALIAS_NEXT] + 1;
  if (id > MOOG_SF_VALIAS_MASK || id < 1) id = 1;
  wsync();
  puti(e, &e.envi[MOOG_EI_VALIAS_NEXT], id);
  wsync();
  return id;
}
// `sprite.angle_vel += dw` with an np.float64 dw
__device__ inline void add_angvel(const Env &e, int s, double dw) {
  double w = DYN(e, MOOG_D_ANGVEL, s) + dw;
  int k = angvel_kind(e, s);
  wsync();
  if (k == KIND_F32)
    w = f32r(w);
  else
    set_angvel_kind(e, s, KIND_F64);
  put(e, &DYN(e, MOOG_D_ANGVEL, s), w);
  wsync();
}
__device__ __forceinline__ double scaled_vel(const Env &e, int s, int field, double c, double dt) {
  double v = DYN(e, field, s);
  return vel32(e, s) ? f32mul(f32mul(c, v), dt) : c * v * dt;
}
__device__ __forceinline__ double scaled_angvel(const Env &e, int s, double c, double dt) {
  double w = DYN(e, MOOG_D_ANGVEL, s);
  return angvel_kind(e, s) == KIND_F32 ? f32mul(f32mul(c, w), dt) : c * w * dt;
}
__device__ __forceinline__ bool is_symmetric_circle(const Env &e, int s) {
  return (META(e, MOOG_M_FLAGS, s) & MOOG_SF_CIRCLE) && STAT(e, MOOG_S_ASPECT, s) == 1.0;  // sprite.py:500-502
}
__device__ __forceinline__ double moment_of_inertia(const Env &e, int s) {
  double m = STAT(e, MOOG_S_MASS, s);  // sprite.py:662-664
  return 0.0 + m * STAT(e, MOOG_S_IX, s) + m * STAT(e, MOOG_S_IY, s);
}

// ---------------------------------------------------------------------------
// bounding boxes of the cached outlines
// ---------------------------------------------------------------------------

// A slot with a NaN / inf coordinate gets an all-covering box: it is never culled.
__device__ __forceinline__ void store_box(const Env &e, int s, double xmin, double ymin, double xmax, double ymax,
                                          bool nonfinite, bool steep = false) {
  BOX(e, 0, s) = nonfinite ? -INFINITY : xmin;
  BOX(e, 1, s) = (nonfinite || steep) ? -INFINITY : ymin;
  BOX(e, 2, s) = nonfinite ? INFINITY : xmax + AABB_PAD;
  BOX(e, 3, s) = (nonfinite || steep) ? INFINITY : ymax + AABB_PAD;
}
__device__ __forceinline__ bool steep_edge(double x0, double x1) {
  const double dx = x1 - x0;
  return dx != 0.0 && fabs(dx) <= STEEP_DX;
}

// lane-parallel over the vertices of slot s: NaN / inf classification (called
// when a setter moved the outline by a non-finite amount)
__device__ inline void classify_slot(const Env &e, int s) {
  int n = META(e, MOOG_M_NV, s);
  const double2 *v = e.vtx + e.voff[s];
  bool nonfinite = false, nan2 = true;
  for (int i = e.lane; i < n; i += 32) {
    const double2 p = v[i];
    nonfinite |= !(isfinite(p.x) && isfinite(p.y));
    nan2 &= isnan(p.x) && isnan(p.y);
  }
  unsigned nf = __ballot_sync(FULL, nonfinite);
  bool allnan = __all_sync(FULL, nan2) && n > 0;
  int fl = (e.sflag[s] & ~(SLF_NONFINITE | SLF_ALLNAN)) | (nf ? SLF_NONFINITE : 0) | (allnan ? SLF_ALLNAN : 0);
  wsync();
  puti(e, &e.sflag[s], fl);
  if (nf && e.lane == 0) store_box(e, s, 0., 0., 0., 0., true);
  wsync();
}

// lane = slot: every lane scans its own outline (used at load time)
__device__ inline void refresh_all_boxes(const Env &e) {
  for (int s = e.lane; s < e.S; s += 32) {
    int n = META(e, MOOG_M_NV, s);
    const double2 *v = e.vtx + e.voff[s];
    double xmin = INFINITY, xmax = -INFINITY, ymin = INFINITY, ymax = -INFINITY;
    bool sh = n < 3, nonfinite = false, allnan = n > 0, steep = false;
    double2 prev = n > 0 ? v[n - 1] : make_double2(0., 0.);
    for (int i = 0; i < n; ++i) {
      double2 p = v[i];
      xmin = fmin(xmin, p.x); xmax = fmax(xmax, p.x);
      ymin = fmin(ymin, p.y); ymax = fmax(ymax, p.y);
      double len2 = (p.x - prev.x) * (p.x - prev.x) + (p.y - prev.y) * (p.y - prev.y);
      sh |= !(len2 > SHORT_EDGE2);
      steep |= steep_edge(prev.x, p.x);
      nonfinite |= !(isfinite(p.x) && isfinite(p.y));
      allnan &= isnan(p.x) && isnan(p.y);
      prev = p;
    }
    store_box(e, s, xmin, ymin, xmax, ymax, nonfinite, steep);
    e.sflag[s] = (sh ? SLF_SHORT_EDGE : 0) | (nonfinite ? SLF_NONFINITE : 0) | (allnan ? SLF_ALLNAN : 0) |
                 (steep ? SLF_STEEP : 0);
  }
  wsync();
}

__device__ __forceinline__ bool boxes_apart(const Env &e, int a, int b) {
  return BOX(e, 2, a) < BOX(e, 0, b) || BOX(e, 2, b) < BOX(e, 0, a) ||
         BOX(e, 3, a) < BOX(e, 1, b) || BOX(e, 3, b) < BOX(e, 1, a);
}

// ---------------------------------------------------------------------------
// position / angle setters (sprite.py:531-540, 616-633): the cached outline is
// transformed incrementally, exactly like the reference's Sprite._path
// ---------------------------------------------------------------------------
// Vertices 32 .. n-1 of a big draw-only outline (MOOG_MAX_OUTLINE): the translation (and
// rotation) the callers apply to the first 32 themselves.  Out of line: the hot paths only
// pay a never-taken branch for it.
__device__ __noinline__ void outline_tail(double2 *v, int n, int lane, double tx, double ty, bool rotates, double r0,
                                          double r1, double r2, double r3, double r4, double r5) {
#pragma unroll 1
  for (int i = lane + 32; i < n; i += 32) {
    const double2 p = v[i];
    double x = (1.0 * p.x + 0.0 * p.y) + tx;
    double y = (0.0 * p.x + 1.0 * p.y) + ty;
    if (rotates) {
      const double rx = r0 * x + r1 * y + r2;
      const double ry = r3 * x + r4 * y + r5;
      x = rx;
      y = ry;
    }
    v[i] = make_double2(x, y);
  }
}

__device__ __forceinline__ void set_position_impl(const Env &e, int s, double nx, double ny) {
  double tx = nx - DYN(e, MOOG_D_X, s), ty = ny - DYN(e, MOOG_D_Y, s);
  int n = META(e, MOOG_M_NV, s);
  double2 *v = e.vtx + e.voff[s];
  double b0 = BOX(e, 0, s), b1 = BOX(e, 1, s), b2 = BOX(e, 2, s), b3 = BOX(e, 3, s);
  wsync();
  if (e.lane < n) {
    double2 p = v[e.lane];
    double x = 1.0 * p.x + 0.0 * p.y + tx;
    double y = 0.0 * p.x + 1.0 * p.y + ty;
    v[e.lane] = make_double2(x, y);
  }
  if (n > 32) outline_tail(v, n, e.lane, tx, ty, false, 1., 0., 0., 0., 1., 0.);
  if (e.lane == 0) {
    DYN(e, MOOG_D_X, s) = nx;
    DYN(e, MOOG_D_Y, s) = ny;
    // x -> fl(x + tx) is monotone, so the translated minima are exactly the minima of the
    // translated vertices; the padded maxima stay conservative
    BOX(e, 0, s) = b0 + tx; BOX(e, 1, s) = b1 + ty; BOX(e, 2, s) = b2 + tx; BOX(e, 3, s) = b3 + ty;
  }
  wsync();
  if (!(isfinite(tx) && isfinite(ty))) classify_slot(e, s);
}

__device__ __noinline__ void set_position_ol(int s, double nx, double ny) {
  const Env e = env_view();
  set_position_impl(e, s, nx, ny);
}
__device__ __forceinline__ void set_position(const Env &, int s, double nx, double ny) { set_position_ol(s, nx, ny); }

struct Aff { double m0, m1, m2, m3, m4, m5; };  // rows 0,1 of the 3x3 (row 2 = 0 0 1)

__device__ __forceinline__ Aff aff_identity() { Aff a = {1., 0., 0., 0., 1., 0.}; return a; }
__device__ __forceinline__ void aff_translate(Aff &m, double tx, double ty) { m.m2 += tx; m.m5 += ty; }
__device__ __noinline__ double2 cos_sin_ol(double theta) { return make_double2(cos(theta), sin(theta)); }

__device__ inline void aff_rotate(Aff &m, double theta) {
  // cos(+-0) == 1 and sin(+-0) == +-0 exactly: skip the libm call for sprites that do not rotate
  double a = 1.0, b = theta;
  if (theta != 0.0) {
    double2 cs = cos_sin_ol(theta);
    a = cs.x;
    b = cs.y;
  }
  double xx = m.m0, xy = m.m1, x0 = m.m2, yx = m.m3, yy = m.m4, y0 = m.m5;
  m.m0 = a * xx - b * yx; m.m1 = a * xy - b * yy; m.m2 = a * x0 - b * y0;
  m.m3 = b * xx + a * yx; m.m4 = b * xy + a * yy; m.m5 = b * x0 + a * y0;
}
__device__ inline void aff_rotate_around(Aff &m, double x, double y, double theta) {
  aff_translate(m, -x, -y);
  aff_rotate(m, theta);
  aff_translate(m, x, y);
}
// out = b . a ("a, then b"); numpy 3x3 matmul fuses: fma(b2,a2, fma(b1,a1, b0*a0)).
// Row 2 of both is (0,0,1) exactly, so the third term of columns 0,1 is fma(b2, 0, .) = exact.
__device__ inline Aff aff_then(const Aff &a, const Aff &b) {
  Aff o;
  o.m0 = fma(b.m2, 0.0, fma(b.m1, a.m3, b.m0 * a.m0));
  o.m1 = fma(b.m2, 0.0, fma(b.m1, a.m4, b.m0 * a.m1));
  o.m2 = fma(b.m2, 1.0, fma(b.m1, a.m5, b.m0 * a.m2));
  o.m3 = fma(b.m5, 0.0, fma(b.m4, a.m3, b.m3 * a.m0));
  o.m4 = fma(b.m5, 0.0, fma(b.m4, a.m4, b.m3 * a.m1));
  o.m5 = fma(b.m5, 1.0, fma(b.m4, a.m5, b.m3 * a.m2));
  return o;
}

// ---------------------------------------------------------------------------
// matplotlib src/_path.h restatement (lane-parallel)
// ---------------------------------------------------------------------------
__device__ __forceinline__ bool isclose_(double a, double b) {
  return fabs(a - b) <= fmax(1e-10 * fmax(fabs(a), fabs(b)), 1e-13);
}

// the parallel case of segments_intersect (rare: kept out of the callers' instruction stream)
__device__ __noinline__ bool segments_parallel_case(double x1, double y1, double x2, double y2, double x3, double y3,
                                                    double x4, double y4) {
  double t_area = (x2 * y3 - x3 * y2) - x1 * (y3 - y2) + y1 * (x3 - x2);
  if (isclose_(t_area, 0.0)) {
    if (x1 == x2 && x2 == x3) {
      return (fmin(y1, y2) <= fmin(y3, y4) && fmin(y3, y4) <= fmax(y1, y2)) ||
             (fmin(y3, y4) <= fmin(y1, y2) && fmin(y1, y2) <= fmax(y3, y4));
    }
    return (fmin(x1, x2) <= fmin(x3, x4) && fmin(x3, x4) <= fmax(x1, x2)) ||
           (fmin(x3, x4) <= fmin(x1, x2) && fmin(x1, x2) <= fmax(x3, x4));
  }
  return false;
}

// (fmin(a, b), fmax(a, b)) for finite a, b: one compare and selects instead of fmin / fmax's NaN handling
__device__ __forceinline__ void minmax_finite(double a, double b, double &lo, double &hi) {
  const bool s = a < b;
  lo = s ? a : b;
  hi = s ? b : a;
}

// the range tests of segments_intersect by division, for the operands seg_param_in_unit leaves
// undecided (rare: kept out of the callers' instruction stream)
__device__ __noinline__ bool segments_params_divide(double n1, double n2, double den) {
  double u1 = n1 / den;
  double u2 = n2 / den;
  return ((u1 > 0.0 || isclose_(u1, 0.0)) && (u1 < 1.0 || isclose_(u1, 1.0)) &&
          (u2 > 0.0 || isclose_(u2, 0.0)) && (u2 < 1.0 || isclose_(u2, 1.0)));
}

// src/_path.h segments_intersect, called by every lane of the warp together; a lane with `act`
// false returns false.  The range tests on u1 = n1 / den and u2 = n2 / den are decided without
// dividing (moog_seg_cross.cuh); when some lane's operands are outside that decision's regime,
// those lanes divide, behind a warp-uniform branch.
__device__ __forceinline__ bool segments_intersect(bool act, double x1, double y1, double x2, double y2, double x3,
                                                   double y3, double x4, double y4) {
  const double den = ((y4 - y3) * (x2 - x1)) - ((x4 - x3) * (y2 - y1));
  const double n1 = ((x4 - x3) * (y1 - y3)) - ((y4 - y3) * (x1 - x3));
  const double n2 = ((x2 - x1) * (y1 - y3)) - ((y2 - y1) * (x1 - x3));
  const bool par = isclose_(den, 0.0);
  bool e1, e2;
  bool r = seg_param_in_unit(n1, den, e1) & seg_param_in_unit(n2, den, e2);
  const bool divide = act && !par && !(e1 && e2);
  if (__any_sync(FULL, divide)) {
    if (divide) r = segments_params_divide(n1, n2, den);
  }
  if (act && par) r = segments_parallel_case(x1, y1, x2, y2, x3, y3, x4, y4);
  return act && r;
}

// point_in_path_impl for one point against the closed outline Q[0..n-1]
// (the reference passes the V+1 closed path; its extra closing edge has zero
// length and never toggles).  All lanes walk the edges together.
__device__ inline bool point_in_poly(double tx, double ty, const double2 *Q, int n) {
  if (n < 2) return false;  // nv = n + 1 < 3
  bool finite = isfinite(tx) && isfinite(ty);
  int inside = 0;
  double2 p0 = Q[0];
  for (int k = 0; k < n; ++k) {
    double2 p1 = Q[(k + 1 == n) ? 0 : k + 1];
    bool f0 = p0.y >= ty, f1 = p1.y >= ty;
    if (f0 != f1) {
      if ((((p1.y - ty) * (p0.x - p1.x)) >= ((p1.x - tx) * (p0.y - p1.y))) == f1) inside ^= 1;
    }
    p0 = p1;
  }
  return finite && inside;
}

// serial restatement of path_intersects_path for outlines with degenerate
// (nearly zero-length) edges, where matplotlib merges consecutive points.
// All lanes run it redundantly (together); it is never on the hot path.
__device__ __noinline__ bool path_intersects_path_serial(const double2 *A, int nA, const double2 *B, int nB) {
  int na = nA + 1, nb = nB + 1;
  if (na < 2 || nb < 2) return false;
  double x11 = A[0].x, y11 = A[0].y;
  for (int i = 1; i < na; ++i) {
    double2 pa = A[i == nA ? 0 : i];
    double x12 = pa.x, y12 = pa.y;
    if (isclose_((x11 - x12) * (x11 - x12) + (y11 - y12) * (y11 - y12), 0.0)) continue;
    double x21 = B[0].x, y21 = B[0].y;
    for (int j = 1; j < nb; ++j) {
      double2 pb = B[j == nB ? 0 : j];
      double x22 = pb.x, y22 = pb.y;
      if (isclose_((x21 - x22) * (x21 - x22) + (y21 - y22) * (y21 - y22), 0.0)) continue;
      if (segments_intersect(true, x11, y11, x12, y12, x21, y21, x22, y22)) return true;
      x21 = x22;
      y21 = y22;
    }
    x11 = x12;
    y11 = y12;
  }
  return false;
}

// all vertices of P (np of them, + the duplicated closing one) inside Q?
__device__ inline bool all_points_in_poly(const Env &e, const double2 *P, int np_, const double2 *Q, int nq) {
  if (nq + 1 < 3) return false;
  bool act = e.lane < np_;
  double2 p = P[act ? e.lane : 0];
  bool in = point_in_poly(p.x, p.y, Q, nq);
  return __all_sync(FULL, in || !act);
}

// the path_in_path fall-backs of path_intersects_filled (boxes nest: rare)
__device__ __noinline__ bool containment_fallback(int a, int b, bool try_b_in_a, bool try_a_in_b) {
  const Env e = env_view();
  const double2 *A = e.vtx + e.voff[a];
  const double2 *B = e.vtx + e.voff[b];
  const int nA = META(e, MOOG_M_NV, a), nB = META(e, MOOG_M_NV, b);
  if (try_b_in_a && all_points_in_poly(e, B, nB, A, nA)) return true;  // b inside a
  if (try_a_in_b && all_points_in_poly(e, A, nA, B, nB)) return true;  // a inside b
  return false;
}

// floor(2^16 / n) + 1 for n = 1..32: (t * PAIR_DIV_MAGIC[n]) >> 16 == t / n for t < 2^16 / n, which
// covers the pair indices t < 32 n of path_intersects_filled_impl (with 2^16 + k = n PAIR_DIV_MAGIC[n],
// 0 < k <= n: t / n + t k / (n 2^16) < floor(t / n) + (n - 1) / n + t / 2^16)
__constant__ unsigned PAIR_DIV_MAGIC[33] = {
    0,    65537, 32769, 21846, 16385, 13108, 10923, 9363, 8193, 7282, 6554, 5958, 5462, 5042, 4682, 4370, 4097,
    3856, 3641,  3450,  3277,  3121,  2979,  2850,  2731, 2622, 2521, 2428, 2341, 2260, 2185, 2115, 2049};

// Path.intersects_path(a, b, filled=True) as MOOG calls it (sprite.py:482-483)
__device__ __forceinline__ bool path_intersects_filled_impl(const Env &e, int a, int b) {
  const double2 *A = e.vtx + e.voff[a];
  const double2 *B = e.vtx + e.voff[b];
  int nA = META(e, MOOG_M_NV, a), nB = META(e, MOOG_M_NV, b);
  const int fl = e.sflag[a] | e.sflag[b];
  // an outline whose every coordinate is NaN intersects nothing and contains /
  // is contained in nothing: every segment test has a NaN denominator, every
  // crossing-number comparison is false
  if (fl & SLF_ALLNAN) return false;
  const bool nocull = (fl & (SLF_NONFINITE | SLF_STEEP)) != 0;  // boxes are meaningless with NaN / inf around
  bool serial = (fl & (SLF_SHORT_EDGE | SLF_NONFINITE | SLF_STEEP)) != 0;
  if (serial) {
    if (path_intersects_path_serial(A, nA, B, nB)) return true;
  } else {
    // Lanes first own the edges of each outline to find the few that can matter:
    // edges of P whose (padded) box meets Q's box and edges of Q whose box meets
    // P's padded box.  The surviving (P edge, Q edge) pairs -- a handful for two
    // touching outlines -- are then tested all at once, one pair per lane.
    // Argument order of segments_intersect is kept.  Every coordinate here is finite (SLF_NONFINITE
    // takes the serial path), so fmin / fmax reduce to a compare and selects, and a bound on
    // fmax(u, v) (fmin) to the same bound on both u and v.
    bool lanesA = nA >= nB;
    const double2 *P = lanesA ? A : B;
    const double2 *Q = lanesA ? B : A;
    int nP = lanesA ? nA : nB, nQ = lanesA ? nB : nA;
    int pslot = lanesA ? a : b, qslot = lanesA ? b : a;
    bool act = e.lane < nP;
    double2 p1 = P[act ? e.lane : 0];
    double2 p2 = P[act ? ((e.lane + 1 == nP) ? 0 : e.lane + 1) : 0];
    double pxmin, pxmax, pymin, pymax;
    minmax_finite(p1.x, p2.x, pxmin, pxmax);
    minmax_finite(p1.y, p2.y, pymin, pymax);
    act = act && !(pxmax + AABB_PAD < BOX(e, 0, qslot) || pxmin - AABB_PAD > BOX(e, 2, qslot) ||
                   pymax + AABB_PAD < BOX(e, 1, qslot) || pymin - AABB_PAD > BOX(e, 3, qslot));
    bool qact = e.lane < nQ;
    {
      double2 q1 = Q[qact ? e.lane : 0];
      double2 q2 = Q[qact ? ((e.lane + 1 == nQ) ? 0 : e.lane + 1) : 0];
      double Pxmin = BOX(e, 0, pslot) - AABB_PAD, Pymin = BOX(e, 1, pslot) - AABB_PAD;
      double Pxmax = BOX(e, 2, pslot), Pymax = BOX(e, 3, pslot);
      qact = qact && !((q1.x < Pxmin && q2.x < Pxmin) || (q1.x > Pxmax && q2.x > Pxmax) ||
                       (q1.y < Pymin && q2.y < Pymin) || (q1.y > Pymax && q2.y > Pymax));
    }
    const unsigned pm = __ballot_sync(FULL, act), qm = __ballot_sync(FULL, qact);
    if (pm && qm) {
      const unsigned lt = (1u << e.lane) - 1u;
      const int np_ = __popc(pm), nq_ = __popc(qm);
      wsync();
      if (act) e.scratch[__popc(pm & lt)] = (unsigned char)e.lane;
      if (qact) e.scratch[32 + __popc(qm & lt)] = (unsigned char)e.lane;
      wsync();
      const int total = np_ * nq_;
      const unsigned qmagic = PAIR_DIV_MAGIC[nq_];
      for (int base = 0; base < total; base += 32) {
        int t = base + e.lane;
        bool v = t < total;
        int pi = v ? (int)(((unsigned)t * qmagic) >> 16) : 0;  // t / nq_
        int qi = v ? t - pi * nq_ : 0;
        int pl = e.scratch[pi], ql = e.scratch[32 + qi];
        double2 a1 = P[pl], a2 = P[(pl + 1 == nP) ? 0 : pl + 1];
        double2 b1 = Q[ql], b2 = Q[(ql + 1 == nQ) ? 0 : ql + 1];
        double axmin, axmax, aymin, aymax;
        minmax_finite(a1.x, a2.x, axmin, axmax);
        minmax_finite(a1.y, a2.y, aymin, aymax);
        axmin -= AABB_PAD, axmax += AABB_PAD, aymin -= AABB_PAD, aymax += AABB_PAD;
        const bool test = v && !((b1.x < axmin && b2.x < axmin) || (b1.x > axmax && b2.x > axmax) ||
                                 (b1.y < aymin && b2.y < aymin) || (b1.y > aymax && b2.y > aymax));
        const double2 f1 = lanesA ? a1 : b1, f2 = lanesA ? a2 : b2;
        const double2 g1 = lanesA ? b1 : a1, g2 = lanesA ? b2 : a2;
        const bool h = segments_intersect(test, f1.x, f1.y, f2.x, f2.y, g1.x, g1.y, g2.x, g2.y);
        if (__any_sync(FULL, h)) return true;
      }
    }
  }
  // containment fall-backs: a point outside the (padded) box of an outline is
  // outside the outline, so "all inside" needs box containment first
  bool b_in_a_box = BOX(e, 0, b) >= BOX(e, 0, a) - AABB_PAD && BOX(e, 2, b) <= BOX(e, 2, a) + AABB_PAD &&
                    BOX(e, 1, b) >= BOX(e, 1, a) - AABB_PAD && BOX(e, 3, b) <= BOX(e, 3, a) + AABB_PAD;
  bool a_in_b_box = BOX(e, 0, a) >= BOX(e, 0, b) - AABB_PAD && BOX(e, 2, a) <= BOX(e, 2, b) + AABB_PAD &&
                    BOX(e, 1, a) >= BOX(e, 1, b) - AABB_PAD && BOX(e, 3, a) <= BOX(e, 3, b) + AABB_PAD;
  if (b_in_a_box || a_in_b_box || nocull) return containment_fallback(a, b, b_in_a_box || nocull, a_in_b_box || nocull);
  return false;
}

__device__ __noinline__ bool path_intersects_filled_ol(int a, int b) {
  const Env e = env_view();
  return path_intersects_filled_impl(e, a, b);
}
__device__ __forceinline__ bool path_intersects_filled(const Env &, int a, int b) { return path_intersects_filled_ol(a, b); }

__device__ __forceinline__ void count_overlap(const Env &e, int a, int b, bool r) {
  if (e.lane == 0) {
    e.ctr[CT_CALLS]++;
    if (r) {
      e.ctr[CT_TRUE]++;
      unsigned long long h = (unsigned long long)e.ctr[CT_HASH];
      h = (h ^ (uint64_t)(((uint32_t)a * 1315423911u) ^ ((uint32_t)b * 2654435761u) ^ 1u)) * 1099511628211ull;
      e.ctr[CT_HASH] = (long long)h;
    }
  }
}

// sprite.py:462-484 Sprite.overlaps_sprite
__device__ inline bool overlaps(const Env &e, int a, int b) {
  bool r = false;
  double dx = DYN(e, MOOG_D_X, a) - DYN(e, MOOG_D_X, b);
  double dy = DYN(e, MOOG_D_Y, a) - DYN(e, MOOG_D_Y, b);
  double center_dist = norm1(dx, dy);
  if (!(center_dist > STAT(e, MOOG_S_MAXR, a) + STAT(e, MOOG_S_MAXR, b))) {
    if (((e.sflag[a] | e.sflag[b]) & SLF_NONFINITE) || !boxes_apart(e, a, b)) r = path_intersects_filled(e, a, b);
  }
  count_overlap(e, a, b, r);
  return r;
}

// ---------------------------------------------------------------------------
// collisions.py
// ---------------------------------------------------------------------------
enum { HELPER_EXIT = 0, HELPER_DCV = 1 };
// named barrier over the owner and helper warps of the CTA (also orders their shared-memory traffic)
// (the warp reconverges first: `bar.sync` is the .aligned form, which every lane of a warp must execute together --
// compute-sanitizer synccheck flagged lanes still apart after an `if (lane == 0)` store in front of it)
__device__ __forceinline__ void cta_bar(int id) {
  __syncwarp();
  asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory");
}

struct CVec {
  int has_point, future, has_since;
  double px, py, nx, ny, sx, sy, qx, qy;  // point, normal, since, perp
};

// the four-transform product of _relative_motion_trajectory when a sprite rotates
__device__ __noinline__ Aff rel_motion_general(double x1, double y1, double th1, double tx2, double ty2, double x3,
                                               double y3, double th3, double tx4, double ty4) {
  Aff m1 = aff_identity(), m2 = aff_identity(), m3 = aff_identity(), m4 = aff_identity();
  aff_rotate_around(m1, x1, y1, th1);
  aff_translate(m2, tx2, ty2);
  aff_rotate_around(m3, x3, y3, th3);
  aff_translate(m4, tx4, ty4);
  Aff t12 = aff_then(m1, m2);
  Aff t123 = aff_then(t12, m3);
  return aff_then(t123, m4);
}

// collisions.py:62-98 _relative_motion_trajectory (matrix only)
__device__ inline Aff rel_motion_matrix(const Env &e, int ps, int as, double dt) {
  const double th1 = scaled_angvel(e, ps, -1.0, dt);
  const double tx2 = scaled_vel(e, ps, MOOG_D_VX, -1.0, dt), ty2 = scaled_vel(e, ps, MOOG_D_VY, -1.0, dt);
  const double th3 = angvel_kind(e, as) == KIND_F32 ? f32mul(DYN(e, MOOG_D_ANGVEL, as), dt)
                                                    : DYN(e, MOOG_D_ANGVEL, as) * dt;
  const double tx4 = vel32(e, as) ? f32mul(DYN(e, MOOG_D_VX, as), dt) : DYN(e, MOOG_D_VX, as) * dt;
  const double ty4 = vel32(e, as) ? f32mul(DYN(e, MOOG_D_VY, as), dt) : DYN(e, MOOG_D_VY, as) * dt;
  const double x1 = DYN(e, MOOG_D_X, ps), y1 = DYN(e, MOOG_D_Y, ps);
  const double x3 = DYN(e, MOOG_D_X, as), y3 = DYN(e, MOOG_D_Y, as);
  if (th1 == 0.0 && th3 == 0.0 && isfinite(x1) && isfinite(y1) && isfinite(x3) && isfinite(y3) && isfinite(tx2) &&
      isfinite(ty2) && isfinite(tx4) && isfinite(ty4)) {
    // Neither sprite rotates: rotate_around(x, y, +-0) is exactly the identity for finite
    // (x, y), and the general product below collapses to one rounded sum per
    // translation component (the + 0.0 is the product's -0 -> +0 normalisation).
    Aff m = {1., 0., tx4 + (tx2 + 0.0), 0., 1., ty4 + (ty2 + 0.0)};
    return m;
  }
  return rel_motion_general(x1, y1, th1, tx2, ty2, x3, y3, th3, tx4, ty4);
}
template <int TILE>
__device__ __forceinline__ void directed_collision_vectors_impl(const Env &e, int s0, int s1, double dt, CVec &o) {
  o.has_point = o.future = o.has_since = 0;
  o.px = o.py = o.nx = o.ny = o.sx = o.sy = o.qx = o.qy = 0.0;
#ifdef MOOG_PROFILE_DCV
  long long tp0 = clock64();
#endif
  const double2 *P0 = e.vtx + e.voff[s0];
  const double2 *P1 = e.vtx + e.voff[s1];
  int n0 = META(e, MOOG_M_NV, s0), n1 = META(e, MOOG_M_NV, s1);
  // sprite.py:442-460 contains_points: lane = vertex of s0
  bool act = e.lane < n0;
  double2 myv = P0[act ? e.lane : 0];
  bool inside;
  if (is_symmetric_circle(e, s1)) {
    inside = norm_ax(myv.x - DYN(e, MOOG_D_X, s1), myv.y - DYN(e, MOOG_D_Y, s1)) <= STAT(e, MOOG_S_MAXR, s1);
  } else {
    inside = point_in_poly(myv.x, myv.y, P1, n1);
  }
  unsigned mask = __ballot_sync(FULL, inside && act);
  if (mask == 0) return;  // (None, None, None, None)

  Aff M = rel_motion_matrix(e, s0, s1, dt);

  // Lanes are tiled as (vertices per pass) x (edges of s1): an outline with few
  // edges -- a wall -- takes several contained vertices per pass.
  const int E = n1 <= 4 ? 4 : (n1 <= 8 ? 8 : (n1 <= 16 ? 16 : 32));
  const int V = 32 / E;
  const int ej = e.lane & (E - 1), tl = e.lane / E;
  bool eact = ej < n1;
  double2 q1 = P1[eact ? ej : 0];
  double2 q2 = P1[eact ? ((ej + 1 == n1) ? 0 : ej + 1) : 0];
  double d1x = q2.x - q1.x, d1y = q2.y - q1.y;

  // Stage A1 (lane = (vertex, edge of s1); no cross-lane traffic but the compaction, so
  // consecutive trips overlap in the pipeline): the crossing pairs go to a list.
  // Stage A2 (lane = crossing pair): cross_a and its np.argmin key, in registers.
  // Stage B: np.argmin per vertex (first edge on ties) by a segmented scan over the pair lanes;
  // lane = vertex gets the winning edge and its cross_a from A2, and the penetration length.
  // Stage C: np.argmax over the vertices by two warp maxima.
  bool my_cross = false;
  bool have = false;
  double b_dist = 0, b_cpx = 0, b_cpy = 0, b_dfx = 0, b_dfy = 0, b_a = 0;
  int b_edge = 0;
  // contained vertex indices, ascending, in the scratch bytes
  const int n_in = __popc(mask);
  wsync();
  if ((mask >> e.lane) & 1u) e.scratch[__popc(mask & ((1u << e.lane) - 1u))] = (unsigned char)e.lane;
  wsync();
#ifdef MOOG_PROFILE_DCV
  ctr_add(e, CT_NARROW, clock64() - tp0);
  ctr_add(e, CT_COLL, n_in);
#endif
  for (int vbase = 0; vbase < (TILE >= MAXV ? 1 : n_in); vbase += TILE) {  // TILE >= MAXV: one pass covers any outline
    const int cnt = min(TILE, n_in - vbase);
#ifdef MOOG_PROFILE_DCV
    long long tp1 = clock64();
    long long tb = 0;
#endif
    // Stage A1 (no division): which (vertex, edge) pairs cross, i.e. 0 <= cross_b <= 1
    // (sprite.py:171-175).  A line meets a convex outline in two edges, so only a couple
    // of pairs per vertex do; they are compacted into a list in ascending (vertex, edge)
    // order (ballots in lane order, later trips hold later vertices), so the pairs of one
    // vertex are one contiguous segment of it.  Every other pair's key is |1 - (-inf)| = +inf.
    // Two passes per iteration for instruction-level parallelism.
    const unsigned lt = (1u << e.lane) - 1u;
    int n_pairs = 0;
    for (int t0 = 0; t0 < cnt; t0 += DCV_U * V) {
      bool cr[DCV_U], inexact = false;
      double nB2[DCV_U], den2[DCV_U];
      bool on2[DCV_U];
#pragma unroll
      for (int u = 0; u < DCV_U; ++u) {
        const int t = t0 + u * V + tl;
        const bool valid = t < cnt;
        const bool on = eact && valid;
        const int c = e.scratch[vbase + (valid ? t : cnt - 1)];
        const double2 ev = P0[c];  // traj[:,1]
        const double ex = ev.x, ey = ev.y;
        const double sx = M.m0 * ex + M.m1 * ey + M.m2;  // traj[:,0]
        const double sy = M.m3 * ex + M.m4 * ey + M.m5;
        const double d0x = ex - sx, d0y = ey - sy;
        // sprite.py:145-161 segment_crossing_coefficients against edge `ej`
        const double den = on ? (d0x * d1y - d0y * d1x) + EPS_INTERP : 1.0;
        const double qx = q1.x - sx, qy = q1.y - sy;
        const double nB = on ? (qx * d0y - qy * d0x) : 1.0;
        bool exact;
        const bool in_unit = unit_ratio(nB, den, exact);
        inexact |= !exact;
        cr[u] = on && in_unit;
        nB2[u] = nB; den2[u] = den; on2[u] = on;
      }
      if (__any_sync(FULL, inexact)) {  // out-of-range operands somewhere in the warp: divide
#pragma unroll
        for (int u = 0; u < DCV_U; ++u) {
          const double Bc = nB2[u] / den2[u];
          cr[u] = on2[u] && (Bc >= 0) && (Bc <= 1);
        }
      }
#pragma unroll
      for (int u = 0; u < DCV_U; ++u) {
        const unsigned cm = __ballot_sync(FULL, cr[u]);
        if (cr[u]) e.plist[n_pairs + __popc(cm & lt)] = (unsigned short)(((t0 + u * V + tl) << 8) | ej);
        n_pairs += __popc(cm);
      }
    }
    my_cross |= n_pairs > 0;
    // a vertex without a crossing pair: np.argmin of an all-inf row is edge 0, whose cross_a is -inf
    if (e.lane < cnt) { e.win_a[e.lane] = -INFINITY; e.win_e[e.lane] = 0; }
    wsync();
    // Stages A2 + B, 32 pairs per pass.  A pass ends after 32 pairs wherever that is, so the
    // running winner of its last vertex is carried into the next pass, where that vertex's
    // segment may go on.
    DcvCarry carry;
    for (int base = 0; base < n_pairs; base += 32) {
      // Stage A2: cross_a of the crossing pairs -- the same IEEE operations on the same operands
      // as above and as the reference, hence the same bits
      const int k = base + e.lane;
      const bool act2 = k < n_pairs;
      const unsigned ent = e.plist[act2 ? k : 0];
      const int t = (int)(ent >> 8), ed = (int)(ent & 255u);
      const double2 ev = P0[e.scratch[vbase + t]];
      const double ex = ev.x, ey = ev.y;
      const double sx = M.m0 * ex + M.m1 * ey + M.m2;
      const double sy = M.m3 * ex + M.m4 * ey + M.m5;
      const double d0x = ex - sx, d0y = ey - sy;
      const double2 w1 = P1[ed], w2 = P1[(ed + 1 == n1) ? 0 : ed + 1];
      const double e1x = w2.x - w1.x, e1y = w2.y - w1.y;
      const double den = act2 ? (d0x * e1y - d0y * e1x) + EPS_INTERP : 1.0;
      const double qx = w1.x - sx, qy = w1.y - sy;
#ifdef MOOG_PROFILE_DCV
      const double A = shfl_d((act2 ? (qx * e1y - qy * e1x) : 1.0) / den, e.lane);  // waits for A2: the clock splits A2 from B
      const long long tb0 = clock64();
#else
      const double A = (act2 ? (qx * e1y - qy * e1x) : 1.0) / den;
#endif
      // Stage B (moog_dcv_argmin.cuh)
      const int t_after = base + 32 < n_pairs ? (int)(e.plist[base + 32] >> 8) : 255;  // first vertex of the next pass
      int w_ed;
      double w_a;
      if (dcv_argmin_pass(act2, t, ed, A, t_after, e.lane, carry, w_ed, w_a)) {
        e.win_a[t] = w_a;
        e.win_e[t] = (unsigned char)w_ed;
      }
#ifdef MOOG_PROFILE_DCV
      tb += clock64() - tb0;
#endif
    }
    wsync();
#ifdef MOOG_PROFILE_DCV
    long long tp2 = clock64();
    ctr_add(e, CT_CYC_NARROW, tp2 - tp1 - tb);
#endif
    const bool vact = e.lane < cnt;
    const int idx = e.win_e[vact ? e.lane : 0];
    double A = e.win_a[vact ? e.lane : 0], cpx = 0, cpy = 0, dfx = 0, dfy = 0, dist = 0;
    {
      const double2 ev = P0[e.scratch[vbase + (vact ? e.lane : 0)]];
      const double ex = ev.x, ey = ev.y;
      const double sx = M.m0 * ex + M.m1 * ey + M.m2;
      const double sy = M.m3 * ex + M.m4 * ey + M.m5;
      cpx = sx + A * (ex - sx);
      cpy = sy + A * (ey - sy);
      dfx = ex - cpx;
      dfy = ey - cpy;
      dist = norm_ax(dfx, dfy);
      if (dist == INFINITY) dist = 0.0;
    }
    // stage C: np.argmax over this tile's vertices: first NaN wins, else first maximum
    unsigned long long k2 = !vact ? 0ull : (isnan(dist) ? ~0ull : (unsigned long long)__double_as_longlong(dist) + 1ull);
    const unsigned hi = (unsigned)(k2 >> 32), lo = (unsigned)k2;
    const unsigned mhi = __reduce_max_sync(FULL, hi);
    const bool t1 = hi == mhi;
    const unsigned mlo = __reduce_max_sync(FULL, t1 ? lo : 0u);
    const int wl = __ffs(__ballot_sync(FULL, t1 && lo == mlo)) - 1;
    const double wdist = shfl_d(dist, wl);
    const bool take = !have || (!isnan(b_dist) && (isnan(wdist) || wdist > b_dist));
    if (take) {
      have = true;
      b_dist = wdist;
      b_cpx = shfl_d(cpx, wl); b_cpy = shfl_d(cpy, wl);
      b_dfx = shfl_d(dfx, wl); b_dfy = shfl_d(dfy, wl);
      b_a = shfl_d(A, wl);
      b_edge = __shfl_sync(FULL, idx, wl);
    }
    wsync();
#ifdef MOOG_PROFILE_DCV
    ctr_add(e, CT_CYC_RESOLVE, clock64() - tp2 + tb);
#endif
  }
  const bool any_cross = __any_sync(FULL, my_cross) != 0;
  if (!any_cross) return;  // collisions.py:177-179
  o.has_point = 1;
  o.has_since = 1;
  o.px = b_cpx; o.py = b_cpy;
  o.sx = b_dfx; o.sy = b_dfy;
  if (b_a > 1) {  // collisions.py:214-217
    o.future = 1;
    return;
  }
  double2 e0 = P1[b_edge], e1 = P1[(b_edge + 1 == n1) ? 0 : b_edge + 1];
  double dvx = e1.x - e0.x, dvy = e1.y - e0.y;
  double nx = dvy, ny = -1.0 * dvx;
  double nn = norm1(nx, ny);
  o.nx = nx / nn;
  o.ny = ny / nn;
  double f = dot2(o.sx, o.sy, dvx, dvy) / dot2(dvx, dvy, dvx, dvy);
  o.qx = o.sx - dvx * f;
  o.qy = o.sy - dvy * f;
}

__device__ __noinline__ void directed_collision_vectors(const Env &, int s0, int s1, double dt, CVec &o) {
  const Env e = env_view();
  if (e.dcv_tile == DCV_TILE_MAX)
    directed_collision_vectors_impl<DCV_TILE_MAX>(e, s0, s1, dt, o);
  else
    directed_collision_vectors_impl<DCV_TILE_MIN>(e, s0, s1, dt, o);
}

// collisions.py:235-289 _get_collision_vectors
__device__ inline void get_collision_vectors(const Env &e, int s0, int s1, double dt, CVec &o) {
  CVec c0, c1;
  if (blockDim.x == 64) {
    // the helper warp computes the second direction while this warp computes the first
    int *req = (int *)e.xchg;
    wsync();
    if (e.lane == 0) { req[0] = HELPER_DCV; req[1] = s0; req[2] = s1; }
#ifdef MOOG_PROFILE_GCV
    long long ta = clock64();
#endif
    cta_bar(1);                                       // request visible, helper released
    directed_collision_vectors(e, s1, s0, dt, c0);
#ifdef MOOG_PROFILE_GCV
    long long tb = clock64();
#endif
    cta_bar(2);                                       // helper's result visible
#ifdef MOOG_PROFILE_GCV
    ctr_add(e, CT_NARROW, 1);
    ctr_add(e, CT_CYC_NARROW, tb - ta);
    ctr_add(e, CT_CYC_RESOLVE, clock64() - tb);
#endif
    c1 = *(const CVec *)(e.xchg + 16);
    wsync();
  } else {
    directed_collision_vectors(e, s1, s0, dt, c0);
    directed_collision_vectors(e, s0, s1, dt, c1);
  }
  double s0x = 0, s0y = 0, s1x = 0, s1y = 0;
  if (c0.has_point) {
    if (!c0.future) {
      c0.nx = -1.0 * c0.nx;
      c0.ny = -1.0 * c0.ny;
    }
    c0.sx = -1.0 * c0.sx;
    c0.sy = -1.0 * c0.sy;
    s0x = c0.sx;
    s0y = c0.sy;
  }
  if (c1.has_since) {
    s1x = c1.sx;
    s1y = c1.sy;
  }
  if (norm1(s0x, s0y) > norm1(s1x, s1y))
    o = c0;
  else
    o = c1;
}

// collisions.py:292-350
__device__ __noinline__ void collide_without_update_angle_vel(const Env &, int s0, int s1, const CVec &cv,
                                                            double elasticity, bool symmetric) {
  const Env e = env_view();
  double nx = cv.nx, ny = cv.ny;
  double nn = norm1(nx, ny);
  if (!(fabs(nn - 1.0) <= 1e-4 + 1e-5 * 1.0)) {
    int err = e.envi[MOOG_EI_ERR] | MOOG_ERR_NORMAL_NOT_UNIT;
    wsync();
    puti(e, &e.envi[MOOG_EI_ERR], err);
    wsync();
    return;
  }
  double v0x = DYN(e, MOOG_D_VX, s0), v0y = DYN(e, MOOG_D_VY, s0);
  double v1x = DYN(e, MOOG_D_VX, s1), v1y = DYN(e, MOOG_D_VY, s1);
  double m0 = STAT(e, MOOG_S_MASS, s0), m1 = STAT(e, MOOG_S_MASS, s1);
  double d0 = dot2(v0x, v0y, nx, ny), d1 = dot2(v1x, v1y, nx, ny);
  double v0nx = d0 * nx, v0ny = d0 * ny, v1nx = d1 * nx, v1ny = d1 * ny;
  double cmx, cmy;
  if (symmetric) {
    cmx = (v0nx * m0 + v1nx * m1) / (m0 + m1);
    cmy = (v0ny * m0 + v1ny * m1) / (m0 + m1);
  } else {
    cmx = v1nx;
    cmy = v1ny;
  }
  double k = 1 + elasticity;
  add_velocity(e, s0, k * (cmx - v0nx), k * (cmy - v0ny));
  add_velocity(e, s1, k * (cmx - v1nx), k * (cmy - v1ny));
}

// collisions.py:353-454
__device__ __noinline__ void collide_with_update_angle_vel(const Env &, int s0, int s1, const CVec &cv,
                                                         double elasticity, bool symmetric) {
  const Env e = env_view();
  double nx = cv.nx, ny = cv.ny;
  double m0 = STAT(e, MOOG_S_MASS, s0), m1 = STAT(e, MOOG_S_MASS, s1);
  double w0 = DYN(e, MOOG_D_ANGVEL, s0), w1 = DYN(e, MOOG_D_ANGVEL, s1);
  double i0 = moment_of_inertia(e, s0), i1 = moment_of_inertia(e, s1);
  double v0 = dot2(DYN(e, MOOG_D_VX, s0), DYN(e, MOOG_D_VY, s0), nx, ny);
  double v1 = dot2(DYN(e, MOOG_D_VX, s1), DYN(e, MOOG_D_VY, s1), nx, ny);
  double c0x = cv.px - DYN(e, MOOG_D_X, s0), c0y = cv.py - DYN(e, MOOG_D_Y, s0);
  double c1x = cv.px - DYN(e, MOOG_D_X, s1), c1y = cv.py - DYN(e, MOOG_D_Y, s1);
  double r0 = norm1(c0x, c0y), r1 = norm1(c1x, c1y);
  double sin0 = (c0x * ny - c0y * nx) / r0;
  double sin1 = (c1x * ny - c1y * nx) / r1;
  double sa = r0 * sin0, sb = r1 * sin1;
  double a = m0 + m1 + m0 * m1 * ((sa * sa / i0) + (sb * sb / i1));
  double b = (1 + elasticity) * (v0 - v1 + w0 * sa - w1 * sb);
  double dv0, dv1;
  if (symmetric) {
    dv0 = -1 * m1 * b / a;
    dv1 = m0 * b / a;
  } else {
    dv0 = -1 * m1 * b / (a - m0);
    dv1 = 0.0;
  }
  double dw0 = m0 * dv0 * sa / i0;
  double dw1 = m1 * dv1 * sb / i1;
  add_velocity(e, s0, dv0 * nx, dv0 * ny);
  add_velocity(e, s1, dv1 * nx, dv1 * ny);
  add_angvel(e, s0, dw0);
  add_angvel(e, s1, dw1);
}

__device__ __forceinline__ double sign_(double x) { return isnan(x) ? x : (double)((x > 0) - (x < 0)); }

// sprite.py:166-226 sprite_edge_crossings, reduced to what _position_correction
// consumes: the number of strict crossings and the crossing closest to (px, py)
// (first in row-major (i, j) order on ties -- argsort()[0] of collisions.py:688).
struct Closest { int count; double ptx, pty; int i0, i1; };

__device__ inline Closest closest_crossing(const Env &e, const double2 *P0, int n0, const double2 *P1, int n1,
                                           double px, double py) {
  bool act = e.lane < n0;
  double2 a1 = P0[act ? e.lane : 0];
  double2 a2 = P0[act ? ((e.lane + 1 == n0) ? 0 : e.lane + 1) : 0];
  double d0x = a2.x - a1.x, d0y = a2.y - a1.y;
  int cnt = 0, bj = 0x7fffffff;
  double bd = INFINITY, bx = 0, by = 0;
  bool bhave = false;
  for (int j = 0; j < n1; ++j) {
    double2 b1 = P1[j], b2 = P1[(j + 1 == n1) ? 0 : j + 1];
    double d1x = b2.x - b1.x, d1y = b2.y - b1.y;
    double den = (d0x * d1y - d0y * d1x) + EPS_INTERP;
    double qx = b1.x - a1.x, qy = b1.y - a1.y;
    double A = (qx * d1y - qy * d1x) / den;
    double B = (qx * d0y - qy * d0x) / den;
    if (act && (A > 0) && (A < 1) && (B > 0) && (B < 1)) {
      ++cnt;
      double cx = a1.x + A * d0x, cy = a1.y + A * d0y;
      double d = norm_ax(cx - px, cy - py);
      if (!bhave || d < bd) { bhave = true; bd = d; bx = cx; by = cy; bj = j; }
    }
  }
  int bi = bhave ? e.lane : 0x7fffffff;
  if (!bhave) bd = INFINITY;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    cnt += __shfl_xor_sync(FULL, cnt, off);
    double od = shflx_d(bd, off), ox = shflx_d(bx, off), oy = shflx_d(by, off);
    int oi = __shfl_xor_sync(FULL, bi, off), oj = __shfl_xor_sync(FULL, bj, off);
    bool take = (oi != 0x7fffffff) && (bi == 0x7fffffff || od < bd || (od == bd && oi < bi));
    if (take) { bd = od; bx = ox; by = oy; bi = oi; bj = oj; }
  }
  Closest c;
  c.count = cnt; c.ptx = bx; c.pty = by; c.i0 = bi; c.i1 = bj;
  return c;
}

// collisions.py:658-748 _position_correction.  `me` / `other` are the function's
// sprite_0 / sprite_1; ind_me / ind_other the edge indices of the closest crossing.
__device__ __noinline__ void position_correction(const Env &, double pt0x, double pt0y, int ind_me, int ind_other,
                                                 int me, int other, double out[2]) {
  const Env e = env_view();
  const double2 *Pme = e.vtx + e.voff[me];
  const double2 *Pother = e.vtx + e.voff[other];
  int n = META(e, MOOG_M_NV, me), no = META(e, MOOG_M_NV, other);
  int pt0_ind = ind_other;  // collisions.py:706 compares a value with itself -> always the edge branch
  int pt1_ind = (pt0_ind - 1 + no) % no;
  double q0x = Pother[pt1_ind].x, q0y = Pother[pt1_ind].y;
  double bx = Pother[pt0_ind].x - q0x, by = Pother[pt0_ind].y - q0y;
  double bn = norm1(bx, by);
  bx /= bn;
  by /= bn;
  double sg = sign_(dot2(DYN(e, MOOG_D_X, other) - q0x, DYN(e, MOOG_D_Y, other) - q0y, bx, by));
  double nvx = bx * -1 * sg, nvy = by * -1 * sg;
  int ind_forward = ind_me;
  int ind_backward = (ind_forward - 1 + n) % n;
  int parity, cur;
  if (dot2(Pme[ind_forward].x - pt0x, Pme[ind_forward].y - pt0y, nvx, nvy) > 0) {
    parity = 1;
    cur = ind_forward;
  } else if (dot2(Pme[ind_backward].x - pt0x, Pme[ind_backward].y - pt0y, nvx, nvy) > 0) {
    parity = -1;
    cur = ind_backward;
  } else {
    out[0] = out[1] = INFINITY;
    return;
  }
  double worst = 0;
  int guard = 0;
  for (;;) {
    double pen = dot2(Pme[cur].x - pt0x, Pme[cur].y - pt0y, nvx, nvy);
    if (!(pen > 0)) break;
    if (pen > worst) worst = pen;
    cur = (cur + parity + n) % n;
    if (++guard > n) {  // the reference would spin forever here
      int err = e.envi[MOOG_EI_ERR] | MOOG_ERR_DISJOINT_LOOP;
      wsync();
      puti(e, &e.envi[MOOG_EI_ERR], err);
      wsync();
      break;
    }
  }
  out[0] = worst * nvx;
  out[1] = worst * nvy;
}

// collisions.py:586-655 Collision._make_disjoint
__device__ __noinline__ void make_disjoint(const Env &, int s0, int s1, bool symmetric) {
  const Env e = env_view();
  const double2 *P0 = e.vtx + e.voff[s0];
  const double2 *P1 = e.vtx + e.voff[s1];
  int n0 = META(e, MOOG_M_NV, s0), n1 = META(e, MOOG_M_NV, s1);
  Closest k0 = closest_crossing(e, P0, n0, P1, n1, DYN(e, MOOG_D_X, s0), DYN(e, MOOG_D_Y, s0));
  if (k0.count <= 1) return;
  Closest k1 = closest_crossing(e, P0, n0, P1, n1, DYN(e, MOOG_D_X, s1), DYN(e, MOOG_D_Y, s1));
  double c0[2], c1[2];
  position_correction(e, k0.ptx, k0.pty, k0.i0, k0.i1, s0, s1, c0);
  position_correction(e, k1.ptx, k1.pty, k1.i1, k1.i0, s1, s0, c1);
  double cx, cy;
  if (norm1(c0[0], c0[1]) > norm1(c1[0], c1[1])) {
    cx = -1 * (1 + EPS_COLL) * c0[0];
    cy = -1 * (1 + EPS_COLL) * c0[1];
  } else {
    cx = (1 + EPS_COLL) * c0[0];
    cy = (1 + EPS_COLL) * c0[1];
  }
  if (!(isfinite(cx) && isfinite(cy))) cx = cy = 0.0;
  if (symmetric) {
    set_position(e, s0, DYN(e, MOOG_D_X, s0) + 0.5 * cx, DYN(e, MOOG_D_Y, s0) + 0.5 * cy);
    set_position(e, s1, DYN(e, MOOG_D_X, s1) - 0.5 * cx, DYN(e, MOOG_D_Y, s1) - 0.5 * cy);
  } else {
    set_position(e, s0, DYN(e, MOOG_D_X, s0) + cx, DYN(e, MOOG_D_Y, s0) + cy);
  }
}

// collisions.py:494-584 Collision.step; returns which sprites were moved
// (bit 0: s0, bit 1: s1)
__device__ inline int collision_step(const Env &e, const moog_op *op, int s0, int s1, bool first_overlap_known) {
  bool symmetric = (op->flags & MOOG_FL_SYMMETRIC) != 0;
  int changed = 0;
  int depth = 0;
  for (;;) {  // tail recursion of collisions.py:583-584
    if (depth > op->i[2]) return changed;
    if (s0 == s1) return changed;
    bool ov;
    long long t0 = clock64();
    if (first_overlap_known && depth == 0) {
      // the caller's broad phase already established that the circles and the
      // boxes meet: go straight to the outline test
      ov = path_intersects_filled(e, s0, s1);
      count_overlap(e, s0, s1, ov);
    } else {
      ov = overlaps(e, s0, s1);
    }
#if defined(MOOG_CYCLE_COUNTERS) && !defined(MOOG_PROFILE_PHASES) && !defined(MOOG_PROFILE_DCV) && !defined(MOOG_PROFILE_GCV) && !defined(MOOG_PROFILE_INTEG)
    ctr_add(e, CT_NARROW, 1);
    ctr_add(e, CT_CYC_NARROW, clock64() - t0);
#endif
    if (!ov) return changed;
    long long t1 = clock64();
    double dt = 1.0 / e.K;
    CVec cv;
    get_collision_vectors(e, s0, s1, dt, cv);
    if (!cv.has_point) {
      make_disjoint(e, s0, s1, symmetric);
      changed |= symmetric ? 3 : 1;
    } else {
      if (cv.future) {
        PROF_RESOLVE(e, t1);
        return changed;
      }
      ctr_add(e, CT_COLL, 1);
      changed |= symmetric ? 3 : 1;
      if (symmetric) {
        set_position(e, s0, DYN(e, MOOG_D_X, s0) - (0.5 + EPS_COLL) * cv.qx,
                     DYN(e, MOOG_D_Y, s0) - (0.5 + EPS_COLL) * cv.qy);
        set_position(e, s1, DYN(e, MOOG_D_X, s1) + (0.5 + EPS_COLL) * cv.qx,
                     DYN(e, MOOG_D_Y, s1) + (0.5 + EPS_COLL) * cv.qy);
      } else {
        set_position(e, s0, DYN(e, MOOG_D_X, s0) - (1. + EPS_COLL) * cv.qx,
                     DYN(e, MOOG_D_Y, s0) - (1. + EPS_COLL) * cv.qy);
      }
      if (op->flags & MOOG_FL_UPDATE_ANGLE_VEL)
        collide_with_update_angle_vel(e, s0, s1, cv, op->p[0], symmetric);
      else
        collide_without_update_angle_vel(e, s0, s1, cv, op->p[0], symmetric);
    }
    PROF_RESOLVE(e, t1);
    depth += 1;
  }
}

// ---------------------------------------------------------------------------
// Broad phase of the Collision entries.
//
// The reference visits every (sprite_0, sprite_1) pair of every Collision entry
// in itertools.product order and starts each visit with overlaps_sprite
// (collisions.py:516).  A visit whose overlap test is False changes nothing, and
// positions only change when a contact is resolved, so the outcome of "could
// this pair overlap at all" -- the circle test of sprite.py:464-466 AND the
// exact padded-box cull -- is evaluated for ALL pairs of ALL entries once per
// substep into bit matrices (row = sprite_0, bit = sprite_1), the set bits are
// visited in the reference's order, and after a resolved contact only the row
// and column of the sprites that moved are re-evaluated.
// ---------------------------------------------------------------------------

// per-lane: can (a, b) overlap?  (false is exact: the reference would return False)
__device__ __forceinline__ bool pair_candidate(const Env &e, int a, int b, bool valid) {
  if (!valid) b = a;
  bool c = valid && !boxes_apart(e, a, b);
  if (__any_sync(FULL, c)) {
    if (c) {
      const int fl = e.sflag[a] | e.sflag[b];
      double dx = DYN(e, MOOG_D_X, a) - DYN(e, MOOG_D_X, b);
      double dy = DYN(e, MOOG_D_Y, a) - DYN(e, MOOG_D_Y, b);
      // sprite.py:464-466 returns False when |centre distance| > r_a + r_b.  A candidate only has
      // to cover every pair for which that test could fail, so the square root is skipped: the
      // pair is dropped when the squared distance exceeds (r_a + r_b)^2 by more than any rounding
      // of either side (1e-9 relative); NaN compares false and stays a candidate, and overlaps()
      // repeats the reference's own test on whatever is left
      const double rr = STAT(e, MOOG_S_MAXR, a) + STAT(e, MOOG_S_MAXR, b);
      c = !(fl & SLF_ALLNAN) && !(dx * dx + dy * dy > rr * rr * (1.0 + 1e-9) && rr >= 0.0);
    }
  }
  return c;
}

// Near list ("Verlet list with a skin").  Evaluating every pair every substep is
// wasted on pairs that are far apart, so the pairs whose boxes could meet are
// listed once, together with a snapshot of the boxes.  Every slot s gets a drift
// allowance nskin[s] -- at least NEAR_SKIN / 2, and enough for the way it travels
// at its current velocity in what is left of this env-step, so that a sprite that
// was kicked out of the arena does not force a rebuild every substep -- and the
// pair (a, b) is listed when the boxes come within nskin[a] + nskin[b] of each
// other.  The list stays a superset of all possible candidates for as long as no
// box coordinate of s has drifted by nskin[s] since the snapshot.  Each refresh
// of the candidate matrices then tests 32 listed pairs per warp pass.

// entry = slot a | slot b << 8 | (bit index in cmask) << 16
__device__ __noinline__ void rebuild_near(const Env &) {
  const Env e = env_view();
  const int32_t *h = e.hdr;
  wsync();  // the caller's lanes have read the old snapshot (refresh_candidates)
  for (int i = e.lane; i < 4 * e.S; i += 32) e.aabb0[i] = (float)e.aabb[i];
  {
    const double rem = (double)(e.K - (int)e.ctr[CT_SUBSTEP]) / (double)e.K;
    for (int s = e.lane; s < e.S; s += 32) {
      const double vmax = fmax(fabs(DYN(e, MOOG_D_VX, s)), fabs(DYN(e, MOOG_D_VY, s)));  // fmax drops a NaN operand
      const bool fin = isfinite(DYN(e, MOOG_D_VX, s)) && isfinite(DYN(e, MOOG_D_VY, s));
      // rounded up to float; the snapshot's own float rounding (<= 2^-24 relative) is far inside the margin
      e.nskin[s] = fin ? __double2float_ru(fmax(0.5 * NEAR_SKIN, 1.2 * vmax * rem + 0.1 * NEAR_SKIN)) : INFINITY;
    }
  }
  wsync();
  int count = 0;
  bool overflow = false;
  for (int f = 0; f < h[MOOG_H_N_FORCES]; ++f) {
    const moog_op *op = e.ops + h[MOOG_H_FORCES] + f;
    if (op->kind != MOOG_F_COLLISION) continue;
    const int la = op->i[0], lb = op->i[1];
    const int na = e.cnt[la], nb = e.cnt[lb], sa = LOFF(e, la), sb = LOFF(e, lb);
    const int wpr = (LOFF(e, lb + 1) - sb + 31) >> 5;
#pragma unroll 1
    for (int i = 0; i < na && !overflow; ++i) {
      const int s0 = sa + i;
      const double k0 = (double)e.nskin[s0];
      const double bx0 = BOX(e, 0, s0) - k0, by0 = BOX(e, 1, s0) - k0;
      const double bx1 = BOX(e, 2, s0) + k0, by1 = BOX(e, 3, s0) + k0;
#pragma unroll 1
      for (int w = 0; w * 32 < nb; ++w) {
        const int j = w * 32 + e.lane;
        const int s1 = (j < nb) ? sb + j : s0;
        // NaN boxes compare false everywhere -> near
        const double k1 = (double)e.nskin[s1];
        const double x0 = bx0 - k1, y0 = by0 - k1, x1 = bx1 + k1, y1 = by1 + k1;
        const bool near = j < nb && s1 != s0 &&
                          !(x1 < BOX(e, 0, s1) || BOX(e, 2, s1) < x0 || y1 < BOX(e, 1, s1) || BOX(e, 3, s1) < y0);
        const unsigned m = __ballot_sync(FULL, near);
        const int n = __popc(m);
        if (count + n > NEAR_CAP) {
          overflow = true;
          break;
        }
        if (near)
          e.nearp[count + __popc(m & ((1u << e.lane) - 1u))] =
              (unsigned)s0 | ((unsigned)s1 << 8) | ((unsigned)((e.cmoff[f] + i * wpr + w) * 32 + e.lane) << 16);
        count += n;
      }
    }
  }
  if (e.lane == 0) e.ctr[CT_NEAR] = overflow ? -1 : count;
  wsync();
}

// every pair of every Collision entry (fallback when the near list overflowed)
__device__ __noinline__ void build_candidates_full(const Env &) {
  const Env e = env_view();
  const int32_t *h = e.hdr;
  for (int f = 0; f < h[MOOG_H_N_FORCES]; ++f) {
    const moog_op *op = e.ops + h[MOOG_H_FORCES] + f;
    if (op->kind != MOOG_F_COLLISION) continue;
    const int la = op->i[0], lb = op->i[1];
    const int na = e.cnt[la], nb = e.cnt[lb], sa = LOFF(e, la), sb = LOFF(e, lb);
    const int wpr = (LOFF(e, lb + 1) - sb + 31) >> 5;
#pragma unroll 1
    for (int i = 0; i < na; ++i)
#pragma unroll 1
      for (int w = 0; w * 32 < nb; ++w) {
        const int j = w * 32 + e.lane;
        unsigned m = __ballot_sync(FULL, pair_candidate(e, sa + i, sb + j, j < nb && sb + j != sa + i));
        if (e.lane == 0) e.cmask[e.cmoff[f] + i * wpr + w] = m;
      }
  }
  wsync();
}

// Bring the candidate matrices up to date with the current positions (start of
// a substep, and after every resolved contact).
__device__ inline void refresh_candidates(const Env &e, int n_cmask_words) {
  wsync();
  // has any box drifted too far since the near list was built?  (NaN -> yes)
  bool bad = false;
  for (int i = e.lane; i < 4 * e.S; i += 32) {
    const double b1 = e.aabb[i], b0 = (double)e.aabb0[i];  // (+-inf == +-inf: the all-covering box of a NaN sprite)
    // the allowance is charged for the float rounding of the snapshot (<= 2^-24 |b0|)
    bad |= !(fabs(b1 - b0) < (double)e.nskin[i >> 2] - (1.2e-7 * fabs(b0) + 1e-9)) && !(b1 == b0);
  }
  if (__any_sync(FULL, bad) || e.ctr[CT_NEAR] == -2) rebuild_near(e);
  const int n_near = (int)e.ctr[CT_NEAR];
  if (n_near < 0) {
    build_candidates_full(e);
    return;
  }
  for (int i = e.lane; i < n_cmask_words; i += 32) e.cmask[i] = 0u;
  wsync();
#pragma unroll 1
  for (int base = 0; base < n_near; base += 32) {
    const int k = base + e.lane;
    const unsigned ent = e.nearp[k < n_near ? k : 0];
    const bool c = pair_candidate(e, (int)(ent & 255u), (int)((ent >> 8) & 255u), k < n_near);
    if (c) atomicOr(&e.cmask[ent >> 21], 1u << ((ent >> 16) & 31u));
  }
  wsync();
}

// The same after a resolved contact, which moved s0 (moved & 1) and / or s1 (moved & 2) and
// nothing else: only their boxes can have drifted past the near list's allowance, and only the
// listed pairs they are part of can have changed their bit.
__device__ inline void refresh_candidates_moved(const Env &e, int n_cmask_words, int s0, int s1, int moved) {
  wsync();
  const int ma = (moved & 1) ? s0 : s1, mb = (moved & 2) ? s1 : ma;
  bool bad = false;
  if (e.lane < 8) {
    const int i = 4 * (e.lane < 4 ? ma : mb) + (e.lane & 3);
    const double b1 = e.aabb[i], b0 = (double)e.aabb0[i];
    bad = !(fabs(b1 - b0) < (double)e.nskin[i >> 2] - (1.2e-7 * fabs(b0) + 1e-9)) && !(b1 == b0);
  }
  const int n_near = (int)e.ctr[CT_NEAR];
  if (__any_sync(FULL, bad) || n_near < 0) {  // rebuild the list / no list: the general path
    refresh_candidates(e, n_cmask_words);
    return;
  }
#pragma unroll 1
  for (int base = 0; base < n_near; base += 32) {
    const int k = base + e.lane;
    const unsigned ent = e.nearp[k < n_near ? k : 0];
    const int a = (int)(ent & 255u), b = (int)((ent >> 8) & 255u);
    const bool inv = k < n_near && (a == ma || a == mb || b == ma || b == mb);
    const bool c = pair_candidate(e, a, b, inv);
    if (inv) {
      const unsigned bit = 1u << ((ent >> 16) & 31u);
      if (c) atomicOr(&e.cmask[ent >> 21], bit); else atomicAnd(&e.cmask[ent >> 21], ~bit);
    }
  }
  wsync();
}

// One Collision entry (physics.py:92-108 for a Collision force): the candidate
// pairs of its matrix in row-major order = itertools.product order.
__device__ inline void collision_op(const Env &e, const moog_op *op, int f, int n_cmask_words) {
  const int la = op->i[0], lb = op->i[1];
  const int na = e.cnt[la], nb = e.cnt[lb];
  const int sa = LOFF(e, la), sb = LOFF(e, lb);
  const int wpr = (LOFF(e, lb + 1) - sb + 31) >> 5;
  // every pair costs the reference one overlaps_sprite call (identical objects
  // return before it, collisions.py:513)
  {
    int lo = max(sa, sb), hi = min(sa + na, sb + nb);
    ctr_add(e, CT_CALLS, (long long)na * nb - (hi > lo ? hi - lo : 0));
  }
  const unsigned *M = e.cmask + e.cmoff[f];
  const int nwords = na * wpr;
  for (int base = 0; base < nwords; base += 32) {
    int widx = base + e.lane;
    unsigned nz = __ballot_sync(FULL, widx < nwords && M[widx] != 0u);
    while (nz) {
      const int t = __ffs(nz) - 1;
      nz &= nz - 1;
      const int wi = base + t;
      const int i = wi / wpr, w = wi - i * wpr;
      unsigned m = M[wi];
      while (m) {
        const int l = __ffs(m) - 1;
        m &= m - 1;
        const int s0 = sa + i, s1 = sb + w * 32 + l;
        ctr_add(e, CT_CALLS, -1);  // collision_step counts this pair's first call itself
        int moved = collision_step(e, op, s0, s1, true);
        if (moved) {
          refresh_candidates_moved(e, n_cmask_words, s0, s1, moved);
          // continue after (i, w, l) with the refreshed matrix
          m = M[wi] & ~((2u << l) - 1u);
          nz = __ballot_sync(FULL, widx < nwords && M[widx] != 0u) & ~((2u << t) - 1u);
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------
// forces (abstract_force.py:64-74 + the individual _compute_forces)
// ---------------------------------------------------------------------------
__device__ inline double noise_at(const Env &e, int col) {
  if (e.noise) return e.noise[(size_t)e.ctr[CT_SUBSTEP] * e.hdr[MOOG_H_NOISE_DIM] + col];
  return philox_uniform(e.seed, (uint32_t)e.env_id, (uint32_t)e.envi[MOOG_EI_STEP_COUNT],
                        (uint32_t)e.ctr[CT_SUBSTEP] | ((uint32_t)e.envi[MOOG_EI_EPISODES] << 8), (uint32_t)col);
}

// lane = sprite of the layer; a unary force only touches its own sprite's velocity
__device__ inline void force_unary_layer(const Env &e, const moog_op *op) {
  int la = op->i[0], n = e.cnt[la];
  // Sprites that share their velocity array (valias) see each other's in-place
  // updates: a layer that holds any is visited one sprite at a time.
  bool shared = false;
  for (int idx = e.lane; idx < n; idx += 32) shared |= valias(e, LOFF(e, la) + idx) != 0;
  const bool sequential = __any_sync(FULL, shared) != 0;
  const int stride = sequential ? 1 : 32;
  for (int base = 0; base < n; base += stride) {
    int idx = sequential ? base : base + e.lane;
    if (sequential) wsync();
    if (idx < n && (!sequential || e.lane == 0)) {
      int s = LOFF(e, la) + idx;
      double m = STAT(e, MOOG_S_MASS, s);
      double vx = DYN(e, MOOG_D_VX, s), vy = DYN(e, MOOG_D_VY, s);
      bool v32 = vel32(e, s);
      double fx = 0, fy = 0;
      bool done = false;
      switch (op->kind) {
        case MOOG_F_DRAG:  // friction.py:54-56
          if (v32) {
            // python-float scalars are weak: the whole chain runs in float32
            if (isfinite(m)) {
              double c = -1 * op->p[0], den = m * (double)e.K;
              DYN(e, MOOG_D_VX, s) = f32add(vx, f32div(f32mul(f32mul(c, vx), m), den));
              DYN(e, MOOG_D_VY, s) = f32add(vy, f32div(f32mul(f32mul(c, vy), m), den));
            }
            done = true;
          } else {
            fx = -1 * op->p[0] * vx * m;
            fy = -1 * op->p[0] * vy * m;
          }
          break;
        case MOOG_F_KINETIC_FRICTION: {  // friction.py:25-33
          double nrm = norm1(vx, vy);
          double ux = 0, uy = 0;
          if (nrm != 0) {
            ux = vx / nrm;
            uy = vy / nrm;
          }
          fx = -1 * op->p[0] * ux * m;
          fy = -1 * op->p[0] * uy * m;
          break;
        }
        case MOOG_F_DOWN_GRAVITY:  // gravity.py:21-23
          fx = op->p[0] * m * 0;
          fy = op->p[0] * m * 1;
          break;
        case MOOG_F_RANDOM: {  // random_force.py:22-26
          double u0 = noise_at(e, op->i[2] + 2 * idx), u1 = noise_at(e, op->i[2] + 2 * idx + 1);
          double r = 0.0 + (op->p[0] - 0.0) * u0;
          double th = 0.0 + (2 * M_PI - 0.0) * u1;
          fx = r * cos(th);
          fy = r * sin(th);
          break;
        }
      }
      if (!done && isfinite(m)) {  // abstract_force.py:64-74
        double den = m * (double)e.K;
        double nvx = vx + div_z(fx, den), nvy = vy + div_z(fy, den);
        if (v32) {
          nvx = f32r(nvx);
          nvy = f32r(nvy);
        }
        const int id = valias(e, s);
        if (id) {  // (sequential mode, lane 0)
          for (int t = 0; t < e.S; ++t)
            if (valias(e, t) == id) {
              DYN(e, MOOG_D_VX, t) = nvx;
              DYN(e, MOOG_D_VY, t) = nvy;
            }
        } else {
          DYN(e, MOOG_D_VX, s) = nvx;
          DYN(e, MOOG_D_VY, s) = nvy;
        }
      }
    }
  }
  wsync();
}

__device__ inline void newton(const Env &e, int s, double fx, double fy) {
  double m = STAT(e, MOOG_S_MASS, s);
  if (!isfinite(m)) return;
  double den = m * (double)e.K;
  add_velocity(e, s, fx / den, fy / den);
}

__device__ inline void force_binary(const Env &e, const moog_op *op, int s0, int s1) {
  // gravity.py:44-60, distance_fn_force.py:30-45
  double dx = DYN(e, MOOG_D_X, s1) - DYN(e, MOOG_D_X, s0);
  double dy = DYN(e, MOOG_D_Y, s1) - DYN(e, MOOG_D_Y, s0);
  double dist = norm1(dx, dy);
  double f0x = 0, f0y = 0, f1x = 0, f1y = 0;
  if (dist != 0.) {
    double ux = dx / dist, uy = dy / dist;
    double mag = 0;
    if (op->kind == MOOG_F_GRAVITY) {
      mag = op->p[0] * STAT(e, MOOG_S_MASS, s0) * STAT(e, MOOG_S_MASS, s1) * dist;
    } else if (op->kind == MOOG_F_DIST_LINEAR) {  // distance_fn_force.py:48-74
      mag = op->p[0] + op->p[1] * dist;
      if (!(op->flags & MOOG_FL_APPLY_DISTANT) && dist > op->p[2]) mag = 0;
      if (!(op->flags & MOOG_FL_APPLY_NEARBY) && dist < op->p[2]) mag = 0;
    } else if (op->kind == MOOG_F_DIST_SPRING) {  // distance_fn_force.py:77-89
      mag = -1. * op->p[0] * (dist - op->p[1]);
    }
    f1x = mag * ux;
    f1y = mag * uy;
    if (op->flags & MOOG_FL_SYMMETRIC) {
      f0x = -1 * f1x;
      f0y = -1 * f1y;
    }
  }
  newton(e, s0, f0x, f0y);
  newton(e, s1, f1x, f1y);
}

// ---------------------------------------------------------------------------
// corrective physics
// ---------------------------------------------------------------------------

// q-th live sprite of a layer list; -1 past the end
__device__ inline int list_slot(const Env &e, int start, int n, int q) {
  for (int k = 0; k < n; ++k) {
    int l = e.ipool[start + k];
    int c = e.cnt[l];
    if (q < c) return LOFF(e, l) + q;
    q -= c;
  }
  return -1;
}
__device__ inline int list_count(const Env &e, int start, int n) {
  int t = 0;
  for (int k = 0; k < n; ++k) t += e.cnt[e.ipool[start + k]];
  return t;
}

// tether_physics.py:16-91.  The sprite set is given by `pick(i)`.
template <class Pick>
__device__ inline void tether_sprites(const Env &e, Pick pick, int n, bool update_angle_vel, bool has_anchor,
                                      double ax, double ay) {
  if (n == 0) return;
  double total_mass = 0;
  for (int i = 0; i < n; ++i) total_mass = total_mass + STAT(e, MOOG_S_MASS, pick(i));
  if (isinf(total_mass)) return;
  double cx = 0, cy = 0, mx = 0, my = 0;
  for (int i = 0; i < n; ++i) {
    int s = pick(i);
    double m = STAT(e, MOOG_S_MASS, s);
    cx = cx + m * DYN(e, MOOG_D_X, s);
    cy = cy + m * DYN(e, MOOG_D_Y, s);
    mx = mx + m * DYN(e, MOOG_D_VX, s);
    my = my + m * DYN(e, MOOG_D_VY, s);
  }
  cx /= total_mass;
  cy /= total_mass;
  double tvx = mx / total_mass, tvy = my / total_mass;
  if (has_anchor) {
    cx = ax;
    cy = ay;
    tvx = tvy = 0;
  }
  if (update_angle_vel) {
    double Ltot = 0, Itot = 0;
    for (int i = 0; i < n; ++i) {
      int s = pick(i);
      double vx = DYN(e, MOOG_D_VX, s), vy = DYN(e, MOOG_D_VY, s);
      double dpx = vx / e.K, dpy = vy / e.K;
      double px = (DYN(e, MOOG_D_X, s) + 0.5 * dpx) - cx;
      double py = (DYN(e, MOOG_D_Y, s) + 0.5 * dpy) - cy;
      double r = norm1(px, py);
      px /= r;
      py /= r;
      double qx = 0 * px + -1 * py, qy = 1 * px + 0 * py;
      double perp_vel = dot2(vx - tvx, vy - tvy, qx, qy);
      double m = STAT(e, MOOG_S_MASS, s);
      double I = moment_of_inertia(e, s);
      double Lz = perp_vel * m * r;
      Lz += DYN(e, MOOG_D_ANGVEL, s) * I;
      Ltot = Ltot + Lz;
      Itot = Itot + (I + m * r * r);
      wsync();
      put(e, &TMP(e, 0, s), r);
      put(e, &TMP(e, 1, s), qx);
      put(e, &TMP(e, 2, s), qy);
      wsync();
    }
    double w = Ltot / Itot;
    for (int i = 0; i < n; ++i) {
      int s = pick(i);
      double r = TMP(e, 0, s), qx = TMP(e, 1, s), qy = TMP(e, 2, s);
      assign_velocity(e, s, tvx + r * qx * w, tvy + r * qy * w);
      put(e, &DYN(e, MOOG_D_ANGVEL, s), w);
      set_angvel_kind(e, s, KIND_F64);
    }
  } else {
    // `s.velocity = total_velocity`: the SAME ndarray object for every sprite
    const int id = new_valias(e);
    for (int i = 0; i < n; ++i) {
      int s = pick(i);
      assign_velocity(e, s, tvx, tvy);
      puti(e, &META(e, MOOG_M_FLAGS, s), META(e, MOOG_M_FLAGS, s) | (id << MOOG_SF_VALIAS_SHIFT));
      put(e, &DYN(e, MOOG_D_ANGVEL, s), 0.);
      set_angvel_kind(e, s, KIND_WEAK);
    }
  }
}


// ---------------------------------------------------------------------------
// maze_lib.Maze, RandomMazeWalk, MazePhysics.  Per-sprite scalar logic on values every
// lane reads from shared memory: all lanes compute the same thing, lane 0 stores.
// ---------------------------------------------------------------------------
#define MAZE_EPS 1e-5 /* maze_physics.py:15, maze_walk.py:14 */

struct MazeV { int n; const double *rows; double grid, half; };

__device__ __forceinline__ MazeV maze_of(const Env &e, int off) {
  MazeV m;
  m.n = (int)e.envf[off];
  m.rows = e.envf + off + 1;
  m.grid = 1. / m.n;      // maze.py:32
  m.half = 0.5 * m.grid;  // maze.py:33
  return m;
}
// maze.py:113-118
__device__ __forceinline__ double maze_open(const MazeV &m, int i, int j) {
  if (i < 0 || j < 0 || i >= m.n || j >= m.n) return 0.0;
  return (((unsigned long long)m.rows[j] >> i) & 1ull) ? 0.0 : 1.0;
}
// maze.py:120-126: v[2 * axis + dir]
__device__ inline void maze_valid(const MazeV &m, int i, int j, double *v) {
  v[0] = maze_open(m, i - 1, j); v[1] = maze_open(m, i + 1, j);
  v[2] = maze_open(m, i, j - 1); v[3] = maze_open(m, i, j + 1);
}
// numpy floor_divide for doubles (npy_divmod)
__device__ inline double np_floor_divide(double a, double b) {
  if (b == 0) return a / b;
  double mod = fmod(a, b);
  double div = (a - mod) / b;
  if (mod != 0) {
    if ((b < 0) != (mod < 0)) div -= 1.0;
  }
  double fl;
  if (div != 0) {
    fl = floor(div);
    if (div - fl > 0.5) fl += 1.0;
  } else {
    fl = copysign(0.0, a / b);
  }
  return fl;
}

// maze_walk.py:159-196 RandomMazeWalk._step_sprite (+ _get_pos_vel :46-79, _update_valid_directions :122-157)
__device__ __noinline__ void maze_walk_layer(const Env &, const moog_op *op) {
  const Env e = env_view();
  const int la = op->i[0];
  const MazeV m = maze_of(e, op->i[3]);
  const double speed = op->p[0];
  const double K = (double)e.K;
  for (int idx = 0; idx < e.cnt[la]; ++idx) {
    const int s = LOFF(e, la) + idx;
    if (isinf(STAT(e, MOOG_S_MASS, s))) continue;
    double pos[2] = {DYN(e, MOOG_D_X, s), DYN(e, MOOG_D_Y, s)};
    double vel[2] = {speed * sign_(DYN(e, MOOG_D_VX, s)), speed * sign_(DYN(e, MOOG_D_VY, s))};
    double nxt[2] = {pos[0] + vel[0] / K, pos[1] + vel[1] / K};
    int near_[2];
    double inter[2];
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      near_[a] = (int)rint(pos[a] / m.grid - 0.5);
      inter[a] = m.grid * near_[a] + m.half;
    }
    const double d_next_cur = fabs(nxt[0] - pos[0]) + fabs(nxt[1] - pos[1]);
    const double d_int_next = fabs(nxt[0] - inter[0]) + fabs(nxt[1] - inter[1]);
    const bool entering = d_next_cur > d_int_next;  // the reference compares against the same quantity twice
    double valid[4];
    if (entering) {
      maze_valid(m, near_[0], near_[1], valid);
      if (op->flags & MOOG_FL_PREVENT_BACKTRACKING) {
        const int axis = fabs(vel[1]) > fabs(vel[0]) ? 1 : 0;  // np.argmax: first maximum
        const double direction = sign_(axis ? vel[1] : vel[0]);
        if (direction != 0) {
          const int fwd = (int)(0.5 * (1 + direction)), back = (int)(0.5 * (1 - direction));
          const bool can_continue = valid[2 * axis + fwd] != 0;
          if (!can_continue && (op->flags & MOOG_FL_ALLOW_WALL_BACKTRACKING)) {
          } else if (can_continue && (op->flags & MOOG_FL_ONLY_TURN_AT_WALL)) {
            valid[0] = valid[1] = valid[2] = valid[3] = 0;
            valid[2 * axis + fwd] = 1;
          } else {
            valid[2 * axis + back] = 0;
          }
        }
      }
    } else if (vel[0] == 0. && vel[1] == 0.) {
      const bool on0 = fabs((m.half + near_[0] * m.grid) - pos[0]) < MAZE_EPS;
      const bool on1 = fabs((m.half + near_[1] * m.grid) - pos[1]) < MAZE_EPS;
      if (on0 && on1) {
        maze_valid(m, near_[0], near_[1], valid);
      } else {
        const int row = 1 - (on0 ? 0 : (on1 ? 1 : 0));  // 1 - np.argmax(on_grid)
        valid[0] = valid[1] = valid[2] = valid[3] = 0;
        valid[2 * row] = valid[2 * row + 1] = 1;
      }
    } else {
      assign_velocity(e, s, vel[0], vel[1]);
      continue;
    }
    // sample = valid_directions * np.random.rand(2, 2); argmax of the ravel (first maximum)
    int best = 0;
    double bv = valid[0] * noise_at(e, op->i[2] + 4 * idx);
#pragma unroll
    for (int k = 1; k < 4; ++k) {
      const double v = valid[k] * noise_at(e, op->i[2] + 4 * idx + k);
      if (v > bv) { bv = v; best = k; }
    }
    const double nvv = (1 + MAZE_EPS) * speed * (2 * (best % 2) - 1);
    if (best / 2 == 0) vel[0] = nvv; else vel[1] = nvv;
    assign_velocity(e, s, vel[0], vel[1]);
  }
}

// maze_physics.py:51-112 _get_position_affordances -> aff[2 * axis + dir]; false when off the grid
__device__ inline bool maze_affordances(const MazeV &m, double p0, double p1, double *aff) {
  int near_[2], inds[2];
  bool on[2];
  const double pos[2] = {p0, p1};
#pragma unroll
  for (int a = 0; a < 2; ++a) {
    near_[a] = (int)rint(pos[a] / m.grid - 0.5);
    const double rounded = m.half + near_[a] * m.grid;
    on[a] = fabs(rounded - pos[a]) < MAZE_EPS;
    inds[a] = (int)np_floor_divide(pos[a] - m.half, m.grid);
    if (on[a]) inds[a] = near_[a];
  }
  aff[0] = aff[1] = aff[2] = aff[3] = 0;
  if (!on[0] && !on[1]) return false;
  if (on[0] && on[1]) {
    double v[4];
    maze_valid(m, inds[0], inds[1], v);
    aff[0] = v[0] * m.grid * -1.; aff[1] = v[1] * m.grid * 1.;
    aff[2] = v[2] * m.grid * -1.; aff[3] = v[3] * m.grid * 1.;
  } else {
    const int i = on[0] ? 1 : 0;
    const double pi_ = i ? p1 : p0;
    aff[2 * i] = inds[i] * m.grid + m.half - pi_;
    aff[2 * i + 1] = (inds[i] + 1) * m.grid + m.half - pi_;
  }
  return true;
}

// maze_physics.py:114-167 _get_new_velocity, the recursion unrolled: every vertex the sprite
// passes pushes the part of the velocity spent on the way there (`velocity *= scaling;
// velocity[1 - axis] = 0`); the sums `velocity += velocity_post_vertex` are taken innermost first.
#define MAZE_MAX_VERTICES 6
__device__ inline bool maze_new_velocity(const MazeV &m, double p0, double p1, double v0, double v1, double *aff0,
                                         double *out) {
  double pre[MAZE_MAX_VERTICES][2];
  int depth = 0;
  double pos[2] = {p0, p1}, vel[2] = {v0, v1};
  double aff[4] = {aff0[0], aff0[1], aff0[2], aff0[3]};
  double r0 = 0, r1 = 0;
  int axis = -1;
  for (int guard = 0; guard < 4 * MAZE_MAX_VERTICES; ++guard) {
    if (axis < 0) axis = fabs(vel[1]) > fabs(vel[0]) ? 1 : 0;
    const double va = axis ? vel[1] : vel[0];
    if (aff[2 * axis] <= va && va <= aff[2 * axis + 1]) {
      if (axis) vel[0] = 0; else vel[1] = 0;
      r0 = vel[0]; r1 = vel[1];
      goto unwind;
    }
    int direction = va > 0 ? 1 : 0;  // int(0.5 + 0.5 * sign)
    if (aff[2 * axis + direction] == 0) {
      axis = 1 - axis;
      const double vb = axis ? vel[1] : vel[0];
      direction = vb > 0 ? 1 : 0;
      if (aff[2 * axis + direction] == 0 || vb == 0) {
        r0 = r1 = 0.;
        goto unwind;
      }
      continue;  // _get_new_velocity(position, velocity, affordances, axis=axis)
    }
    if (depth >= MAZE_MAX_VERTICES) return false;
    const double step = aff[2 * axis + direction];
    if (axis) pos[1] += step; else pos[0] += step;
    double vaff[4];
    if (!maze_affordances(m, pos[0], pos[1], vaff)) return false;
    const double scaling = step / va;
    const double rem0 = (1. - scaling) * vel[0], rem1 = (1. - scaling) * vel[1];
    vel[0] *= scaling; vel[1] *= scaling;
    if (axis) vel[0] = 0; else vel[1] = 0;
    pre[depth][0] = vel[0]; pre[depth][1] = vel[1];
    ++depth;
    vel[0] = rem0; vel[1] = rem1;
    aff[0] = vaff[0]; aff[1] = vaff[1]; aff[2] = vaff[2]; aff[3] = vaff[3];
    axis = -1;
  }
  return false;
unwind:
  while (depth > 0) {
    --depth;
    r0 = pre[depth][0] + r0;
    r1 = pre[depth][1] + r1;
  }
  out[0] = r0; out[1] = r1;
  return true;
}

// sprite.py:531-540 angle setter (`sprite.angle = a`, a an np.float64): rotate_around(x, y, a - angle)
__device__ inline void set_angle_f64(const Env &e, int s, double a, int kind = KIND_F64) {
  Aff mtx = aff_identity();
  aff_rotate_around(mtx, DYN(e, MOOG_D_X, s), DYN(e, MOOG_D_Y, s), a - DYN(e, MOOG_D_ANG, s));
  const int n = META(e, MOOG_M_NV, s);
  double2 *v = e.vtx + e.voff[s];
  wsync();
  // the rotated outline, its box and NaN / inf classification
  bool fin = true, nan_all = true;
  double xmin = INFINITY, xmax = -INFINITY, ymin = INFINITY, ymax = -INFINITY;
  for (int i = e.lane; i < n; i += 32) {
    const double2 p = v[i];
    const double2 q = make_double2(mtx.m0 * p.x + mtx.m1 * p.y + mtx.m2, mtx.m3 * p.x + mtx.m4 * p.y + mtx.m5);
    v[i] = q;
    fin &= isfinite(q.x) && isfinite(q.y);
    nan_all &= isnan(q.x) && isnan(q.y);
    xmin = fmin(xmin, q.x); xmax = fmax(xmax, q.x);
    ymin = fmin(ymin, q.y); ymax = fmax(ymax, q.y);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    xmin = fmin(xmin, shflx_d(xmin, o)); xmax = fmax(xmax, shflx_d(xmax, o));
    ymin = fmin(ymin, shflx_d(ymin, o)); ymax = fmax(ymax, shflx_d(ymax, o));
  }
  const bool nonfinite = !__all_sync(FULL, fin);
  const bool allnan = n > 0 && __all_sync(FULL, nan_all);
  wsync();
  bool st = false;
  for (int i = e.lane; i < n; i += 32) st |= steep_edge(v[i].x, v[(i + 1 == n) ? 0 : i + 1].x);
  const bool steep = __any_sync(FULL, st) != 0;
  if (e.lane == 0) {
    DYN(e, MOOG_D_ANG, s) = a;
    META(e, MOOG_M_FLAGS, s) = (META(e, MOOG_M_FLAGS, s) & ~(3 << MOOG_SF_ANG_SHIFT)) | (kind << MOOG_SF_ANG_SHIFT);
    e.sflag[s] = (e.sflag[s] & SLF_SHORT_EDGE) | (nonfinite ? SLF_NONFINITE : 0) | (allnan ? SLF_ALLNAN : 0) |
                 (steep ? SLF_STEEP : 0);
    store_box(e, s, xmin, ymin, xmax, ymax, nonfinite, steep);
  }
  wsync();
}

// maze_physics.py:189-211 _update_sprite_in_maze (+ _update_sprite_angle :169-187) for the avatar layers
__device__ __noinline__ void maze_physics(const Env &, const moog_op *op) {
  const Env e = env_view();
  const MazeV m = maze_of(e, op->i[2]);
  const int n = list_count(e, op->i[0], op->i[1]);
  for (int q = 0; q < n; ++q) {
    const int s = list_slot(e, op->i[0], op->i[1], q);
    double v0 = DYN(e, MOOG_D_VX, s), v1 = DYN(e, MOOG_D_VY, s);
    if ((v0 == 0 && v1 == 0) || isnan(v0) || isnan(v1)) continue;
    if (!isnan(op->p[1])) {  // np.clip(velocity, -max_speed, max_speed)
      v0 = fmin(fmax(v0, -op->p[1]), op->p[1]);
      v1 = fmin(fmax(v1, -op->p[1]), op->p[1]);
    }
    if (!isnan(op->p[0])) {
      v0 += sign_(v0); v0 *= op->p[0];
      v1 += sign_(v1); v1 *= op->p[0];
    }
    const double p0 = DYN(e, MOOG_D_X, s), p1 = DYN(e, MOOG_D_Y, s);
    double aff[4], nv[2];
    bool ok = maze_affordances(m, p0, p1, aff);
    if (ok) {
      set_position(e, s, p0, p1);  // sprite.position = np.copy(position): a translation by exactly zero
      ok = maze_new_velocity(m, p0, p1, v0, v1, aff, nv);
    }
    if (!ok) {
      const int err = e.envi[MOOG_EI_ERR] | MOOG_ERR_OFF_MAZE_GRID;
      wsync();
      puti(e, &e.envi[MOOG_EI_ERR], err);
      wsync();
      continue;
    }
    double new_angle;
    if (nv[0] == 0 && nv[1] == 0) {
      new_angle = NAN;
    } else if (nv[1] == 0) {
      new_angle = -0.5 * sign_(nv[0]) * M_PI;
    } else if (sign_(nv[1]) > 0) {
      new_angle = atan(-nv[0] / nv[1]);
    } else {
      new_angle = M_PI + atan(-nv[0] / nv[1]);
    }
    if (!isnan(new_angle) && fabs(new_angle - DYN(e, MOOG_D_ANG, s)) > MAZE_EPS) set_angle_f64(e, s, new_angle);
    assign_velocity(e, s, nv[0], nv[1]);
  }
}

__device__ __noinline__ void corrective(const Env &, const moog_op *op) {
  const Env e = env_view();
  switch (op->kind) {
    case MOOG_C_MAZE_PHYSICS:  // maze_physics.py:205-211
      maze_physics(e, op);
      break;
    case MOOG_C_TETHER: {  // tether_physics.py:126-140
      int st = op->i[0], nl = op->i[1];
      int n = list_count(e, st, nl);
      tether_sprites(e, [&](int i) { return list_slot(e, st, nl, i); }, n,
                     (op->flags & MOOG_FL_UPDATE_ANGLE_VEL) != 0, (op->flags & MOOG_FL_HAS_ANCHOR) != 0, op->p[0],
                     op->p[1]);
      break;
    }
    case MOOG_C_TETHER_ZIPPED: {  // tether_physics.py:186-201
      int nl = op->i[1];
      int c0 = nl ? e.cnt[e.ipool[op->i[0]]] : 0;
      for (int q = 1; q < nl; ++q)
        if (e.cnt[e.ipool[op->i[0] + q]] != c0) {
          int err = e.envi[MOOG_EI_ERR] | MOOG_ERR_TETHER_ZIP;
          wsync();
          puti(e, &e.envi[MOOG_EI_ERR], err);
          wsync();
          return;
        }
      for (int i = 0; i < c0; ++i) {
        int st = op->i[0];
        tether_sprites(e, [&](int q) { return LOFF(e, e.ipool[st + q]) + i; }, nl,
                       (op->flags & MOOG_FL_UPDATE_ANGLE_VEL) != 0, (op->flags & MOOG_FL_HAS_ANCHOR) != 0,
                       op->p[0], op->p[1]);
      }
      break;
    }
    case MOOG_C_CONSTANT_SPEED: {  // constant_speed.py:34-46
      int n = list_count(e, op->i[0], op->i[1]);
      for (int i = 0; i < n; ++i) {
        int s = list_slot(e, op->i[0], op->i[1], i);
        double vx = DYN(e, MOOG_D_VX, s), vy = DYN(e, MOOG_D_VY, s);
        if (vel32(e, s)) {
          // a float32 velocity array: np.linalg.norm is sqrt(x.dot(x)) in float32 (products and
          // sum each rounded, no fma) and `speed * velocity / norm` stays float32
          const float fx = (float)vx, fy = (float)vy;
          const float nf = __fsqrt_rn(__fadd_rn(__fmul_rn(fx, fx), __fmul_rn(fy, fy)));
          if (nf != 0) {
            const float sp32 = (float)op->p[0];
            assign_velocity(e, s, (double)__fdiv_rn(__fmul_rn(sp32, fx), nf), (double)__fdiv_rn(__fmul_rn(sp32, fy), nf));
            const int fl = META(e, MOOG_M_FLAGS, s) | MOOG_SF_VEL32;
            wsync();
            puti(e, &META(e, MOOG_M_FLAGS, s), fl);
            wsync();
          }
          continue;
        }
        double nv = norm1(vx, vy);
        if (nv != 0) assign_velocity(e, s, op->p[0] * vx / nv, op->p[0] * vy / nv);
      }
      break;
    }
  }
}

// ---------------------------------------------------------------------------
// Euler integration of every sprite (physics.py:113-117, sprite.py:426-430)
// ---------------------------------------------------------------------------
#define TF_MOVE 1
#define TF_ROT 2
#define TF_CLASSIFY 4

__device__ __forceinline__ void integrate_all_impl(const Env &e) {
  double dt = 1. / e.K;
#ifdef MOOG_PROFILE_INTEG
  long long ti0 = clock64(), ti1 = 0;
#endif
  for (int base = 0; base < e.S; base += 32) {
    // phase 1: lane = slot.  New position / angle and the affine update of the outline
    // (kept in this lane's registers; phase 2 fetches them by shuffle).
    const int s = base + e.lane;
    int flag = 0;
    double tx = 0.0, ty = 0.0;
    Aff m = aff_identity();
    if (s < e.S) {
      int vs_layer_live = 0;
      // live?  slots of layer l are [LOFF(l), LOFF(l) + cnt[l])
      for (int l = 0; l < e.L; ++l)
        if (s >= LOFF(e, l) && s < LOFF(e, l) + e.cnt[l]) vs_layer_live = 1;
      if (vs_layer_live) {
        bool v32 = vel32(e, s);
        double vx = DYN(e, MOOG_D_VX, s), vy = DYN(e, MOOG_D_VY, s);
        double dx = v32 ? f32mul(dt, vx) : dt * vx;
        double dy = v32 ? f32mul(dt, vy) : dt * vy;
        double ox = DYN(e, MOOG_D_X, s), oy = DYN(e, MOOG_D_Y, s);
        double nx = ox + dx, ny = oy + dy;
        tx = nx - ox;
        ty = ny - oy;
        DYN(e, MOOG_D_X, s) = nx;
        DYN(e, MOOG_D_Y, s) = ny;
        if (!(tx == 0.0 && ty == 0.0)) {
          flag |= TF_MOVE;
          BOX(e, 0, s) = BOX(e, 0, s) + tx;
          BOX(e, 1, s) = BOX(e, 1, s) + ty;
          BOX(e, 2, s) = BOX(e, 2, s) + tx;
          BOX(e, 3, s) = BOX(e, 3, s) + ty;
        }
        double w = DYN(e, MOOG_D_ANGVEL, s);
        if (w != 0) {  // `if self._angle_vel:` (NaN is truthy)
          int wk = angvel_kind(e, s), ak = ang_kind(e, s);
          double t = (wk == KIND_F32) ? f32mul(dt, w) : dt * w;
          double a = DYN(e, MOOG_D_ANG, s), na;
          int nk;
          if (ak == KIND_F64 || wk == KIND_F64) { na = a + t; nk = KIND_F64; }
          else if (ak == KIND_WEAK && wk == KIND_WEAK) { na = a + t; nk = KIND_WEAK; }
          else { na = f32add(a, t); nk = KIND_F32; }
          // sprite.py:531-540: rotate_around(x, y, a_new - a_old) about the NEW position
          double dth = (nk == KIND_F32 && ak != KIND_F64) ? f32sub(na, a) : na - a;
          aff_rotate_around(m, nx, ny, dth);
          DYN(e, MOOG_D_ANG, s) = na;
          META(e, MOOG_M_FLAGS, s) = (META(e, MOOG_M_FLAGS, s) & ~(3 << MOOG_SF_ANG_SHIFT)) | (nk << MOOG_SF_ANG_SHIFT);
          flag |= TF_ROT;
        }
        if (!(isfinite(tx) && isfinite(ty))) flag |= TF_CLASSIFY;
      }
      if ((flag & TF_ROT) && (e.sflag[s] & SLF_NONFINITE)) flag |= TF_CLASSIFY;
      e.sflag[s] = (e.sflag[s] & SLF_MASK) | (flag << 8);
    }
#ifdef MOOG_PROFILE_INTEG
    ti1 = clock64();
    ctr_add(e, CT_NARROW, ti1 - ti0);
#endif
    // phase 2a: the slots that also rotate, one at a time, lane = vertex of the outline (the
    // translate-only slots -- the common case -- are left to the flat pass below)
    unsigned mv = __ballot_sync(FULL, flag != 0);
    const unsigned rot = __ballot_sync(FULL, (flag & TF_ROT) != 0);
    if (s < e.S) ((double2 *)e.tmp)[s] = make_double2(tx, ty);
    if (e.lane == 0) ((unsigned *)e.scratch)[base >> 5] = mv & ~rot;
    mv &= rot;
    while (mv) {
      const int src = __ffs(mv) - 1;
      mv &= mv - 1;
      const int s2 = base + src;
      const int n = META(e, MOOG_M_NV, s2);
      double2 *v = e.vtx + e.voff[s2];
      const double ttx = shfl_d(tx, src), tty = shfl_d(ty, src);
      double x = 0.0, y = 0.0;
      if (e.lane < n) {
        double2 p = v[e.lane];
        // Affine2D().translate(tx, ty): 1.0 * x is exact, the 0.0 * y term keeps the
        // reference's NaN / signed-zero behaviour
        x = (p.x + 0.0 * p.y) + ttx;
        y = (0.0 * p.x + p.y) + tty;
      }
      const double r0 = shfl_d(m.m0, src), r1 = shfl_d(m.m1, src), r2 = shfl_d(m.m2, src);
      const double r3 = shfl_d(m.m3, src), r4 = shfl_d(m.m4, src), r5 = shfl_d(m.m5, src);
      const double rx = r0 * x + r1 * y + r2;
      const double ry = r3 * x + r4 * y + r5;
      if (e.lane < n) v[e.lane] = make_double2(rx, ry);
      if (n > 32) outline_tail(v, n, e.lane, ttx, tty, true, r0, r1, r2, r3, r4, r5);
    }
  }
  wsync();
  // phase 2b: every vertex of every slot that only translates, lane = cached vertex.  Which slot a
  // vertex belongs to is a constant of the program (vmap); the iterations are independent, so
  // their shared-memory round trips overlap instead of queueing behind one another slot by slot.
  if (e.vmap) {
    const unsigned *smask = (const unsigned *)e.scratch;
    const double2 *tt = (const double2 *)e.tmp;
    const uint8_t *vmap = e.vmap;
    const int *nvs = &META(e, MOOG_M_NV, 0);
    const int *voffs = e.voff;
    double2 *vtx = e.vtx;
    const int VT = e.VT, S = e.S;
    // four vertices per lane and trip, every load issued before the first use and no branch but
    // the stores' predicates: straight-line code whose shared-memory round trips overlap
#pragma unroll 1
    for (int v0 = e.lane; v0 < VT; v0 += 128) {
      unsigned u[4], sl[4], word[4];
      int nv[4], vo[4];
      bool ok[4];
      double2 p[4], t[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int v = v0 + 32 * q;
        ok[q] = v < VT;
        u[q] = vmap[ok[q] ? v : 0];
        p[q] = vtx[ok[q] ? v : 0];
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const unsigned raw = u[q];
        sl[q] = raw < (unsigned)S ? raw : 0u;
        ok[q] = ok[q] & (raw < (unsigned)S);
        word[q] = smask[sl[q] >> 5];
        nv[q] = nvs[sl[q]];
        vo[q] = voffs[sl[q]];
        t[q] = tt[sl[q]];
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        ok[q] = ok[q] & (((word[q] >> (sl[q] & 31u)) & 1u) != 0u) & (v0 + 32 * q - vo[q] < nv[q]);
        // Affine2D().translate(tx, ty): 1.0 * x is exact, the 0.0 * y term keeps the
        // reference's NaN / signed-zero behaviour
        const double2 o = make_double2((p[q].x + 0.0 * p[q].y) + t[q].x, (0.0 * p[q].x + p[q].y) + t[q].y);
        if (ok[q]) vtx[v0 + 32 * q] = o;
      }
    }
  }
  wsync();
#ifdef MOOG_PROFILE_INTEG
  const long long ti2 = clock64();
  ctr_add(e, CT_CYC_NARROW, ti2 - ti1);
#endif
  // phase 3: boxes of rotated outlines, NaN / inf classification (lane = slot)
  for (int s = e.lane; s < e.S; s += 32) {
    const int flag = e.sflag[s] >> 8;
    int low = e.sflag[s] & SLF_MASK;
    if (flag & (TF_ROT | TF_CLASSIFY)) {
      int n = META(e, MOOG_M_NV, s);
      const double2 *v = e.vtx + e.voff[s];
      double xmin = INFINITY, xmax = -INFINITY, ymin = INFINITY, ymax = -INFINITY;
      bool nonfinite = false, allnan = n > 0, steep = false;
      double px = n > 0 ? v[n - 1].x : 0.0;
#pragma unroll 1
      for (int i = 0; i < n; ++i) {
        double2 p = v[i];
        xmin = fmin(xmin, p.x); xmax = fmax(xmax, p.x);
        ymin = fmin(ymin, p.y); ymax = fmax(ymax, p.y);
        nonfinite |= !(isfinite(p.x) && isfinite(p.y));
        allnan &= isnan(p.x) && isnan(p.y);
        steep |= steep_edge(px, p.x);
        px = p.x;
      }
      if (flag & TF_CLASSIFY)
        low = (low & (SLF_SHORT_EDGE | SLF_STEEP)) | (nonfinite ? SLF_NONFINITE : 0) | (allnan ? SLF_ALLNAN : 0);
      low = (low & ~SLF_STEEP) | (steep ? SLF_STEEP : 0);
      store_box(e, s, xmin, ymin, xmax, ymax, (low & SLF_NONFINITE) != 0, steep);
    }
    e.sflag[s] = low;
  }
  wsync();
#ifdef MOOG_PROFILE_INTEG
  ctr_add(e, CT_CYC_RESOLVE, clock64() - ti2);
#endif
}

// out of line, with its own view of the env: the pass keeps its pointers in registers instead of
// sharing the register file with everything apply_physics inlines
__device__ __noinline__ void integrate_all_ol() {
  const Env e = env_view();
  integrate_all_impl(e);
}
__device__ __forceinline__ void integrate_all(const Env &) { integrate_all_ol(); }

// physics.py:88-117 Physics.apply_physics (one substep)
__device__ inline void apply_physics(const Env &e, int n_cmask_words) {
  const int32_t *h = e.hdr;
#ifdef MOOG_PROFILE_PHASES
  long long t0 = clock64();
#endif
  refresh_candidates(e, n_cmask_words);
#ifdef MOOG_PROFILE_PHASES
  long long t1 = clock64();
  ctr_add(e, CT_NARROW, t1 - t0);
#endif
  for (int f = 0; f < h[MOOG_H_N_FORCES]; ++f) {
    const moog_op *op = e.ops + h[MOOG_H_FORCES] + f;
    int la = op->i[0], lb = op->i[1];
    if (op->kind == MOOG_F_MAZE_WALK) {
      maze_walk_layer(e, op);
    } else if (lb < 0) {
      force_unary_layer(e, op);
    } else if (op->kind == MOOG_F_COLLISION) {
      collision_op(e, op, f, n_cmask_words);
    } else {
      for (int i = 0; i < e.cnt[la]; ++i)
        for (int j = 0; j < e.cnt[lb]; ++j) force_binary(e, op, LOFF(e, la) + i, LOFF(e, lb) + j);
    }
  }
  for (int c = 0; c < h[MOOG_H_N_CORR]; ++c) corrective(e, e.ops + h[MOOG_H_CORR] + c);
#ifdef MOOG_PROFILE_PHASES
  long long t2 = clock64();
  ctr_add(e, CT_CYC_NARROW, t2 - t1);
#endif
  integrate_all(e);
#ifdef MOOG_PROFILE_PHASES
  ctr_add(e, CT_CYC_RESOLVE, clock64() - t2);
#endif
}

// sprite.py:411-424 Sprite._set_path, what the `scale` / `aspect_ratio` setters (:546-558) call:
// the outline is re-derived from the COM-centred shape (shape record of the blob) by
//   Affine2D().scale(s, s * aspect) + Affine2D().rotate(angle) + Affine2D().translate(*position)
// (two 3x3 numpy products, then x' = m00 x + m01 y + m02 unfused), the circumscribed radius is
// re-measured and the rotational inertia multiplied by the squared scales -- again on every call:
// the reference's inertia compounds.  Lane = vertex; box and flags of the slot are rebuilt.
__device__ __noinline__ void set_path(const Env &, int s) {
  const Env e = env_view();
  const int32_t *shape_off = e.ipool + e.hdr[MOOG_H_SHAPE_TAB];
  const double *R = e.dpool + shape_off[META(e, MOOG_M_SHAPE, s)];
  const int nv = (int)R[0];
  const double sx = STAT(e, MOOG_S_SCALE, s), sy = STAT(e, MOOG_S_SCALE, s) * STAT(e, MOOG_S_ASPECT, s);
  const double px = DYN(e, MOOG_D_X, s), py = DYN(e, MOOG_D_Y, s);
  Aff S = {1.0 * sx, 0.0 * sx, 0.0 * sx, 0.0 * sy, 1.0 * sy, 0.0 * sy};
  Aff Rm = aff_identity();
  aff_rotate(Rm, DYN(e, MOOG_D_ANG, s));
  Aff T = aff_identity();
  aff_translate(T, px, py);
  const Aff M = aff_then(aff_then(S, Rm), T);
  double2 *v = e.vtx + e.voff[s];
  wsync();
  double r = -INFINITY;
  bool rnan = false;
  double xmin = INFINITY, xmax = -INFINITY, ymin = INFINITY, ymax = -INFINITY;
  bool fin = true, nan_all = true;
  for (int i = e.lane; i < nv; i += 32) {
    const double bx = R[6 + 2 * i], by = R[7 + 2 * i];
    const double2 q = make_double2(M.m0 * bx + M.m1 * by + M.m2, M.m3 * bx + M.m4 * by + M.m5);
    v[i] = q;
    const double d = norm_ax(q.x - px, q.y - py);
    rnan |= isnan(d);
    r = fmax(r, d);
    fin &= isfinite(q.x) && isfinite(q.y);
    nan_all &= isnan(q.x) && isnan(q.y);
    xmin = fmin(xmin, q.x); xmax = fmax(xmax, q.x);
    ymin = fmin(ymin, q.y); ymax = fmax(ymax, q.y);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    r = fmax(r, shflx_d(r, o));
    xmin = fmin(xmin, shflx_d(xmin, o)); xmax = fmax(xmax, shflx_d(xmax, o));
    ymin = fmin(ymin, shflx_d(ymin, o)); ymax = fmax(ymax, shflx_d(ymax, o));
  }
  if (__any_sync(FULL, rnan)) r = NAN;  // np.max propagates a NaN
  const bool nonfinite = !__all_sync(FULL, fin);
  const bool allnan = nv > 0 && __all_sync(FULL, nan_all);
  wsync();
  bool st = false, sh = nv < 3;
  for (int i = e.lane; i < nv; i += 32) {
    const double2 p = v[i], q = v[(i + 1 == nv) ? 0 : i + 1];
    st |= steep_edge(p.x, q.x);
    sh |= !((q.x - p.x) * (q.x - p.x) + (q.y - p.y) * (q.y - p.y) > SHORT_EDGE2);
  }
  const bool steep = __any_sync(FULL, st) != 0, shortedge = __any_sync(FULL, sh) != 0;
  if (e.lane == 0) {
    META(e, MOOG_M_NV, s) = nv;
    STAT(e, MOOG_S_MAXR, s) = r;
    STAT(e, MOOG_S_IX, s) = STAT(e, MOOG_S_IX, s) * (sx * sx);
    STAT(e, MOOG_S_IY, s) = STAT(e, MOOG_S_IY, s) * (sy * sy);
    e.sflag[s] = (shortedge ? SLF_SHORT_EDGE : 0) | (nonfinite ? SLF_NONFINITE : 0) | (allnan ? SLF_ALLNAN : 0) |
                 (steep ? SLF_STEEP : 0);
    store_box(e, s, xmin, ymin, xmax, ymax, nonfinite, steep);
  }
  wsync();
}

// ---------------------------------------------------------------------------
// expression VM (config lambdas compiled by the host)
// ---------------------------------------------------------------------------
__device__ inline double *attr_ptr(const Env &e, int s, int at) {
  if (at >= MOOG_AT_META0) return &e.envf[e.hdr[MOOG_H_META_OFF] + (at - MOOG_AT_META0) * e.S + s];
  switch (at) {
    case MOOG_AT_X: return &DYN(e, MOOG_D_X, s);
    case MOOG_AT_Y: return &DYN(e, MOOG_D_Y, s);
    case MOOG_AT_X_VEL: return &DYN(e, MOOG_D_VX, s);
    case MOOG_AT_Y_VEL: return &DYN(e, MOOG_D_VY, s);
    case MOOG_AT_ANGLE: return &DYN(e, MOOG_D_ANG, s);
    case MOOG_AT_ANGLE_VEL: return &DYN(e, MOOG_D_ANGVEL, s);
    case MOOG_AT_MASS: return &STAT(e, MOOG_S_MASS, s);
    case MOOG_AT_SCALE: return &STAT(e, MOOG_S_SCALE, s);
    case MOOG_AT_ASPECT_RATIO: return &STAT(e, MOOG_S_ASPECT, s);
    case MOOG_AT_C0: return &STAT(e, MOOG_S_C0, s);
    case MOOG_AT_C1: return &STAT(e, MOOG_S_C1, s);
    case MOOG_AT_C2: return &STAT(e, MOOG_S_C2, s);
    case MOOG_AT_OPACITY: return &STAT(e, MOOG_S_OPACITY, s);
  }
  return &DYN(e, MOOG_D_X, s);
}

__device__ inline double py_fmod(double a, double b) {
  double r = fmod(a, b);
  if (r != 0) {
    if ((r < 0) != (b < 0)) r += b;
  } else {
    r = copysign(0.0, b);  // CPython float_rem / numpy remainder
  }
  return r;
}

__device__ double rule_noise_at(const Env &e, int col);
__device__ __noinline__ double eval_expr(const Env &, int start, int s0, int s1) {
  const Env e = env_view();
  if (start < 0) return 1.0;
  double st[16];
  int sp = 0;
  for (const moog_ex *x = e.expr + start; x->op != MOOG_X_END; ++x) {
    double a, b;
    switch (x->op) {
      case MOOG_X_CONST: st[sp++] = x->c; break;
      case MOOG_X_ATTR0: st[sp++] = *attr_ptr(e, s0, x->arg); break;
      case MOOG_X_ATTR1: st[sp++] = *attr_ptr(e, s1, x->arg); break;
      case MOOG_X_NOT: st[sp - 1] = !(st[sp - 1] != 0); break;
      case MOOG_X_NEG: st[sp - 1] = -st[sp - 1]; break;
      case MOOG_X_ABS: st[sp - 1] = fabs(st[sp - 1]); break;
      case MOOG_X_STORE_POS: {
        const double ny = st[--sp], nx = st[--sp];
        set_position(e, s0, nx, ny);
        break;
      }
      case MOOG_X_STORE: {
        double v = st[--sp];
        if (x->arg == MOOG_AT_ANGLE) {  // sprite.py:531-540; x->c: NumPy kind of the assigned value
          // (c = 4: computed from the sprite's own angle and python floats only -- the NumPy kind it has stays)
          set_angle_f64(e, s0, v, x->c == 4.0 ? ((META(e, MOOG_M_FLAGS, s0) >> MOOG_SF_ANG_SHIFT) & 3) : (int)x->c);
          break;
        }
        wsync();
        put(e, attr_ptr(e, s0, x->arg), v);
        wsync();
        if (x->arg == MOOG_AT_SCALE || x->arg == MOOG_AT_ASPECT_RATIO) set_path(e, s0);
        // sprite.py:639-643: the velocity setter installs a fresh array; x->c = 3: a float64 one
        if ((x->arg == MOOG_AT_X_VEL || x->arg == MOOG_AT_Y_VEL) && x->c == 3.0) {
          const int fl = META(e, MOOG_M_FLAGS, s0) & ~(MOOG_SF_VEL32 | (MOOG_SF_VALIAS_MASK << MOOG_SF_VALIAS_SHIFT));
          wsync();
          puti(e, &META(e, MOOG_M_FLAGS, s0), fl);
          wsync();
        }
        break;
      }
      case MOOG_X_RULE_NOISE: st[sp++] = rule_noise_at(e, x->arg); break;  // a draw of a traced rule
      case MOOG_X_NORM2: {  // np.linalg.norm of a 2-vector
        const double vy = st[--sp], vx = st[--sp];
        st[sp++] = norm1(vx, vy);
        break;
      }
      case MOOG_X_ENVF: st[sp++] = e.envf[x->arg]; break;  // a user-defined rule's own attribute
      case MOOG_X_STORE_ENVF: {
        const double v = st[--sp];
        wsync();
        put(e, &e.envf[x->arg], v);
        wsync();
        break;
      }
      case MOOG_X_SELECT: {  // c ? a : b
        const double vb = st[--sp], va = st[--sp], vc = st[--sp];
        st[sp++] = vc != 0 ? va : vb;
        break;
      }
      default:
        b = st[--sp];
        a = st[--sp];
        switch (x->op) {
          case MOOG_X_LT: a = a < b; break;
          case MOOG_X_LE: a = a <= b; break;
          case MOOG_X_GT: a = a > b; break;
          case MOOG_X_GE: a = a >= b; break;
          case MOOG_X_EQ: a = a == b; break;
          case MOOG_X_NE: a = a != b; break;
          case MOOG_X_AND: a = (a != 0) && (b != 0); break;
          case MOOG_X_OR: a = (a != 0) || (b != 0); break;
          case MOOG_X_ADD: a = a + b; break;
          case MOOG_X_SUB: a = a - b; break;
          case MOOG_X_MUL: a = a * b; break;
          case MOOG_X_DIV: a = a / b; break;
          case MOOG_X_MOD: a = py_fmod(a, b); break;
        }
        st[sp++] = a;
    }
  }
  return sp ? st[sp - 1] : 1.0;
}

// A decision tree of lambdas.state_tree / lambdas.trace_rule (MOOG_SC_TREE, MOOG_R_TREE), walked lazily from
// node 0: the tests made -- overlap calls included -- are the ones Python would make, in its order.  Node: kind,
// expr, layer / index of sprite 0, layer / index of sprite 1, next if true, next if false.  A sprite index
// beyond its layer's count is the reference's IndexError (MOOG_ERR_BAD_INDEX).
__device__ __noinline__ double walk_tree(const Env &, const int32_t *nodes, int n) {
  const Env e = env_view();
  int j = 0;
  for (int guard = 0; guard <= n; ++guard) {
    const int32_t *nd = nodes + 8 * j;
    if (nd[0] == 3) {  // index < len(state[layer])
      j = nd[3] < e.cnt[nd[2]] ? nd[6] : nd[7];
      continue;
    }
    int sl[2] = {0, 0};
    for (int q = 0; q < 2; ++q) {
      const int l = nd[2 + 2 * q], k = nd[3 + 2 * q];
      if (l < 0) continue;
      if (k >= e.cnt[l]) {
        const int err = e.envi[MOOG_EI_ERR] | MOOG_ERR_BAD_INDEX;
        wsync();
        puti(e, &e.envi[MOOG_EI_ERR], err);
        wsync();
        return 0;
      }
      sl[q] = LOFF(e, l) + k;
    }
    if (nd[0] == 0) return nd[1] >= 0 ? eval_expr(e, nd[1], sl[0], sl[1]) : 0.0;  // leaf: the value / end of the rule
    if (nd[0] == 4) {  // the assignments this path made
      eval_expr(e, nd[1], sl[0], sl[1]);
      j = nd[6];
      continue;
    }
    const bool yes = nd[0] == 2 ? overlaps(e, sl[0], sl[1]) : eval_expr(e, nd[1], sl[0], sl[1]) != 0;
    j = yes ? nd[6] : nd[7];
  }
  return 0;
}

// The step's uniform of one rule-noise column: supplied by the caller (io.rule_noise), else drawn from the
// Philox stream keyed by (seed, env, number of rules_step passes so far, episode, column)
__device__ double rule_noise_at(const Env &e, int col) {
  if (e.rule_noise) return e.rule_noise[col];
  return philox_uniform(e.seed ^ 0x9E3779B97F4A7C15ull, (uint32_t)e.env_id, (uint32_t)e.envi[MOOG_EI_RULE_PASSES],
                        (uint32_t)e.envi[MOOG_EI_EPISODES], (uint32_t)col);
}

__device__ __noinline__ double eval_condition_leaf(const Env &, int op_index) {
  const Env e = env_view();
  const moog_op *op = e.ops + op_index;
  switch (op->kind) {
    case MOOG_SC_CONST: return op->p[0];
    case MOOG_SC_BERNOULLI: return rule_noise_at(e, op->i[0]) < op->p[0];  // np.random.binomial(1, p)
    case MOOG_SC_TREE: return walk_tree(e, e.ipool + op->i[0], op->i[1]);
    case MOOG_SC_ALL:
    case MOOG_SC_ANY:
    case MOOG_SC_COUNT: {
      int n = list_count(e, op->i[0], op->i[1]);
      int cnt = 0;
      for (int i = 0; i < n; ++i) {
        int s = list_slot(e, op->i[0], op->i[1], i);
        cnt += eval_expr(e, op->i[2], s, s) != 0;
      }
      if (op->kind == MOOG_SC_ALL) return cnt == n;
      if (op->kind == MOOG_SC_ANY) return cnt > 0;
      return cnt;
    }
    case MOOG_SC_FIRST: {
      const int n = list_count(e, op->i[0], op->i[1]);
      return n > 0 ? eval_expr(e, op->i[2], list_slot(e, op->i[0], op->i[1], 0), list_slot(e, op->i[0], op->i[1], 0)) : 0.0;
    }
    case MOOG_SC_CONTACT_COUNT: {  // contact_rules.py:15-51
      int la = op->i[0], lb = op->i[1], cnt = 0;
      for (int i = 0; i < e.cnt[la]; ++i)
        for (int j = 0; j < e.cnt[lb]; ++j) cnt += overlaps(e, LOFF(e, la) + i, LOFF(e, lb) + j);
      return cnt;
    }
    case MOOG_SC_CONTACT_ANY_COUNT: {
      int n = list_count(e, op->i[0], op->i[1]);
      int m = list_count(e, op->i[2], op->i[3]);
      int cnt = 0;
      for (int i = 0; i < n; ++i) {
        int s = list_slot(e, op->i[0], op->i[1], i);
        if (eval_expr(e, op->i[4], s, s) == 0) continue;
        bool any = false;
        for (int j = 0; j < m && !any; ++j) any = overlaps(e, s, list_slot(e, op->i[2], op->i[3], j));
        cnt += any;
      }
      return cnt;
    }
  }
  return 0;
}


// MOOG_SC_BINARY / MOOG_SC_NOT nodes over the leaves above, evaluated with an explicit
// stack (no device recursion); the compiler bounds the nesting at MOOG_MAX_SC_DEPTH
#define MOOG_MAX_SC_DEPTH 8
__device__ __noinline__ double eval_condition(const Env &, int op_index) {
  const Env e = env_view();
  int idx[MOOG_MAX_SC_DEPTH], stage[MOOG_MAX_SC_DEPTH];
  double lhs[MOOG_MAX_SC_DEPTH];
  int sp = 1;
  double ret = 0.0;
  idx[0] = op_index;
  stage[0] = 0;
  while (sp > 0) {
    const moog_op *op = e.ops + idx[sp - 1];
    const int st = stage[sp - 1];
    if (op->kind == MOOG_SC_NOT) {
      if (st == 0 && sp < MOOG_MAX_SC_DEPTH) {
        stage[sp - 1] = 1;
        idx[sp] = op->i[0]; stage[sp] = 0; ++sp;
      } else {
        ret = !(ret != 0);
        --sp;
      }
    } else if (op->kind == MOOG_SC_BINARY) {
      const int x = op->i[2];
      if (st == 0 && sp < MOOG_MAX_SC_DEPTH) {
        stage[sp - 1] = 1;
        idx[sp] = op->i[0]; stage[sp] = 0; ++sp;
      } else if (st == 1) {
        const double a = ret;
        if ((x == MOOG_X_AND && !(a != 0)) || (x == MOOG_X_OR && a != 0)) {
          --sp;  // python and / or: the deciding operand is the value
        } else {
          lhs[sp - 1] = a;
          stage[sp - 1] = 2;
          idx[sp] = op->i[1]; stage[sp] = 0; ++sp;
        }
      } else {
        const double a = lhs[sp - 1], b = ret;
        switch (x) {
          case MOOG_X_LT: ret = a < b; break;
          case MOOG_X_LE: ret = a <= b; break;
          case MOOG_X_GT: ret = a > b; break;
          case MOOG_X_GE: ret = a >= b; break;
          case MOOG_X_EQ: ret = a == b; break;
          case MOOG_X_NE: ret = a != b; break;
          case MOOG_X_ADD: ret = a + b; break;
          case MOOG_X_SUB: ret = a - b; break;
          case MOOG_X_MUL: ret = a * b; break;
          default: ret = b; break;  // and / or: the right operand decided
        }
        --sp;
      }
    } else {
      ret = eval_condition_leaf(e, idx[sp - 1]);
      --sp;
    }
  }
  return ret;
}

// ---------------------------------------------------------------------------
// rules
// ---------------------------------------------------------------------------
__device__ inline void copy_slot(const Env &e, int dst, int src) {
  wsync();
  int nv = META(e, MOOG_M_NV, src);
  if (e.lane < MOOG_DYN_FIELDS) DYN(e, e.lane, dst) = DYN(e, e.lane, src);
  if (e.lane < MOOG_STAT_FIELDS) STAT(e, e.lane, dst) = STAT(e, e.lane, src);
  if (e.lane < MOOG_META_FIELDS) META(e, e.lane, dst) = META(e, e.lane, src);
  if (e.lane < 4) BOX(e, e.lane, dst) = BOX(e, e.lane, src);
  if (e.lane == 0) e.sflag[dst] = e.sflag[src];
  if (e.lane < e.hdr[MOOG_H_N_META]) {  // the sprite's metadata columns travel with it
    double *m = e.envf + e.hdr[MOOG_H_META_OFF] + e.lane * e.S;
    m[dst] = m[src];
  }
  for (int i = e.lane; i < nv; i += 32) e.vtx[e.voff[dst] + i] = e.vtx[e.voff[src] + i];
  wsync();
}

// vanish.py:31-39: pop the flagged sprites of layer l, preserving order.
// `gone` is a per-lane bitmask chunk list: bit i of word w flags sprite 32*w+i.
__device__ inline void vanish(const Env &e, int l, const unsigned *gone) {
  int base = LOFF(e, l), n = e.cnt[l], w = 0;
  for (int i = 0; i < n; ++i) {
    if ((gone[i >> 5] >> (i & 31)) & 1u) continue;
    if (w != i) copy_slot(e, base + w, base + i);
    ++w;
  }
  wsync();
  puti(e, &e.cnt[l], w);
  wsync();
}

// ---------------------------------------------------------------------------
// Device-side reset sampler (SURVEY section 8 f1): one generate_sprites group
// (state_initialization/sprite_generators.py:26-105) for this env.  Factors are drawn from
// the Philox stream keyed by (seed, env, episode, slot, try, factor); the sprite is built
// like Sprite.__init__ does on the host (sprite.py:261-424: centroid-centred outline scaled
// by (scale, scale * aspect_ratio), rotated, translated; position += raw centroid;
// circumscribed radius; inertia * scale^2) and redrawn while it overlaps a sprite it must avoid.
// ---------------------------------------------------------------------------
// one factor from a leaf sampler (MOOG_ZK_*): a constant, np.float32(rng.uniform(lo, hi)), or one of n values
__device__ __forceinline__ double sample_leaf(const double *dpool, int kind, int idx, int n, double u) {
  if (kind == MOOG_ZK_CONST) return dpool[idx];
  if (kind == MOOG_ZK_UNIFORM32) return (double)(float)(dpool[idx] + (dpool[idx + 1] - dpool[idx]) * u);
  if (kind == MOOG_ZK_DISCRETE_P) {  /* rng.choice(n, p=probs): the first candidate whose cumulative probability exceeds u */
    int k = 0;
    while (k < n - 1 && !(u < dpool[idx + n + k])) ++k;
    return dpool[idx + k];
  }
  const int pick = (int)(u * n);
  return dpool[idx + (pick < n ? pick : n - 1)];
}

// A DependentDistribution's expression (distributions.py:420-470) over the factors drawn so far:
// the arithmetic subset of the expression VM, X_ATTR0 reading factor `arg` of the sample
__device__ inline double eval_factor_expr(const moog_ex *x, const double *v) {
  double st[16];
  int sp = 0;
  for (; x->op != MOOG_X_END && sp < 15; ++x) {
    double a, b;
    switch (x->op) {
      case MOOG_X_CONST: st[sp++] = x->c; break;
      case MOOG_X_ATTR0: st[sp++] = v[x->arg]; break;
      case MOOG_X_NOT: st[sp - 1] = !(st[sp - 1] != 0); break;
      case MOOG_X_NEG: st[sp - 1] = -st[sp - 1]; break;
      case MOOG_X_ABS: st[sp - 1] = fabs(st[sp - 1]); break;
      default:
        if (sp < 2) return NAN;
        b = st[--sp];
        a = st[--sp];
        switch (x->op) {
          case MOOG_X_LT: a = a < b; break;
          case MOOG_X_LE: a = a <= b; break;
          case MOOG_X_GT: a = a > b; break;
          case MOOG_X_GE: a = a >= b; break;
          case MOOG_X_EQ: a = a == b; break;
          case MOOG_X_NE: a = a != b; break;
          case MOOG_X_AND: a = (a != 0) && (b != 0); break;
          case MOOG_X_OR: a = (a != 0) || (b != 0); break;
          case MOOG_X_ADD: a = a + b; break;
          case MOOG_X_SUB: a = a - b; break;
          case MOOG_X_MUL: a = a * b; break;
          case MOOG_X_DIV: a = a / b; break;
          default: a = NAN; break;
        }
        st[sp++] = a;
    }
  }
  return sp ? st[sp - 1] : NAN;
}

// One generate_sprites call.  op: a MOOG_Z_GENERATE (reset) or MOOG_R_CREATE_SPRITES (rule) op -- both carry
// the sampler table in i[4], the dtype flags in i[5] and max_recursion_depth in p[0].  The `count`
// sprites go to slots first.. of `layer`; they must not overlap the slots avoid[0..n_avoid)
// (avoid_layers = 0) or the sprites that the LAYERS avoid[..] held when the call began
// (avoid_layers = 1: create_sprites.py:31-33).  Draws: Philox(key; env, c1, slot << 20 | try, tag | factor).
__device__ __noinline__ void generate_sprites_dev(const Env &, const moog_op *op, uint64_t key, uint32_t c1, int layer,
                                                  int first, int count, const int32_t *avoid, int n_avoid,
                                                  int avoid_layers) {
  const Env e = env_view();
  const double *dpool = e.dpool;
  const int32_t *shape_off = e.ipool + e.hdr[MOOG_H_SHAPE_TAB];
  const int32_t *tab = e.ipool + op->i[4];
  const int max_depth = (int)fmin(op->p[0], 1048575.0);
  const uint32_t episode = c1;
  int placed = 0;
  for (int k = 0; k < count; ++k) {
    const int s = first + k;
    bool stop = false;
    for (int tries = 0;; ++tries) {
      double v[MOOG_Z_N_ATTRS];
#pragma unroll 1
      for (int a = 0; a < MOOG_Z_N_ATTRS; ++a) {
        const int kind = tab[3 * a], idx = tab[3 * a + 1], n = tab[3 * a + 2];
        const double u = kind == MOOG_ZK_CONST ? 0.0
                                               : philox_uniform(key, (uint32_t)e.env_id, episode,
                                                                ((uint32_t)s << 20) | (uint32_t)tries, (0x5Au << 24) | (uint32_t)a);
        v[a] = sample_leaf(dpool, kind, idx, n, u);
      }
      {
        // extension components of the factor distribution (distributions.py: Mixture picks one
        // alternative; SetMinus / Selection redraw their base until it is outside / inside a box)
        const int32_t *x = tab + 3 * MOOG_Z_N_ATTRS;
        const int n_ext = *x++;
        uint32_t draw = 0;
        for (int c = 0; c < n_ext; ++c) {
          const int kind = *x++;
          if (kind == 3) {  // DependentDistribution: attr, expression, float32?
            const int n_dep = *x++;
            for (int q = 0; q < n_dep; ++q, x += 3) {
              const double val = eval_factor_expr(e.expr + x[1], v);
              v[x[0]] = x[2] ? (double)(float)val : val;
            }
          } else if (kind == 1) {
            const int n_alt = *x++;
            const double *cum = dpool + *x++;
            const double u = philox_uniform(key, (uint32_t)e.env_id, episode,
                                            ((uint32_t)s << 20) | (uint32_t)tries, (0x5Bu << 24) | (draw++ & 0xffffffu));
            int pick = 0;
            while (pick < n_alt - 1 && !(u < cum[pick])) ++pick;   // rng.choice(n, p=probs)
            for (int a = 0; a < n_alt; ++a) {
              const int n_leaves = *x++;
              for (int q = 0; q < n_leaves; ++q, x += 4) {
                if (a != pick) continue;
                const double uu = philox_uniform(key, (uint32_t)e.env_id, episode,
                                                 ((uint32_t)s << 20) | (uint32_t)tries, (0x5Bu << 24) | (draw++ & 0xffffffu));
                v[x[0]] = sample_leaf(dpool, x[1], x[2], x[3], uu);
              }
            }
          } else {
            const int keep_inside = *x++;
            const int n_leaves = *x++;
            const int32_t *leaves = x;
            x += 4 * n_leaves;
            const int n_box = *x++;
            const int32_t *box = x;
            x += 2 * n_box;
            // distributions.py:341-349, 394-404: redraw the base until it is outside / inside the box,
            // at most _MAX_TRIES = 1e5 times, then raise
            bool accepted = false;
            for (int inner = 0; inner < 100000 && !accepted; ++inner) {
              for (int q = 0; q < n_leaves; ++q) {
                const double uu = philox_uniform(key, (uint32_t)e.env_id, episode,
                                                 ((uint32_t)s << 20) | (uint32_t)tries, (0x5Bu << 24) | (draw++ & 0xffffffu));
                v[leaves[4 * q]] = sample_leaf(dpool, leaves[4 * q + 1], leaves[4 * q + 2], leaves[4 * q + 3], uu);
              }
              bool inside = true;
              for (int q = 0; q < n_box; ++q) {
                const double val = v[box[2 * q]], lo = dpool[box[2 * q + 1]], hi = dpool[box[2 * q + 1] + 1];
                inside = inside && val >= lo && val < hi;   // Continuous.contains
              }
              accepted = inside == (keep_inside != 0);
            }
            if (!accepted) {  // the reference raises ValueError here; the env carries the error bit
              const int err = e.envi[MOOG_EI_ERR] | MOOG_ERR_RESET_REJECTED;
              wsync();
              puti(e, &e.envi[MOOG_EI_ERR], err);
              wsync();
            }
          }
        }
      }
      // Sprite.__init__ (sprite.py:261-327) then the shape setter (:329-409): the outline is laid out at
      // (x, y) by _set_path (:411-424: circumscribed radius, inertia * scale^2), THEN the position setter
      // (:616-633) moves sprite and cached outline by the shape's raw centroid
      const double *R = dpool + shape_off[(int)v[MOOG_Z_SHAPE_ATTR]];
      wsync();
      if (e.lane == 0) {
        DYN(e, MOOG_D_X, s) = v[MOOG_AT_X]; DYN(e, MOOG_D_Y, s) = v[MOOG_AT_Y];
        DYN(e, MOOG_D_VX, s) = v[MOOG_AT_X_VEL]; DYN(e, MOOG_D_VY, s) = v[MOOG_AT_Y_VEL];
        DYN(e, MOOG_D_ANG, s) = v[MOOG_AT_ANGLE]; DYN(e, MOOG_D_ANGVEL, s) = v[MOOG_AT_ANGLE_VEL];
        STAT(e, MOOG_S_MASS, s) = v[MOOG_AT_MASS]; STAT(e, MOOG_S_SCALE, s) = v[MOOG_AT_SCALE];
        STAT(e, MOOG_S_ASPECT, s) = v[MOOG_AT_ASPECT_RATIO];
        STAT(e, MOOG_S_IX, s) = R[2]; STAT(e, MOOG_S_IY, s) = R[3];
        STAT(e, MOOG_S_C0, s) = v[MOOG_AT_C0]; STAT(e, MOOG_S_C1, s) = v[MOOG_AT_C1];
        STAT(e, MOOG_S_C2, s) = v[MOOG_AT_C2]; STAT(e, MOOG_S_OPACITY, s) = v[MOOG_AT_OPACITY];
        META(e, MOOG_M_SHAPE, s) = (int)v[MOOG_Z_SHAPE_ATTR];
        META(e, MOOG_M_FLAGS, s) = op->i[5] | (R[1] != 0.0 ? MOOG_SF_CIRCLE : 0);
        META(e, MOOG_M_NV, s) = (int)R[0];
        e.cnt[layer] = s - LOFF(e, layer) + 1;
        for (int m = 0; m < e.hdr[MOOG_H_N_META]; ++m)  // a new sprite's metadata is {}
          e.envf[e.hdr[MOOG_H_META_OFF] + m * e.S + s] = NAN;
      }
      wsync();
      set_path(e, s);
      set_position(e, s, v[MOOG_AT_X] + R[4], v[MOOG_AT_Y] + R[5]);
      wsync();
      refresh_all_boxes(e);
      bool hit = false;
      if (avoid_layers) {
        for (int q = 0; q < n_avoid; ++q) {
          const int la = avoid[q], n_la = la == layer ? first - LOFF(e, la) : e.cnt[la];
          for (int j = 0; j < n_la; ++j) hit |= overlaps(e, s, LOFF(e, la) + j);
        }
      } else {
        for (int q = 0; q < n_avoid; ++q) hit |= overlaps(e, s, avoid[q]);  // every pair is evaluated
      }
      if (op->flags & MOOG_FL_DISJOINT)
        for (int j = first; j < s; ++j) hit |= overlaps(e, s, j);
      if (!hit) break;
      if (tries > max_depth) {  // sprite_generators.py:92-98
        if (op->flags & MOOG_FL_FAIL_GRACEFULLY) {
          stop = true;
        } else {
          const int err = e.envi[MOOG_EI_ERR] | MOOG_ERR_RESET_REJECTED;
          wsync();
          puti(e, &e.envi[MOOG_EI_ERR], err);
          wsync();
        }
        break;
      }
    }
    if (stop) break;
    placed = k + 1;
  }
  wsync();
  puti(e, &e.cnt[layer], first - LOFF(e, layer) + placed);
  wsync();
}

// sprite_generators.py:26-105 at a reset: the group's slots are fixed by the traced initializer
__device__ inline void reset_generate(const Env &e, const moog_op *op, uint64_t seed) {
  const int first = op->i[0];
  int count = op->i[1];
  if (op->p[2] > op->p[1]) {  // num_sprites = np.random.randint(p1, p2): drawn per env and episode
    const double u = philox_uniform(seed ^ 0x6A09E667F3BCC908ull, (uint32_t)e.env_id, (uint32_t)e.envi[MOOG_EI_EPISODES],
                                    ((uint32_t)first << 20) | 0xfffffu, (0x5Cu << 24));
    const int lo = (int)op->p[1], hi = (int)op->p[2];
    int c = lo + (int)(u * (double)(hi - lo));
    if (c >= hi) c = hi - 1;
    if (c < count) count = c < 0 ? 0 : c;
  }
  int layer = 0;
  for (int l = 0; l < e.L; ++l)
    if (first >= LOFF(e, l) && first < LOFF(e, l + 1)) layer = l;
  generate_sprites_dev(e, op, seed ^ 0x6A09E667F3BCC908ull, (uint32_t)e.envi[MOOG_EI_EPISODES], layer, first, count,
                       e.ipool + op->i[2], op->i[3], 0);
}

// one non-conditional rule
__device__ __noinline__ void rule_leaf(const Env &, int r) {
  const Env e = env_view();
  const moog_op *op = e.ops + r;
  unsigned flag[MOOG_MAX_SLOTS / 32];
  switch (op->kind) {
    case MOOG_R_KEEP_NEAR_CENTER: {  // re_center.py:60-76
      const int la = op->i[0];
      if (e.cnt[la] < 1) return;
      const int a = LOFF(e, la);
      const double px = DYN(e, MOOG_D_X, a) - 0.5, py = DYN(e, MOOG_D_Y, a) - 0.5;
      const double gx = op->p[0], gy = op->p[1];
      const double dx = -1. * gx * (double)(px > gx) + gx * (double)(px < -1. * gx);
      const double dy = -1. * gy * (double)(py > gy) + gy * (double)(py < -1. * gy);
      if (dx != 0 || dy != 0) {
        const int n = list_count(e, op->i[1], op->i[2]);
        for (int i = 0; i < n; ++i) {
          const int s = list_slot(e, op->i[1], op->i[2], i);
          set_position(e, s, DYN(e, MOOG_D_X, s) + dx, DYN(e, MOOG_D_Y, s) + dy);
        }
      }
      return;
    }
    case MOOG_R_PORTAL: {  // portal.py:41-76
      const int la = op->i[0], lp = op->i[1], np_ = e.cnt[lp];
      if (np_ & 1) {
        const int err = e.envi[MOOG_EI_ERR] | MOOG_ERR_PORTAL_ODD;
        wsync();
        puti(e, &e.envi[MOOG_EI_ERR], err);
        wsync();
        return;
      }
      for (int i = 0; i < e.cnt[la]; ++i) {
        const int s = LOFF(e, la) + i;
        const double px = DYN(e, MOOG_D_X, s), py = DYN(e, MOOG_D_Y, s);
        int first = -1;
        for (int q = 0; q < np_; ++q) {  // in_portals: every portal is asked (sprite.py:432-440)
          const int p = LOFF(e, lp) + q;
          bool in;
          if (is_symmetric_circle(e, p))
            in = norm1(px - DYN(e, MOOG_D_X, p), py - DYN(e, MOOG_D_Y, p)) < STAT(e, MOOG_S_MAXR, p);
          else
            in = point_in_poly(px, py, e.vtx + e.voff[p], META(e, MOOG_M_NV, p));
          if (in && first < 0) first = q;
        }
        const int fl = META(e, MOOG_M_FLAGS, s);
        wsync();
        if (first < 0) {
          puti(e, &META(e, MOOG_M_FLAGS, s), fl & ~MOOG_SF_TELEPORTING);
          wsync();
          continue;
        }
        if (fl & MOOG_SF_TELEPORTING) continue;
        const int ex = LOFF(e, lp) + ((first & 1) ? first - 1 : first + 1);
        set_position(e, s, DYN(e, MOOG_D_X, ex), DYN(e, MOOG_D_Y, ex));
        puti(e, &META(e, MOOG_M_FLAGS, s), fl | MOOG_SF_TELEPORTING);
        wsync();
      }
      return;
    }
    case MOOG_R_FIXATION: {  // fixation.py:45-54
      if (e.cnt[op->i[0]] < 1 || e.cnt[op->i[1]] < 1) {  // state[layer][0]: IndexError
        const int err = e.envi[MOOG_EI_ERR] | MOOG_ERR_BAD_INDEX;
        wsync();
        puti(e, &e.envi[MOOG_EI_ERR], err);
        wsync();
        return;
      }
      const int sa = LOFF(e, op->i[0]), st2 = LOFF(e, op->i[1]);
      const double dist = norm1(DYN(e, MOOG_D_X, sa) - DYN(e, MOOG_D_X, st2), DYN(e, MOOG_D_Y, sa) - DYN(e, MOOG_D_Y, st2));
      const double count = dist < op->p[0] ? e.envf[op->i[2]] + 1 : 0.0;
      wsync();
      put(e, &e.envf[op->i[2]], count);
      wsync();
      return;
    }
    case MOOG_R_PHASESEQ_BEGIN: {  // task_phases.py:126-141: the phase that is current when the pass begins is stepped
      const double now = e.envf[op->i[0]];
      wsync();
      put(e, &e.envf[op->i[0] + 1], now);
      wsync();
      return;
    }
    case MOOG_R_PHASE_END: {  // task_phases.py:90-95, 133-141
      const double count = e.envf[op->i[1] + 1] + 1;
      wsync();
      put(e, &e.envf[op->i[1] + 1], count);
      wsync();
      if (count >= e.envf[op->i[1] + 2] || (op->i[0] >= 0 && eval_condition(e, op->i[0]) != 0)) {
        wsync();
        put(e, &e.envf[op->i[1]], 1.0);
        if (op->i[2] >= 0) {
          const double next = e.envf[op->i[2]] + 1;
          const int ind = (int)next;
          put(e, &e.envf[op->i[2]], next);
          if (ind >= op->i[5])
            puti(e, &e.envi[MOOG_EI_ERR], e.envi[MOOG_EI_ERR] | MOOG_ERR_BAD_INDEX);  // self._phases[ind]: IndexError
          else if (op->i[3] >= 0)
            put(e, &e.envf[op->i[3]], e.dpool[op->i[4] + ind]);
        }
        wsync();
      }
      return;
    }
    case MOOG_R_TREE:  // a user-defined rule's step(), path by path
      walk_tree(e, e.ipool + op->i[0], op->i[1]);
      return;
    case MOOG_R_CREATE_SPRITES: {  // create_sprites.py:27-34
      const int layer = op->i[0], have = e.cnt[layer], cap = LOFF(e, layer + 1) - LOFF(e, layer);
      int count = op->i[1];
      if (op->p[2] > op->p[1]) {  // num_sprites = lambda: np.random.randint(p1, p2): drawn per call
        const int lo = (int)op->p[1], hi = (int)op->p[2];
        const int c = lo + (int)(rule_noise_at(e, (int)op->p[3]) * (double)(hi - lo));
        count = c >= hi ? hi - 1 : (c < 0 ? 0 : c);
      }
      const int serial = e.envi[MOOG_EI_CREATED];
      wsync();
      puti(e, &e.envi[MOOG_EI_CREATED], serial + 1);
      wsync();
      if (have + count > cap) {  // the reference's lists grow without bound; a layer of the record does not
        const int err = e.envi[MOOG_EI_ERR] | MOOG_ERR_LAYER_OVERFLOW;
        wsync();
        puti(e, &e.envi[MOOG_EI_ERR], err);
        wsync();
        count = cap - have;
      }
      generate_sprites_dev(e, op, e.seed ^ 0x3C6EF372FE94F82Bull, (uint32_t)serial, layer, LOFF(e, layer) + have, count,
                           e.ipool + op->i[2], op->i[3], 1);
      return;
    }
    case MOOG_R_CHANGE_LAYER: {  // change_layer.py:34-45
      const int lo = op->i[0], ln = op->i[1], n = e.cnt[lo];
      const int cap = LOFF(e, ln + 1) - LOFF(e, ln);
      for (int w = 0; w < MOOG_MAX_SLOTS / 32; ++w) flag[w] = 0;
      for (int i = 0; i < n; ++i)  // should_change is evaluated for every sprite before anything moves
        if (op->i[2] < 0 || eval_expr(e, op->i[2], LOFF(e, lo) + i, LOFF(e, lo) + i) != 0) flag[i >> 5] |= 1u << (i & 31);
      for (int i = 0; i < n; ++i) {
        if (!((flag[i >> 5] >> (i & 31)) & 1u)) continue;
        const int have = e.cnt[ln];
        if (have >= cap) {
          const int err = e.envi[MOOG_EI_ERR] | MOOG_ERR_LAYER_OVERFLOW;
          wsync();
          puti(e, &e.envi[MOOG_EI_ERR], err);
          wsync();
          flag[i >> 5] &= ~(1u << (i & 31));
          continue;
        }
        copy_slot(e, LOFF(e, ln) + have, LOFF(e, lo) + i);
        puti(e, &e.cnt[ln], have + 1);
        wsync();
      }
      vanish(e, lo, flag);
      return;
    }
    case MOOG_R_VANISH_ON_CONTACT: {  // vanish.py:66-86, contact_rules.py:28-35
      int la = op->i[0], lb = op->i[1];
      for (int w = 0; w < MOOG_MAX_SLOTS / 32; ++w) flag[w] = 0;
      for (int i = 0; i < e.cnt[la]; ++i)
        for (int j = 0; j < e.cnt[lb]; ++j)  // every pair is evaluated (no short-circuit)
          if (overlaps(e, LOFF(e, la) + i, LOFF(e, lb) + j)) flag[i >> 5] |= 1u << (i & 31);
      vanish(e, la, flag);
      return;
    }
    case MOOG_R_VANISH_BY_FILTER: {  // vanish.py:42-63
      int la = op->i[0];
      for (int w = 0; w < MOOG_MAX_SLOTS / 32; ++w) flag[w] = 0;
      for (int i = 0; i < e.cnt[la]; ++i)
        if (eval_expr(e, op->i[2], LOFF(e, la) + i, LOFF(e, la) + i) != 0) flag[i >> 5] |= 1u << (i & 31);
      vanish(e, la, flag);
      return;
    }
    case MOOG_R_MODIFY_ON_CONTACT: {  // contact_rules.py:86-120
      const int32_t *q = e.ipool + op->i[4];  // mod0 filt0 mod1 filt1
      for (int pass = 0; pass < 2; ++pass) {
        int as = pass ? op->i[2] : op->i[0], an = pass ? op->i[3] : op->i[1];
        int bs = pass ? op->i[0] : op->i[2], bn = pass ? op->i[1] : op->i[3];
        int na = list_count(e, as, an), nb = list_count(e, bs, bn);
        int mod = q[2 * pass], filt = q[2 * pass + 1];
        if (mod < 0) continue;
        for (int i = 0; i < na; ++i) {
          int sa = list_slot(e, as, an, i);
          if (eval_expr(e, filt, sa, sa) == 0) continue;
          bool any = false;
          for (int j = 0; j < nb; ++j) {
            int sb = list_slot(e, bs, bn, j);
            if (sb != sa && overlaps(e, sa, sb)) any = true;  // list comprehension: all evaluated
          }
          if (any) eval_expr(e, mod, sa, sa);
        }
      }
      return;
    }
    case MOOG_R_MODIFY_SPRITES: {  // modify_sprites.py:35-52
      int n = list_count(e, op->i[0], op->i[1]);
      // the filter sees the pre-modification state of every sprite (the reference
      // builds the filtered list first): flag, then modify
      int m = 0;
      for (int w = 0; w < MOOG_MAX_SLOTS / 32; ++w) flag[w] = 0;
      for (int i = 0; i < n; ++i) {
        int s = list_slot(e, op->i[0], op->i[1], i);
        if (op->i[3] < 0 || eval_expr(e, op->i[3], s, s) != 0) {
          flag[i >> 5] |= 1u << (i & 31);
          ++m;
        }
      }
      if (m == 0) return;
      int pick = -1;
      if (op->flags & MOOG_FL_SAMPLE_ONE) {
        double u = rule_noise_at(e, op->i[4]);
        pick = (int)(u * m);
        if (pick >= m) pick = m - 1;
      }
      int k = 0;
      for (int i = 0; i < n; ++i) {
        if (!((flag[i >> 5] >> (i & 31)) & 1u)) continue;
        int s = list_slot(e, op->i[0], op->i[1], i);
        if (pick < 0 || k == pick) eval_expr(e, op->i[2], s, s);
        ++k;
      }
      return;
    }
  }
}

// game_rules in order; ConditionalRule blocks (conditional.py:55-58) run their
// sub-rules `int(condition(state))` times.  Iterative (explicit block stack) so
// that the kernel's stack size is static.
#define MOOG_MAX_COND_DEPTH 4
__device__ __noinline__ void rules_step(const Env &) {
  const Env e = env_view();
  const int32_t *h = e.hdr;
  int r = h[MOOG_H_RULES];
  const int end = h[MOOG_H_RULES] + h[MOOG_H_N_RULES];
  int blk_start[MOOG_MAX_COND_DEPTH], blk_end[MOOG_MAX_COND_DEPTH], blk_left[MOOG_MAX_COND_DEPTH];
  int depth = 0;
  {
    const int passes = e.envi[MOOG_EI_RULE_PASSES] + 1;
    wsync();
    puti(e, &e.envi[MOOG_EI_RULE_PASSES], passes);
    wsync();
  }
  for (;;) {
    if (depth > 0 && r >= blk_end[depth - 1]) {
      if (--blk_left[depth - 1] > 0) {
        r = blk_start[depth - 1];
      } else {
        r = blk_end[depth - 1];
        --depth;
      }
      continue;
    }
    if (depth == 0 && r >= end) break;
    const moog_op *op = e.ops + r;
    if (op->kind == MOOG_R_COND_BEGIN || op->kind == MOOG_R_TIMED_BEGIN || op->kind == MOOG_R_PHASE_BEGIN) {
      int times;
      if (op->kind == MOOG_R_PHASE_BEGIN) {  // task_phases.py:79-95: not ended, and the sequence's current phase
        times = (e.envf[op->i[3]] == 0 && (op->i[0] < 0 || e.envf[op->i[0] + 1] == (double)op->i[2])) ? 1 : 0;
      } else if (op->kind == MOOG_R_TIMED_BEGIN) {  // timing.py:50-56; the guarded rules never read the countdowns
        const double c0 = e.envf[op->i[2]], c1 = e.envf[op->i[2] + 1];
        times = (c0 <= 0 && c1 > 0) ? 1 : 0;
        wsync();
        put(e, &e.envf[op->i[2]], c0 - 1);
        put(e, &e.envf[op->i[2] + 1], c1 - 1);
        wsync();
      } else {
        times = (int)eval_condition(e, op->i[0]);
      }
      int nsub = op->i[1];
      if (times <= 0 || nsub <= 0 || depth == MOOG_MAX_COND_DEPTH) {
        r += 1 + nsub;
        continue;
      }
      blk_start[depth] = r + 1;
      blk_end[depth] = r + 1 + nsub;
      blk_left[depth] = times;
      ++depth;
      r += 1;
      continue;
    }
    rule_leaf(e, r);
    r += 1;
  }
}

// ---------------------------------------------------------------------------
// action spaces
// ---------------------------------------------------------------------------
__device__ __noinline__ void actions_step(const Env &, const double *action) {
  const Env e = env_view();
  const int32_t *h = e.hdr;
  for (int a = 0; a < h[MOOG_H_N_ACTIONS]; ++a) {
    const moog_op *op = e.ops + h[MOOG_H_ACTIONS] + a;
    double a0 = action ? action[op->i[2]] : 0.0;
    double a1 = (action && op->kind != MOOG_A_GRID) ? action[op->i[2] + 1] : 0.0;
    int n = list_count(e, op->i[0], op->i[1]);
    if (op->kind == MOOG_A_SET_POSITION) {  // set_position.py:34-47
      for (int i = 0; i < n; ++i) {
        int s = list_slot(e, op->i[0], op->i[1], i);
        set_position(e, s, op->p[0] * DYN(e, MOOG_D_X, s) + (1 - op->p[0]) * a0,
                     op->p[0] * DYN(e, MOOG_D_Y, s) + (1 - op->p[0]) * a1);
      }
      continue;
    }
    double *mem = e.envf + op->i[5];
    double m0 = mem[0], m1 = mem[1];
    if (op->kind == MOOG_A_JOYSTICK) {  // joystick.py:45-65
      double ax = a0;
      double ay = (op->flags & MOOG_FL_CONSTRAINED_LR) ? 0. : a1;
      m0 = m0 * op->p[1] + op->p[0] * ax;
      m1 = m1 * op->p[1] + op->p[0] * ay;
    } else {  // grid.py:52-70: the UNIT action is added, then clipped
      int k = action ? (int)a0 : 4;
      if (k < 0 || k > 4) k = 4;
      double gx = (k == 0) ? -1. : (k == 1) ? 1. : 0.;
      double gy = (k == 2) ? -1. : (k == 3) ? 1. : 0.;
      m0 = m0 * op->p[1] + gx;
      m1 = m1 * op->p[1] + gy;
    }
    m0 = fmin(fmax(m0, -op->p[0]), op->p[0]);
    m1 = fmin(fmax(m1, -op->p[0]), op->p[0]);
    wsync();
    put(e, &mem[0], m0);
    put(e, &mem[1], m1);
    wsync();
    for (int i = 0; i < n; ++i) {
      int s = list_slot(e, op->i[0], op->i[1], i);
      double m = STAT(e, MOOG_S_MASS, s);
      if (op->flags & MOOG_FL_CONTROL_VELOCITY)
        assign_velocity(e, s, m0 / m, m1 / m);
      else
        add_velocity(e, s, m0 / m, m1 / m);
    }
  }
}

// ---------------------------------------------------------------------------
// tasks
// ---------------------------------------------------------------------------
__device__ inline void tasks_reset(const Env &e) {
  const int32_t *h = e.hdr;
  wsync();
  for (int t = 0; t < h[MOOG_H_N_TASKS]; ++t) {
    const moog_op *op = e.ops + h[MOOG_H_TASKS] + t;
    if (op->kind == MOOG_T_CONTACT_REWARD || op->kind == MOOG_T_RESET)
      put(e, &e.envf[op->i[5]], INFINITY);  // contact_reward.py:67-68, reset.py:45-46
  }
  wsync();
}

__device__ inline void actions_reset(const Env &e) {
  const int32_t *h = e.hdr;
  wsync();
  for (int a = 0; a < h[MOOG_H_N_ACTIONS]; ++a) {
    const moog_op *op = e.ops + h[MOOG_H_ACTIONS] + a;
    if (op->kind == MOOG_A_JOYSTICK || op->kind == MOOG_A_GRID) {
      put(e, &e.envf[op->i[5]], 0.);  // joystick.py:67-70, grid.py:72-75
      put(e, &e.envf[op->i[5] + 1], 0.);
    }
  }
  wsync();
}

// composite_task.py:32-42 flattened over the task tree
__device__ __noinline__ void tasks_reward(const Env &, int step_count, double *reward, int *should_reset) {
  const Env e = env_view();
  const int32_t *h = e.hdr;
  double total = 0;
  int reset = 0;
  for (int t = 0; t < h[MOOG_H_N_TASKS]; ++t) {
    const moog_op *op = e.ops + h[MOOG_H_TASKS] + t;
    switch (op->kind) {
      case MOOG_T_TIMEOUT:
        if (step_count >= op->p[0]) reset = 1;
        break;
      case MOOG_T_STAY_ALIVE:  // stay_alive.py:22-32
        if (((step_count + 1) % (int)op->p[0]) == 0) total += op->p[1];
        break;
      case MOOG_T_CONTACT_REWARD: {  // contact_reward.py:70-102
        double r = 0;
        double cd = e.envf[op->i[5]];
        int n = list_count(e, op->i[0], op->i[1]);
        int m = list_count(e, op->i[2], op->i[3]);
        for (int i = 0; i < n; ++i) {
          int sa = list_slot(e, op->i[0], op->i[1], i);
          for (int j = 0; j < m; ++j) {
            int sb = list_slot(e, op->i[2], op->i[3], j);
            if (eval_expr(e, op->i[4], sa, sb) == 0) continue;
            if (overlaps(e, sa, sb)) {
              r = op->p[2] > 0 ? eval_expr(e, (int)op->p[2] - 1, sa, sb) : op->p[0];
              if (cd == INFINITY) cd = op->p[1];
            }
          }
        }
        cd -= 1;
        if (cd < 0) reset = 1;
        wsync();
        put(e, &e.envf[op->i[5]], cd);
        wsync();
        total += r;
        break;
      }
      case MOOG_T_RESET: {  // reset.py:48-61
        double r = 0.;
        double cd = e.envf[op->i[5]];
        if (cd == INFINITY && eval_condition(e, op->i[0]) != 0) {
          r = op->i[1] > 0 ? eval_condition(e, op->i[1] - 1) : op->p[1];  // reward_fn(state), only now
          cd = op->p[0];
        }
        cd -= 1;
        if (cd < 0) reset = 1;
        wsync();
        put(e, &e.envf[op->i[5]], cd);
        wsync();
        total += r;
        break;
      }
    }
  }
  *reward = total;
  *should_reset = reset;
}

// ---------------------------------------------------------------------------
// staging: global <-> shared
// ---------------------------------------------------------------------------
__device__ __noinline__ void copy_d(double *dst, const double *src, int n, int lane) {
#pragma unroll 4
  for (int i = lane; i < n; i += 32) dst[i] = src[i];
}
__device__ __noinline__ void copy_i(int *dst, const int *src, int n, int lane) {
#pragma unroll 1
  for (int i = lane; i < n; i += 32) dst[i] = src[i];
}

// Bulk asynchronous copies (TMA, `cp.async.bulk`, SASS UBLKCP): the big arrays of the record --
// dyn, stat and the cached vertices, whose rows are multiples of 16 bytes -- move between HBM
// and shared memory without going through the warp's registers; one lane issues them, the copy
// engine completes them on an mbarrier (loads) or a bulk group (stores).
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ bool bulk_ok(const void *g, const void *sm, size_t bytes) {
  return bytes >= 16 && (((size_t)g | (size_t)smem_u32(sm) | bytes) & 15) == 0;
}
__device__ __forceinline__ void bulk_load(void *sm, const void *g, unsigned bytes, unsigned long long *mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(sm)),
               "l"(g), "r"(bytes), "r"(smem_u32(mbar))
               : "memory");
}
__device__ __forceinline__ void bulk_store(void *g, const void *sm, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(g), "r"(smem_u32(sm)), "r"(bytes)
               : "memory");
}

__device__ inline void load_env(const Env &e, const moog_state &st, size_t n, bool with_envi) {
  const int S = e.S, NF = e.hdr[MOOG_H_N_ENVF], VT = e.hdr[MOOG_H_N_VTX];
  const double *gdyn = st.dyn + n * MOOG_DYN_FIELDS * S, *gstat = st.stat + n * MOOG_STAT_FIELDS * S;
  const double *gvtx = st.vtx + n * 2 * (size_t)VT;
  const size_t bdyn = 8 * (size_t)MOOG_DYN_FIELDS * S, bstat = 8 * (size_t)MOOG_STAT_FIELDS * S, bvtx = 16 * (size_t)VT;
  const bool kd = bulk_ok(gdyn, e.dyn, bdyn), ks = bulk_ok(gstat, e.stat, bstat), kv = bulk_ok(gvtx, e.vtx, bvtx);
  const unsigned mb = smem_u32(e.mbar);
  if (e.lane == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mb) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const unsigned tx = (unsigned)((kd ? bdyn : 0) + (ks ? bstat : 0) + (kv ? bvtx : 0));
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(tx) : "memory");
    if (kd) bulk_load(e.dyn, gdyn, (unsigned)bdyn, e.mbar);
    if (ks) bulk_load(e.stat, gstat, (unsigned)bstat, e.mbar);
    if (kv) bulk_load(e.vtx, gvtx, (unsigned)bvtx, e.mbar);
  }
  wsync();
  // the small / oddly sized arrays go through the lanes while the bulk copies are in flight
  if (!kd) copy_d(e.dyn, gdyn, MOOG_DYN_FIELDS * S, e.lane);
  if (!ks) copy_d(e.stat, gstat, MOOG_STAT_FIELDS * S, e.lane);
  copy_i(e.meta, st.meta + n * MOOG_META_FIELDS * S, MOOG_META_FIELDS * S, e.lane);
  copy_i(e.cnt, st.cnt + n * MOOG_MAX_LAYERS, MOOG_MAX_LAYERS, e.lane);
  copy_d(e.envf, st.envf + n * NF, NF, e.lane);
  if (!kv) copy_d((double *)e.vtx, gvtx, 2 * VT, e.lane);
  if (with_envi) copy_i(e.envi, st.envi + n * MOOG_ENVI_WORDS, MOOG_ENVI_WORDS, e.lane);
  // wait for the bytes (phase 0 of the barrier: this is its only use in the launch)
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "MOOG_LOAD_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n"
      "@p bra MOOG_LOAD_DONE;\n"
      "bra MOOG_LOAD_WAIT;\n"
      "MOOG_LOAD_DONE:\n"
      "}" ::"r"(mb)
      : "memory");
  wsync();
}

__device__ inline void store_env(const Env &e, const moog_state &st, size_t n) {
  const int S = e.S, NF = e.hdr[MOOG_H_N_ENVF], VT = e.hdr[MOOG_H_N_VTX];
  double *gdyn = st.dyn + n * MOOG_DYN_FIELDS * S, *gstat = st.stat + n * MOOG_STAT_FIELDS * S;
  double *gvtx = st.vtx + n * 2 * (size_t)VT;
  const size_t bdyn = 8 * (size_t)MOOG_DYN_FIELDS * S, bstat = 8 * (size_t)MOOG_STAT_FIELDS * S, bvtx = 16 * (size_t)VT;
  const bool kd = bulk_ok(gdyn, e.dyn, bdyn), ks = bulk_ok(gstat, e.stat, bstat), kv = bulk_ok(gvtx, e.vtx, bvtx);
  // the lanes' shared-memory writes become visible to the copy engine (async proxy)
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  wsync();
  if (e.lane == 0) {
    if (kd) bulk_store(gdyn, e.dyn, (unsigned)bdyn);
    if (ks) bulk_store(gstat, e.stat, (unsigned)bstat);
    if (kv) bulk_store(gvtx, e.vtx, (unsigned)bvtx);
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  }
  if (!kd) copy_d(gdyn, e.dyn, MOOG_DYN_FIELDS * S, e.lane);
  if (!ks) copy_d(gstat, e.stat, MOOG_STAT_FIELDS * S, e.lane);
  copy_i(st.meta + n * MOOG_META_FIELDS * S, e.meta, MOOG_META_FIELDS * S, e.lane);
  copy_i(st.cnt + n * MOOG_MAX_LAYERS, e.cnt, MOOG_MAX_LAYERS, e.lane);
  copy_d(st.envf + n * NF, e.envf, NF, e.lane);
  if (!kv) copy_d(gvtx, (const double *)e.vtx, 2 * VT, e.lane);
  copy_i(st.envi + n * MOOG_ENVI_WORDS, e.envi, MOOG_ENVI_WORDS, e.lane);
  if (e.lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // done before the CTA retires
  wsync();
}

// environment.py:88-96: task / action reset, every rule reset and stepped once
__device__ inline void post_reset(const Env &e) {
  wsync();
  puti(e, &e.envi[MOOG_EI_STEP_COUNT], 0);
  puti(e, &e.envi[MOOG_EI_RESET_NEXT], 0);
  wsync();
  {  // environment.py:86: meta_state = meta_state_initializer() -- its entries are variables of the record
    const int32_t *h = e.hdr;
    for (int q = e.lane; q < h[MOOG_H_N_METAVAR]; q += 32) e.envf[h[MOOG_H_METAVAR_OFF] + q] = e.dpool[h[MOOG_H_METAVAR_INIT] + q];
    wsync();
  }
  tasks_reset(e);
  actions_reset(e);
  {  // AbstractRule.reset of the rules that keep state: TimedRule re-arms its interval (timing.py:45-48)
    const int32_t *h = e.hdr;
    wsync();
    for (int r = h[MOOG_H_RULES]; r < h[MOOG_H_RULES] + h[MOOG_H_N_RULES]; ++r) {
      const moog_op *op = e.ops + r;
      if (op->kind == MOOG_R_TIMED_BEGIN) {
        put(e, &e.envf[op->i[2]], op->p[0]);
        put(e, &e.envf[op->i[2] + 1], op->p[1]);
      }
      if (op->kind == MOOG_R_PORTAL)  // portal.py:36-39: _currently_teleporting = set()
        for (int s2 = e.lane; s2 < e.S; s2 += 32) META(e, MOOG_M_FLAGS, s2) &= ~MOOG_SF_TELEPORTING;
      if (op->kind == MOOG_R_FIXATION) put(e, &e.envf[op->i[2]], 0.0);  // fixation.py:41-43
      if (op->kind == MOOG_R_PHASESEQ_BEGIN) {  // task_phases.py:118-124
        put(e, &e.envf[op->i[0]], 0.0);
        put(e, &e.envf[op->i[0] + 1], 0.0);
        if (op->i[2] >= 0) put(e, &e.envf[op->i[2]], e.dpool[op->i[4]]);
      }
      if (op->kind == MOOG_R_PHASE_BEGIN) {  // task_phases.py:71-77: the duration is drawn anew
        double dur = op->p[0];
        if (op->p[2] > op->p[1]) {  // np.random.randint(p1, p2)
          const int lo = (int)op->p[1], hi = (int)op->p[2];
          const int d = lo + (int)(rule_noise_at(e, op->i[4]) * (double)(hi - lo));
          dur = d >= hi ? hi - 1 : d;
        }
        put(e, &e.envf[op->i[3]], 0.0);
        put(e, &e.envf[op->i[3] + 1], 0.0);
        put(e, &e.envf[op->i[3] + 2], dur);
      }
      if (op->kind == MOOG_R_TREE)  // the rule's own reset(): its attributes back to their first values
        for (int q = e.lane; q < op->i[3]; q += 32) e.envf[op->i[2] + q] = e.dpool[op->i[4] + q];
    }
    wsync();
  }
  rules_step(e);
}

// One warp = one CTA = one env: every shared-memory address below is a
// CTA-uniform offset from the dynamic shared-memory base, and the program's
// dimensions arrive in the parameter bank, so address arithmetic stays on the
// uniform datapath instead of occupying vector registers.
__device__ __forceinline__ void owner_warp(const StepArgs &a, unsigned char *smem_raw, const int lane) {
  // CTAs are dispatched in blockIdx order: with `order` the envs that were the most
  // expensive on the previous call go first, so the longest-running env does not
  // start in the last wave (longest-processing-time-first)
  const int n = a.order ? a.order[blockIdx.x] : (int)blockIdx.x;
  const long long t_begin = clock64();
  unsigned long long trace_t0 = 0;
  if (a.trace) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(trace_t0));
  unsigned smid = 0;
  if (a.sm_active) {
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    if (lane == 0) atomicAdd(a.sm_active + (smid & 255), 1);
  }

  ProgramView pv = view_of(a.blob);
  const int NF = a.NF;
  const SmemLayout lay = smem_layout(a.S, a.VT > 0 ? a.VT : 1, NF, a.CMW, (int)(blockDim.x >> 5), a.dcv_tile);
  unsigned char *base = smem_raw;
  {
    int *h = (int *)(base + lay.hdr);
    for (int i = lane; i < MOOG_HDR_WORDS; i += 32) h[i] = pv.hdr[i];
    if (lane < 12) ((long long *)(base + lay.ctr))[lane] = lane == CT_NEAR ? -2 : 0;
    if (lane == 0) {
      EnvRec *r = (EnvRec *)(base + lay.rec);
      r->lay = lay;
      r->S = a.S; r->L = a.L; r->K = a.K; r->VT = a.VT;
      r->env_id = n;
      r->ops = pv.ops; r->ipool = pv.ipool; r->expr = pv.expr;
      r->vmap = a.vmap;
      r->dpool = pv.dpool;
      const int ND = pv.hdr[MOOG_H_NOISE_DIM], RND = pv.hdr[MOOG_H_RULE_NOISE_DIM];
      r->noise = a.io.noise ? a.io.noise + (size_t)n * a.K * ND : nullptr;
      r->rule_noise = a.io.rule_noise ? a.io.rule_noise + (size_t)n * RND : nullptr;
      r->seed = a.io.seed;
    }
    wsync();
  }
  const Env e = env_view();

  // slot -> first cached vertex
  for (int s = lane; s <= e.S; s += 32) e.voff[s] = pv.voff[s];
  if (a.vmap) {
    uint8_t *vm = (uint8_t *)(base + lay.vmap);
    for (int v = lane; v < a.VT; v += 32) vm[v] = (uint8_t)(a.vmap[v] >> 8);
  }
  wsync();

  if (lane == 0) {  // offsets of the candidate matrices of the Collision entries
    int off = 0;
    for (int f = 0; f < pv.hdr[MOOG_H_N_FORCES] && f < MOOG_MAX_FORCE_OPS; ++f) {
      const moog_op *op = pv.ops + pv.hdr[MOOG_H_FORCES] + f;
      e.cmoff[f] = off;
      if (op->kind == MOOG_F_COLLISION) {
        int ca = pv.hdr[MOOG_H_LAYER_OFF + op->i[0] + 1] - pv.hdr[MOOG_H_LAYER_OFF + op->i[0]];
        int cb = pv.hdr[MOOG_H_LAYER_OFF + op->i[1] + 1] - pv.hdr[MOOG_H_LAYER_OFF + op->i[1]];
        off += ca * ((cb + 31) >> 5);
      }
    }
  }
  copy_i(e.envi, a.st.envi + (size_t)n * MOOG_ENVI_WORDS, MOOG_ENVI_WORDS, lane);
  wsync();
  const bool do_reset = a.mode == MODE_ENV_STEP && a.io.pool != nullptr && e.envi[MOOG_EI_RESET_NEXT] != 0;
  {
    const moog_state *src = &a.st;
    size_t row = (size_t)n;
    if (do_reset) {
      int idx;
      if (a.io.reset_index) {
        idx = a.io.reset_index[n];
      } else {
        double u = philox_uniform(a.io.seed ^ 0xD1B54A32D192ED03ull, (uint32_t)n, (uint32_t)e.envi[MOOG_EI_EPISODES], 0u, 0u);
        idx = (int)(u * a.io.pool_size);
      }
      idx = idx < 0 ? 0 : (idx >= a.io.pool_size ? a.io.pool_size - 1 : idx);
      if (a.io.sample_resets && pv.hdr[MOOG_H_N_RESET] > 0) idx = 0;  // pool entry 0 is the template
      src = &a.pool;
      row = (size_t)idx;
    }
    load_env(e, *src, row, false);
  }
  wsync();
  refresh_all_boxes(e);
  if (do_reset && a.io.sample_resets && pv.hdr[MOOG_H_N_RESET] > 0) {
    // the generated sprites of the template are drawn afresh for this env and episode
    for (int z = 0; z < pv.hdr[MOOG_H_N_RESET]; ++z)
      reset_generate(e, pv.ops + pv.hdr[MOOG_H_RESET] + z, a.io.seed);
  }

  double reward = 0.0;
  int step_type = MOOG_STEP_MID;
  double ep_len_done = 0.0, ep_done = 0.0;

  const bool full_step = a.mode == MODE_ENV_STEP && !do_reset;
  if (a.mode == MODE_POST_RESET || do_reset) {
    if (do_reset) {
      int ep = e.envi[MOOG_EI_EPISODES] + 1;
      wsync();
      puti(e, &e.envi[MOOG_EI_EPISODES], ep);
    }
    post_reset(e);
    reward = NAN;
    step_type = MOOG_STEP_FIRST;
  } else if (a.mode == MODE_OVERLAP) {
    int la = a.layer_a, lb = a.layer_b;
    int ca = LOFF(e, la + 1) - LOFF(e, la), cb = LOFF(e, lb + 1) - LOFF(e, lb);
    uint8_t *o = a.overlap_out + (size_t)n * ca * cb;
    for (int i = lane; i < ca * cb; i += 32) o[i] = 0;
    wsync();
    for (int i = 0; i < e.cnt[la]; ++i)
      for (int j = 0; j < e.cnt[lb]; ++j) {
        bool r = overlaps(e, LOFF(e, la) + i, LOFF(e, lb) + j);
        if (lane == 0) o[i * cb + j] = (uint8_t)r;
      }
  } else {
    // environment.py:98-126 (MODE_PHYSICS: abstract_physics.py:39-42 alone)
    if (full_step) {
      rules_step(e);
      actions_step(e, a.io.actions ? a.io.actions + (size_t)n * e.hdr[MOOG_H_ACTION_DIM] : nullptr);
    }
    for (int k = 0; k < e.K; ++k) {
      wsync();
      if (lane == 0) e.ctr[CT_SUBSTEP] = k;
      wsync();
      apply_physics(e, a.CMW);
    }
    if (full_step) {
      int sc = e.envi[MOOG_EI_STEP_COUNT] + 1;
      wsync();
      puti(e, &e.envi[MOOG_EI_STEP_COUNT], sc);
      wsync();
      int reset;
      tasks_reward(e, sc, &reward, &reset);
      step_type = reset ? MOOG_STEP_LAST : MOOG_STEP_MID;
      wsync();
      puti(e, &e.envi[MOOG_EI_RESET_NEXT], reset);
      wsync();
      if (reset) {
        ep_len_done = (double)sc;
        ep_done = 1.0;
      }
    }
  }
  wsync();
  if (blockDim.x == 64) {  // release the helper warp
    if (lane == 0) ((int *)e.xchg)[0] = HELPER_EXIT;
    cta_bar(1);
  }
  if (a.mode != MODE_OVERLAP) store_env(e, a.st, (size_t)n);
  if (a.done && lane == 0) {
    // this env's record is in HBM (store_env waited for its bulk stores): append the env to the
    // list of finished envs, release order, for the render CTA that waits on that entry
    __threadfence();
    const int k = atomicAdd(a.done, 1);
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(a.done + 1 + k), "r"(n + 1) : "memory");
    if (a.sm_active) atomicSub(a.sm_active + (smid & 255), 1);
  }
  if (lane == 0) {
    if (a.cost) {
      long long c = (clock64() - t_begin) >> 6;
      a.cost[n] = c > 0x7fffffffll ? 0x7fffffff : (int)c;
    }
    if (a.io.reward) a.io.reward[n] = (float)reward;
    if (a.io.step_type) a.io.step_type[n] = step_type;
    if (a.io.discount)
      a.io.discount[n] = step_type == MOOG_STEP_FIRST ? NAN : (step_type == MOOG_STEP_LAST ? 0.0f : 1.0f);
    if (a.io.counters) {
      a.io.counters[MOOG_N_COUNTERS * (size_t)n + 0] = e.ctr[CT_CALLS];
      a.io.counters[MOOG_N_COUNTERS * (size_t)n + 1] = e.ctr[CT_TRUE];
      a.io.counters[MOOG_N_COUNTERS * (size_t)n + 2] = e.ctr[CT_COLL];
      a.io.counters[MOOG_N_COUNTERS * (size_t)n + 3] = e.ctr[CT_HASH];
      a.io.counters[MOOG_N_COUNTERS * (size_t)n + 4] = clock64() - t_begin;
      a.io.counters[MOOG_N_COUNTERS * (size_t)n + 5] = e.ctr[CT_NARROW];
      a.io.counters[MOOG_N_COUNTERS * (size_t)n + 6] = e.ctr[CT_CYC_NARROW];
      a.io.counters[MOOG_N_COUNTERS * (size_t)n + 7] = e.ctr[CT_CYC_RESOLVE];
      if (a.trace) {
        unsigned long long t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        a.io.counters[MOOG_N_COUNTERS * (size_t)n + 6] = (long long)trace_t0;
        a.io.counters[MOOG_N_COUNTERS * (size_t)n + 7] = (long long)t1;
      }
    }
    if (a.io.stats && a.mode == MODE_ENV_STEP) {
      if (step_type != MOOG_STEP_FIRST) {
        if (reward != 0.0) atomicAdd(&a.io.stats[0], reward);
        atomicAdd(&a.io.stats[3], 1.0);
      }
      if (ep_done != 0.0) {
        atomicAdd(&a.io.stats[1], ep_len_done);
        atomicAdd(&a.io.stats[2], ep_done);
      }
    }
  }
}

__global__ void __launch_bounds__(64) moog_step_kernel(const StepArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31;
  // A kernel launched behind this one with programmatic stream serialization (the tail render
  // kernel, moog_render.cu) may start as soon as every CTA of this grid has got here, i.e. once
  // no env is waiting for an SM any more; it consumes the envs in the order they finish (a.done).
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (threadIdx.x >= 32) {
    // Helper warp (launched when the step is bound by its longest-running env and the SMs
    // have registers to spare): sleeps on a named barrier until the owner posts a request,
    // runs one direction of _get_collision_vectors (collisions.py:268-283: the two directed
    // computations are independent) on the env's shared-memory record, posts the result.
    for (;;) {
      cta_bar(1);
      const Env e = env_view();
      const int *req = (const int *)e.xchg;
      if (req[0] == HELPER_EXIT) break;
      CVec out;
      directed_collision_vectors(e, req[1], req[2], 1.0 / e.K, out);
      if (e.lane == 0) *(CVec *)(e.xchg + 16) = out;
      cta_bar(2);
    }
  } else {
    owner_warp(a, smem_raw, lane);
  }
  if (!a.frames) return;
  // PILRenderer.__call__ (pil_renderer.py:88-120) of the state the env was left in, by every
  // thread of the CTA, from the record that is still in shared memory: the canvas, edge lists and
  // int vertices go where the step's scratch was, the item spans into the vertex cache once the
  // int vertices exist (the owner's bulk stores have completed: store_env waits for them).
  // Frames leave the SM while the longest-running envs of the batch are still being stepped.
  __syncthreads();
  {
    const Env e = env_view();
    const int OH = e.hdr[MOOG_H_R_HEIGHT], OW = e.hdr[MOOG_H_R_WIDTH];
    const int C = e.hdr[MOOG_H_R_MODIFIER] == MOOG_PMOD_TORUS ? 9 : 1;
    const int VTr = a.VT > 0 ? a.VT : 1;
    const RenderLayout lay = render_layout(OH, OW, a.S * C, VTr * C, OW, 16 * VTr);
    RenderSrc src;
    src.dyn = e.dyn; src.stat = e.stat; src.meta = e.meta; src.cnt = e.cnt;
    src.vtx = e.vtx; src.hdr = e.hdr; src.voff = e.voff; src.view = e.hdr + MOOG_H_R_HEIGHT;
    const int T = (int)blockDim.x;
    const int P = (OH * 2 <= T) ? 2 : 1;
    render_env(src, lay, smem_raw + a.render_off, (unsigned *)e.vtx, (int)threadIdx.x, T, P, true,
               a.frames + (size_t)e.env_id * OH * OW * 3, [] { __syncthreads(); });
  }
}

// order[] = env indices by decreasing cost[] (bucket sort; the order inside a bucket
// is arbitrary, which only affects scheduling, never results).  One CTA.
#define ORDER_BUCKETS 256
__global__ void __launch_bounds__(1024) moog_order_kernel(const int *cost, int *order, int n) {
  __shared__ int hist[ORDER_BUCKETS];
  __shared__ int start[ORDER_BUCKETS];
  __shared__ int smax;
  const int t = threadIdx.x;
  if (t < ORDER_BUCKETS) hist[t] = 0;
  if (t == 0) smax = 0;
  __syncthreads();
  int m = 0;
  for (int i = t; i < n; i += blockDim.x) m = max(m, cost[i]);
  atomicMax(&smax, m);
  __syncthreads();
  const int shift_div = smax / ORDER_BUCKETS + 1;
  for (int i = t; i < n; i += blockDim.x) atomicAdd(&hist[min(cost[i] / shift_div, ORDER_BUCKETS - 1)], 1);
  __syncthreads();
  if (t == 0) {
    int acc = 0;
    for (int b = ORDER_BUCKETS - 1; b >= 0; --b) {
      start[b] = acc;
      acc += hist[b];
    }
  }
  __syncthreads();
  for (int i = t; i < n; i += blockDim.x) {
    int b = min(cost[i] / shift_div, ORDER_BUCKETS - 1);
    order[atomicAdd(&start[b], 1)] = i;
  }
}

cudaError_t launch_order(const int *cost, int *order, int n, cudaStream_t stream, int *n_launches) {
  moog_order_kernel<<<1, 1024, 0, stream>>>(cost, order, n);
  if (n_launches) *n_launches += 1;
  return cudaGetLastError();
}

// How a step call launches a batch of n_envs on a device with `sms` multiprocessors.
StepPlan plan_step(const int32_t *hdr, int mode, int n_envs, bool frames, int sms, const LaunchOptions &opt) {
  StepPlan p = {};
  // Longest-processing-time-first dispatch from the costs of the previous call (moog_order_kernel):
  // a large batch runs in waves, and the env that was the most expensive must not start in the last one.
  p.ordered = (mode == MODE_ENV_STEP || mode == MODE_PHYSICS) && n_envs >= 1024;
  // The step ends when its longest-running env does, and a warp runs ~2.4x slower next to 11
  // others than alone (profiles/README.md): with the envs dispatched longest-first, capping
  // the envs resident per SM at about n_envs / (5.5 .. 7 x SMs) finishes the step sooner than filling
  // the SMs (4096 envs on 148 SMs: 5 per SM; measured with the frames drawn behind the step, step
  // + render per 4096 envs: 3: 5.33 ms, 4: 4.66 ms, 5: 4.46 ms, and 5.6 ms at 12 with one warp per env).
  // In that regime the SMs have registers to spare, and every env gets a helper warp that
  // computes one of the two directions of _get_collision_vectors (option "helper" overrides).
  if (sms > 0) {
    int resident = (n_envs + 7 * sms / 2) / (7 * sms);  // n_envs / (7 x SMs), rounded
    // helper-warp regime (few envs per SM): one more env per SM pays once the frames are drawn
    // behind the step (4096 envs: 4 -> 5 per SM, 4.66 -> 4.46 ms); larger batches keep 7 waves
    // (8192 / 32768 envs measured slower at 10 / 40 per SM than at 8 / 32)
    if (resident <= 4) resident = (2 * n_envs + 11 * sms / 2) / (11 * sms);
    if (resident < 2) resident = 2;
    p.helper = resident <= 6;
    if (p.ordered) p.resident = resident;
  }
  if (opt.helper >= 0) p.helper = opt.helper != 0;
  if (opt.ctas_per_sm > 0) p.resident = opt.ctas_per_sm;
  // The residency cap is a padded dynamic shared-memory request (option "ctas_per_sm" sets the cap).
  size_t smem = (size_t)env_smem_bytes(hdr, p.helper);
  if (p.resident > 0 && (size_t)233472 / (smem + 1024) > (size_t)p.resident) {
    // (when the records alone allow exactly `resident` envs nothing is padded, and the SM keeps
    // the shared memory it does not need as L1: launch_step sets the carve-out)
    size_t per_cta = (size_t)233472 / (size_t)p.resident;  // 228 KB per SM, 1 KB of it reserved per CTA
    if (per_cta > 1024 + smem) smem = ((per_cta - 1024) & ~(size_t)127);
    if (smem > 227 * 1024) smem = 227 * 1024;
  }
  // The frame of the state the env is left in (io.frames), drawn by the env's own CTA right after
  // its step when one CTA can hold the canvas: the renderer reads the record where it lies in shared
  // memory and builds its canvas where the step's scratch was.  Small batches (every env has an SM
  // to itself) gain one launch and no second pass over the state; for large ones the render kernel is
  // the better choice: measured on 4096 falling_balls20 envs, two warps per env drawing between the
  // steps of their neighbours cost more (6.0 ms) than the render kernel behind the step (4.3 + 0.55 ms).
  if (frames && n_envs <= 2 * sms && hdr[MOOG_H_R_ENABLED] && hdr[MOOG_H_R_AA] == 1) {
    const int VTr = hdr[MOOG_H_N_VTX] > 0 ? hdr[MOOG_H_N_VTX] : 1;
    const SmemLayout sl = smem_layout(hdr[MOOG_H_N_SLOTS], VTr, hdr[MOOG_H_N_ENVF], hdr[MOOG_H_CMASK_WORDS],
                                      p.helper ? 2 : 1, p.helper ? DCV_TILE_MAX : DCV_TILE_MIN);
    const int C = hdr[MOOG_H_R_MODIFIER] == MOOG_PMOD_TORUS ? 9 : 1;
    const RenderLayout rl = render_layout(hdr[MOOG_H_R_HEIGHT], hdr[MOOG_H_R_WIDTH], hdr[MOOG_H_N_SLOTS] * C, VTr * C,
                                          hdr[MOOG_H_R_WIDTH], 16 * VTr);
    const int render_off = (sl.scratch + 15) & ~15;  // everything from the warps' scratch on is dead after the step
    const size_t need = (size_t)render_off + (size_t)rl.total;
    if (need <= 227 * 1024) {
      p.fuse = true;
      p.render_off = render_off;
      if (smem < need) smem = need;
    }
  }
  p.smem = smem;
  // Frames of a large batch: the step ends when its longest-running env does, and long before
  // that most SMs have no env left to step.  The render kernel is launched behind the step kernel
  // with programmatic stream serialization, starts as soon as the last env has got an SM, and
  // draws the envs in the order they finish (the `done` list) on the SMs the step left idle.
  p.tail = frames && p.ordered && !p.fuse;
  return p;
}

cudaError_t launch_step(const StepArgs &a, const int32_t *hdr, const StepPlan &plan, cudaStream_t stream,
                        int *n_launches) {
  if (a.n_envs <= 0) return cudaSuccess;
  const size_t smem = plan.smem;
  static size_t configured = 0;
  if (smem > configured) {
    cudaError_t err = cudaFuncSetAttribute(moog_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    configured = smem;
  }
  {
    // Shared-memory carve-out: the smallest supported capacity (.. 100, 132, 164, 196, 228 KB) that
    // holds the CTAs that will be resident; what is left of the SM's 256 KB serves as L1 for the
    // spills and the program's ops / expressions in global memory
    static int carve_set = -1;
    const size_t per_sm = ((size_t)233472 / (smem + 1024)) * (smem + 1024);
    const int caps[] = {100, 132, 164, 196, 228};
    int pick = 228;
    for (int c : caps)
      if (per_sm <= (size_t)c * 1024) { pick = c; break; }
    const int pct = pick == 228 ? 100 : (pick * 100) / 228;   // rounded down: the driver takes the next capacity up
    if (pct != carve_set) {
      cudaFuncSetAttribute(moog_step_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
      carve_set = pct;
    }
  }
  StepArgs b = a;
  b.S = hdr[MOOG_H_N_SLOTS];
  b.L = hdr[MOOG_H_N_LAYERS];
  b.K = hdr[MOOG_H_K];
  b.VT = hdr[MOOG_H_N_VTX];
  b.NF = hdr[MOOG_H_N_ENVF];
  b.CMW = hdr[MOOG_H_CMASK_WORDS];
  b.dcv_tile = plan.helper ? DCV_TILE_MAX : DCV_TILE_MIN;
  b.render_off = plan.render_off;
  b.frames = plan.fuse ? a.io.frames : nullptr;
  moog_step_kernel<<<a.n_envs, plan.helper ? 64 : 32, smem, stream>>>(b);
  if (n_launches) *n_launches += 1;
  return cudaGetLastError();
}

}  // namespace moog
