// moog_capi.cu -- the extern "C" boundary declared in include/moog_b200.h.
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <string>
#include <vector>

#include "moog_common.cuh"

struct moog_program {
  void *dev_blob;
  size_t nbytes;
  int32_t hdr[MOOG_HDR_WORDS];
  // scheduling scratch owned by the program (the only device memory besides the
  // blob the library allocates): per-env cost of the previous step and the
  // dispatch order derived from it
  int *sched;  // [2][sched_cap]: cost, order
  int sched_cap;
  const void *sched_state;  // the state the costs belong to
  int *done;                // [1 + done_cap]: envs in the order the running step finishes them
  int done_cap;
  // views (one per PILRenderer): their settings and where they lie in the blob (int32 words)
  int n_views;
  int32_t view[MOOG_MAX_VIEWS][MOOG_VIEW_WORDS];
  int view_off[MOOG_MAX_VIEWS];
  // anti_aliasing > 1: Lanczos coefficient tables (Resample.c) per view, built on first use
  int *resample[MOOG_MAX_VIEWS];
  moog::RenderPlan plan[MOOG_MAX_VIEWS];  // how the render kernels draw each view (render_plan)
  int ksize_h[MOOG_MAX_VIEWS], ksize_v[MOOG_MAX_VIEWS];
  // masks (one per SpriteMask): where their rows lie in the blob, and how the mask kernel draws them
  int n_masks;
  int mask_off[MOOG_MAX_VIEWS];
  moog::RenderPlan mask_plan[MOOG_MAX_VIEWS];
  // largest outline a slot of each layer can hold (from the blob's voff table)
  int layer_vcap[MOOG_MAX_LAYERS];
  // cached vertex -> (slot << 8 | index within the slot's outline), [VT]: the Euler pass of the step
  // kernel walks the vertex cache flat, lane = vertex
  uint16_t *dev_vmap;
  moog::LaunchOptions opt;  // MOOG_* environment variables at creation time, then moog_program_set_option
};

namespace {
std::atomic<int64_t> g_launches{0};
thread_local std::string g_cuda_error;

int cuda_fail(cudaError_t err) {
  g_cuda_error = cudaGetErrorString(err);
  return MOOG_E_CUDA;
}

bool valid_state(const moog_state *st) {
  return st && st->dyn && st->stat && st->meta && st->cnt && st->envi && st->envf && st->vtx;
}
}  // namespace

namespace moog {
LaunchOptions launch_options_from_env() {
  LaunchOptions o;
  static const struct { const char *env, *name; } kVars[] = {
      {"MOOG_HELPER", "helper"}, {"MOOG_CTAS_PER_SM", "ctas_per_sm"}, {"MOOG_TRACE_TIMES", "trace_times"}};
  for (const auto &v : kVars) {
    const char *t = getenv(v.env);
    if (t && *t) set_launch_option(o, v.name, atoi(t));
  }
  return o;
}
bool set_launch_option(LaunchOptions &o, const char *name, int value) {
  if (!name) return false;
  const std::string n(name);
  if (n == "helper") o.helper = value;
  else if (n == "ctas_per_sm") o.ctas_per_sm = value;
  else if (n == "trace_times") o.trace_times = value;
  else if (n == "seed") o.seed = value;
  else return false;
  return true;
}
}  // namespace moog

extern "C" {

// Every offset, count and pool index a kernel (or this file) will follow is checked here, before the blob
// is accepted: a malformed program is MOOG_E_INVAL, not an out-of-bounds read on the host or the device.
int moog_program_validate(const void *blob, size_t nbytes) {
  if (!blob || nbytes < sizeof(int32_t) * MOOG_HDR_WORDS) return MOOG_E_INVAL;
  const int32_t *hdr = (const int32_t *)blob;
  if ((uint32_t)hdr[MOOG_H_MAGIC] != MOOG_MAGIC || hdr[MOOG_H_VERSION] != MOOG_VERSION) return MOOG_E_INVAL;
  if ((size_t)hdr[MOOG_H_BYTES] != nbytes) return MOOG_E_INVAL;
  const int S = hdr[MOOG_H_N_SLOTS], L = hdr[MOOG_H_N_LAYERS], NO = hdr[MOOG_H_N_OPS], NI = hdr[MOOG_H_N_IPOOL],
            NX = hdr[MOOG_H_N_EXPR], ND = hdr[MOOG_H_N_DPOOL], VT = hdr[MOOG_H_N_VTX], NF = hdr[MOOG_H_N_ENVF];
  if (S < 0 || S > MOOG_MAX_SLOTS || L < 0 || L > MOOG_MAX_LAYERS || hdr[MOOG_H_K] < 1) return MOOG_E_INVAL;
  if (NO < 0 || NI < 0 || NX < 0 || ND < 0 || VT < 0 || NF < 0) return MOOG_E_INVAL;
  if (hdr[MOOG_H_ACTION_DIM] < 0 || hdr[MOOG_H_NOISE_DIM] < 0 || hdr[MOOG_H_RULE_NOISE_DIM] < 0) return MOOG_E_INVAL;
  const size_t need = sizeof(int32_t) * MOOG_HDR_WORDS + sizeof(moog_op) * (size_t)NO +
                      sizeof(int32_t) * (((size_t)NI + 1) & ~(size_t)1) + sizeof(moog_ex) * (size_t)NX +
                      sizeof(double) * (size_t)ND;
  if (need != nbytes) return MOOG_E_INVAL;
  const moog::ProgramView pv = moog::view_of(blob);
  // metadata columns: N_META blocks of S doubles inside envf
  if (hdr[MOOG_H_N_META] < 0 || hdr[MOOG_H_N_META] > MOOG_MAX_META ||
      (hdr[MOOG_H_N_META] > 0 && (hdr[MOOG_H_META_OFF] < 0 || (long long)hdr[MOOG_H_META_OFF] + (long long)hdr[MOOG_H_N_META] * S > NF)))
    return MOOG_E_INVAL;
  if (hdr[MOOG_H_N_METAVAR] < 0 ||
      (hdr[MOOG_H_N_METAVAR] > 0 && (hdr[MOOG_H_METAVAR_OFF] < 0 || (long long)hdr[MOOG_H_METAVAR_OFF] + hdr[MOOG_H_N_METAVAR] > NF ||
                                     hdr[MOOG_H_METAVAR_INIT] < 0 || (long long)hdr[MOOG_H_METAVAR_INIT] + hdr[MOOG_H_N_METAVAR] > ND)))
    return MOOG_E_INVAL;
  // layers partition the slots
  if (hdr[MOOG_H_LAYER_OFF] != 0 || hdr[MOOG_H_LAYER_OFF + L] != S) return MOOG_E_INVAL;
  for (int l = 0; l < L; ++l)
    if (hdr[MOOG_H_LAYER_OFF + l + 1] < hdr[MOOG_H_LAYER_OFF + l]) return MOOG_E_INVAL;
  // cached vertices: voff[S + 1] in ipool, non-decreasing, inside [0, VT]
  const int vo = hdr[MOOG_H_VOFF];
  if (vo < 0 || (long long)vo + S + 1 > NI) return MOOG_E_INVAL;
  if (pv.ipool[vo] != 0 || pv.ipool[vo + S] > VT) return MOOG_E_INVAL;
  for (int s2 = 0; s2 < S; ++s2) {
    const int nv = pv.ipool[vo + s2 + 1] - pv.ipool[vo + s2];
    if (nv < 0 || nv > MOOG_MAX_OUTLINE) return MOOG_E_INVAL;
  }
  // op sections
  const int sect[6][2] = {{MOOG_H_FORCES, MOOG_H_N_FORCES}, {MOOG_H_CORR, MOOG_H_N_CORR},   {MOOG_H_RULES, MOOG_H_N_RULES},
                          {MOOG_H_TASKS, MOOG_H_N_TASKS},   {MOOG_H_ACTIONS, MOOG_H_N_ACTIONS}, {MOOG_H_RESET, MOOG_H_N_RESET}};
  for (int k = 0; k < 6; ++k) {
    const int a = hdr[sect[k][0]], n = hdr[sect[k][1]];
    if (n < 0 || (n > 0 && (a < 0 || (long long)a + n > NO))) return MOOG_E_INVAL;
  }
  // expression programs end inside the pool
  if (NX > 0 && pv.expr[NX - 1].op != MOOG_X_END) return MOOG_E_INVAL;
  for (int x = 0; x < NX; ++x) {
    const moog_ex &e = pv.expr[x];
    if (e.op < 0 || e.op > MOOG_X_NORM2) return MOOG_E_INVAL;
    if (e.op == MOOG_X_RULE_NOISE && (e.arg < 0 || e.arg >= hdr[MOOG_H_RULE_NOISE_DIM])) return MOOG_E_INVAL;
    if ((e.op == MOOG_X_ENVF || e.op == MOOG_X_STORE_ENVF) && (e.arg < 0 || e.arg >= NF)) return MOOG_E_INVAL;
    if ((e.op == MOOG_X_ATTR0 || e.op == MOOG_X_ATTR1 || e.op == MOOG_X_STORE) &&
        !((e.arg >= 0 && e.arg <= MOOG_AT_OPACITY) || (e.arg >= MOOG_AT_META0 && e.arg < MOOG_AT_META0 + hdr[MOOG_H_N_META])))
      return MOOG_E_INVAL;
  }
  const int n_shapes_max = NI;  // shape table: offsets into dpool
  const int st = hdr[MOOG_H_SHAPE_TAB];
  if (st < 0 || st > NI) return MOOG_E_INVAL;
  (void)n_shapes_max;
  auto layer_ok = [&](int l) { return l >= 0 && l < L; };
  auto list_ok = [&](int start, int count, int limit) {  // ipool[start, start + count): values in [0, limit)
    if (count < 0 || (count > 0 && (start < 0 || (long long)start + count > NI))) return false;
    for (int q = 0; q < count; ++q)
      if (pv.ipool[start + q] < 0 || pv.ipool[start + q] >= limit) return false;
    return true;
  };
  auto expr_ok = [&](int x) { return x == -1 || (x >= 0 && x < NX); };
  auto cond_ok = [&](int o) { return o >= 0 && o < NO && pv.ops[o].kind >= MOOG_SC_ALL && pv.ops[o].kind <= MOOG_SC_TREE; };
  auto envf_ok = [&](int f, int n) { return f >= 0 && (long long)f + n <= NF; };
  auto table_ok = [&](int t) {  // sampler table: MOOG_Z_N_ATTRS leaves (kind, dpool index, n) + the extension count
    if (t < 0 || (long long)t + 3 * MOOG_Z_N_ATTRS + 1 > NI) return false;
    for (int a = 0; a < MOOG_Z_N_ATTRS; ++a) {
      const int kind = pv.ipool[t + 3 * a], idx = pv.ipool[t + 3 * a + 1], n = pv.ipool[t + 3 * a + 2];
      if (kind < MOOG_ZK_CONST || kind > MOOG_ZK_DISCRETE_P || idx < 0 || n < 1 ||
          (long long)idx + (kind == MOOG_ZK_UNIFORM32 ? 2 : (kind == MOOG_ZK_DISCRETE_P ? 2 * n : n)) > ND)
        return false;
    }
    return pv.ipool[t + 3 * MOOG_Z_N_ATTRS] >= 0;
  };
  auto tree_ok = [&](int start, int n, bool rule) {  // decision tree nodes of 8 ints (MOOG_SC_TREE / MOOG_R_TREE)
    if (n < 1 || start < 0 || (long long)start + 8LL * n > NI) return false;
    for (int j = 0; j < n; ++j) {
      const int32_t *nd = pv.ipool + start + 8 * j;
      const int kind = nd[0];
      if (kind < 0 || kind > 4 || (!rule && kind == 4)) return false;
      if ((kind == 1 || kind == 4 || (kind == 0 && !rule)) && !(nd[1] >= 0 && nd[1] < NX)) return false;
      if (!(nd[2] == -1 || layer_ok(nd[2])) || !(nd[4] == -1 || layer_ok(nd[4])) || nd[3] < 0 || nd[5] < 0) return false;
      if ((kind == 2 && !(layer_ok(nd[2]) && layer_ok(nd[4]))) || (kind == 3 && !layer_ok(nd[2]))) return false;
      if (kind != 0 && !(nd[6] > j && nd[6] < n && nd[7] > j && nd[7] < n)) return false;  // forward only: the walk ends
    }
    return true;
  };
  for (int o = 0; o < NO; ++o) {
    const moog_op &op = pv.ops[o];
    bool ok = true;
    switch (op.kind) {
      case MOOG_F_DRAG: case MOOG_F_KINETIC_FRICTION: case MOOG_F_DOWN_GRAVITY: case MOOG_F_GRAVITY: case MOOG_F_RANDOM:
      case MOOG_F_DIST_LINEAR: case MOOG_F_DIST_SPRING: case MOOG_F_COLLISION: case MOOG_F_MAZE_WALK:
        ok = layer_ok(op.i[0]) && (op.i[1] == -1 || layer_ok(op.i[1]));
        if (op.kind == MOOG_F_MAZE_WALK) ok = ok && envf_ok(op.i[3], 1);
        break;
      case MOOG_C_TETHER: case MOOG_C_TETHER_ZIPPED: case MOOG_C_CONSTANT_SPEED: case MOOG_C_MAZE_PHYSICS:
        ok = list_ok(op.i[0], op.i[1], L);
        if (op.kind == MOOG_C_MAZE_PHYSICS) ok = ok && envf_ok(op.i[2], 1);
        break;
      case MOOG_R_VANISH_ON_CONTACT: case MOOG_R_PORTAL: ok = layer_ok(op.i[0]) && layer_ok(op.i[1]); break;
      case MOOG_R_VANISH_BY_FILTER: ok = layer_ok(op.i[0]) && expr_ok(op.i[2]); break;
      case MOOG_R_CHANGE_LAYER: ok = layer_ok(op.i[0]) && layer_ok(op.i[1]) && expr_ok(op.i[2]); break;
      case MOOG_R_MODIFY_ON_CONTACT:
        ok = list_ok(op.i[0], op.i[1], L) && list_ok(op.i[2], op.i[3], L) && op.i[4] >= 0 && (long long)op.i[4] + 4 <= NI;
        for (int q = 0; ok && q < 4; ++q) ok = expr_ok(pv.ipool[op.i[4] + q]);
        break;
      case MOOG_R_MODIFY_SPRITES:
        ok = list_ok(op.i[0], op.i[1], L) && expr_ok(op.i[2]) && expr_ok(op.i[3]) && op.i[4] >= 0 &&
             op.i[4] <= hdr[MOOG_H_RULE_NOISE_DIM];
        break;
      case MOOG_R_COND_BEGIN: ok = cond_ok(op.i[0]) && op.i[1] >= 0 && (long long)o + 1 + op.i[1] <= NO; break;
      case MOOG_R_TIMED_BEGIN: ok = op.i[1] >= 0 && (long long)o + 1 + op.i[1] <= NO && envf_ok(op.i[2], 2); break;
      case MOOG_R_KEEP_NEAR_CENTER: ok = layer_ok(op.i[0]) && list_ok(op.i[1], op.i[2], L); break;
      case MOOG_R_CREATE_SPRITES:
        ok = layer_ok(op.i[0]) && op.i[1] >= 0 && list_ok(op.i[2], op.i[3], L) && table_ok(op.i[4]) &&
             (!(op.p[2] > op.p[1]) || (op.p[3] >= 0 && op.p[3] < hdr[MOOG_H_RULE_NOISE_DIM]));
        break;
      case MOOG_T_CONTACT_REWARD:
        ok = list_ok(op.i[0], op.i[1], L) && list_ok(op.i[2], op.i[3], L) && expr_ok(op.i[4]) && envf_ok(op.i[5], 1) &&
             (!(op.p[2] > 0) || expr_ok((int)op.p[2] - 1));
        break;
      case MOOG_T_RESET: ok = cond_ok(op.i[0]) && envf_ok(op.i[5], 1) && (op.i[1] == 0 || cond_ok(op.i[1] - 1)); break;
      case MOOG_T_STAY_ALIVE: ok = op.p[0] >= 1; break;
      case MOOG_T_TIMEOUT: break;
      case MOOG_A_JOYSTICK: case MOOG_A_GRID: case MOOG_A_SET_POSITION:
        ok = list_ok(op.i[0], op.i[1], L) && op.i[2] >= 0 &&
             op.i[2] + (op.kind == MOOG_A_GRID ? 1 : 2) <= (hdr[MOOG_H_ACTION_DIM] > 0 ? hdr[MOOG_H_ACTION_DIM] : 1) + 1 &&
             (op.kind == MOOG_A_SET_POSITION || envf_ok(op.i[5], 2));
        break;
      case MOOG_Z_GENERATE:
        ok = op.i[0] >= 0 && op.i[1] >= 0 && (long long)op.i[0] + op.i[1] <= S && list_ok(op.i[2], op.i[3], S > 0 ? S : 1) &&
             table_ok(op.i[4]);
        break;
      case MOOG_SC_ALL: case MOOG_SC_ANY: case MOOG_SC_COUNT: case MOOG_SC_FIRST:
        ok = list_ok(op.i[0], op.i[1], L) && expr_ok(op.i[2]);
        break;
      case MOOG_SC_CONTACT_COUNT: ok = layer_ok(op.i[0]) && layer_ok(op.i[1]); break;
      case MOOG_SC_CONTACT_ANY_COUNT: ok = list_ok(op.i[0], op.i[1], L) && list_ok(op.i[2], op.i[3], L) && expr_ok(op.i[4]); break;
      case MOOG_SC_CONST: break;
      case MOOG_SC_BINARY: ok = cond_ok(op.i[0]) && cond_ok(op.i[1]); break;
      case MOOG_SC_NOT: ok = cond_ok(op.i[0]); break;
      case MOOG_SC_BERNOULLI: ok = op.i[0] >= 0 && op.i[0] < hdr[MOOG_H_RULE_NOISE_DIM]; break;
      case MOOG_R_FIXATION: ok = layer_ok(op.i[0]) && layer_ok(op.i[1]) && envf_ok(op.i[2], 1); break;
      case MOOG_R_PHASESEQ_BEGIN:
        ok = envf_ok(op.i[0], 2) && op.i[1] >= 1 && (op.i[2] == -1 || envf_ok(op.i[2], 1)) && op.i[4] >= 0 &&
             (long long)op.i[4] + op.i[1] <= ND;
        break;
      case MOOG_R_PHASE_BEGIN:
        ok = (op.i[0] == -1 || envf_ok(op.i[0], 2)) && op.i[1] >= 1 && (long long)o + 1 + op.i[1] <= NO && envf_ok(op.i[3], 3) &&
             op.i[4] >= 0 && (!(op.p[2] > op.p[1]) || op.i[4] < hdr[MOOG_H_RULE_NOISE_DIM]);
        break;
      case MOOG_R_PHASE_END:
        ok = (op.i[0] == -1 || cond_ok(op.i[0])) && envf_ok(op.i[1], 3) && (op.i[2] == -1 || envf_ok(op.i[2], 2)) &&
             (op.i[3] == -1 || envf_ok(op.i[3], 1)) && op.i[4] >= 0 && op.i[5] >= 0 && (long long)op.i[4] + op.i[5] <= ND;
        break;
      case MOOG_SC_TREE: ok = tree_ok(op.i[0], op.i[1], false); break;
      case MOOG_R_TREE:
        ok = tree_ok(op.i[0], op.i[1], true) && op.i[3] >= 0 && (op.i[3] == 0 || envf_ok(op.i[2], op.i[3])) && op.i[4] >= 0 &&
             (long long)op.i[4] + op.i[3] <= ND;
        break;
      default: ok = false; break;  // an op kind no kernel knows
    }
    if (!ok) return MOOG_E_INVAL;
  }
  if (hdr[MOOG_H_R_ENABLED]) {
    if (hdr[MOOG_H_R_HEIGHT] < 1 || hdr[MOOG_H_R_WIDTH] < 1 || hdr[MOOG_H_R_AA] < 1 || hdr[MOOG_H_R_HEIGHT] > 8192 ||
        hdr[MOOG_H_R_WIDTH] > 8192 || hdr[MOOG_H_R_AA] > 16)
      return MOOG_E_INVAL;
    if (hdr[MOOG_H_R_MODIFIER] == MOOG_PMOD_FIRST_PERSON && !layer_ok(hdr[MOOG_H_R_MOD_LAYER])) return MOOG_E_INVAL;
  }
  // views 1..: rows of the view table, each a renderer next to view 0
  const int nv = hdr[MOOG_H_N_VIEWS], vt = hdr[MOOG_H_VIEWS];
  if (nv < 0 || nv >= MOOG_MAX_VIEWS) return MOOG_E_INVAL;
  if (nv > 0) {
    if (!hdr[MOOG_H_R_ENABLED] || vt < 0 || (long long)vt + (long long)MOOG_VIEW_WORDS * nv > NI) return MOOG_E_INVAL;
    for (int k = 0; k < nv; ++k) {
      const int32_t *v = pv.ipool + vt + MOOG_VIEW_WORDS * k;
      if (v[MOOG_V_ENABLED] != 1 || v[MOOG_V_HEIGHT] < 1 || v[MOOG_V_WIDTH] < 1 || v[MOOG_V_AA] < 1 ||
          v[MOOG_V_HEIGHT] > 8192 || v[MOOG_V_WIDTH] > 8192 || v[MOOG_V_AA] > 16)
        return MOOG_E_INVAL;
      if (v[MOOG_V_COLORMAP] != MOOG_CMAP_NONE && v[MOOG_V_COLORMAP] != MOOG_CMAP_HSV) return MOOG_E_INVAL;
      if (v[MOOG_V_MODIFIER] != MOOG_PMOD_NONE && v[MOOG_V_MODIFIER] != MOOG_PMOD_FIRST_PERSON &&
          v[MOOG_V_MODIFIER] != MOOG_PMOD_TORUS)
        return MOOG_E_INVAL;
      if (v[MOOG_V_MODIFIER] == MOOG_PMOD_FIRST_PERSON && !layer_ok(v[MOOG_V_MOD_LAYER])) return MOOG_E_INVAL;
    }
  }
  // masks: rows of the mask table, with a renderer row's bounds and the words a mask fixes
  const int nm = hdr[MOOG_H_N_MASKS], mt = hdr[MOOG_H_MASKS];
  if (nm < 0 || nm > MOOG_MAX_VIEWS) return MOOG_E_INVAL;
  if (nm > 0) {
    if (mt < 0 || (long long)mt + (long long)MOOG_VIEW_WORDS * nm > NI) return MOOG_E_INVAL;
    for (int k = 0; k < nm; ++k) {
      const int32_t *m = pv.ipool + mt + MOOG_VIEW_WORDS * k;
      if (m[MOOG_V_ENABLED] != 1 || m[MOOG_V_AA] != 1 || m[MOOG_V_BG] != 0 || m[MOOG_V_COLORMAP] != MOOG_CMAP_NONE ||
          m[MOOG_V_HEIGHT] < 1 || m[MOOG_V_WIDTH] < 1 || m[MOOG_V_HEIGHT] > 8192 || m[MOOG_V_WIDTH] > 8192)
        return MOOG_E_INVAL;
      if (m[MOOG_V_MODIFIER] != MOOG_PMOD_NONE && m[MOOG_V_MODIFIER] != MOOG_PMOD_FIRST_PERSON &&
          m[MOOG_V_MODIFIER] != MOOG_PMOD_TORUS)
        return MOOG_E_INVAL;
      if (m[MOOG_V_MODIFIER] == MOOG_PMOD_FIRST_PERSON && !layer_ok(m[MOOG_V_MOD_LAYER])) return MOOG_E_INVAL;
    }
  }
  return 0;
}

int moog_mask_plan(const void *blob, size_t nbytes, int mask, int *band_rows, int *smem_bytes) {
  const int bad = moog_program_validate(blob, nbytes);
  if (bad) return bad;
  const int32_t *hdr = (const int32_t *)blob;
  if (mask < 0 || mask >= hdr[MOOG_H_N_MASKS]) return MOOG_E_INVAL;
  const int32_t *m = moog::view_of(blob).ipool + hdr[MOOG_H_MASKS] + MOOG_VIEW_WORDS * mask;
  const moog::RenderPlan plan = moog::render_plan(hdr, m);
  if (!plan.ok) return MOOG_E_UNSUPPORTED;
  if (band_rows) *band_rows = plan.rows;
  if (smem_bytes) *smem_bytes = plan.env_bytes;
  return 0;
}

int moog_render_plan(const void *blob, size_t nbytes, int view, int *chunk_rows, int *smem_bytes) {
  const int bad = moog_program_validate(blob, nbytes);
  if (bad) return bad;
  const int32_t *hdr = (const int32_t *)blob;
  if (!hdr[MOOG_H_R_ENABLED] || view < 0 || view > hdr[MOOG_H_N_VIEWS]) return MOOG_E_INVAL;
  const int32_t *v = view == 0 ? hdr + MOOG_H_R_HEIGHT
                               : moog::view_of(blob).ipool + hdr[MOOG_H_VIEWS] + MOOG_VIEW_WORDS * (view - 1);
  const moog::RenderPlan plan = moog::render_plan(hdr, v);
  if (!plan.ok) return MOOG_E_UNSUPPORTED;
  if (chunk_rows) *chunk_rows = plan.rows;
  if (smem_bytes) *smem_bytes = plan.env_bytes;
  return 0;
}

int moog_program_create(const void *blob, size_t nbytes, moog_program **out) {
  if (!out) return MOOG_E_INVAL;
  const int bad = moog_program_validate(blob, nbytes);
  if (bad) return bad;
  const int32_t *hdr = (const int32_t *)blob;
  if (hdr[MOOG_H_N_FORCES] > moog::kMaxForceOps) return MOOG_E_TOO_BIG;
  moog_program *p = (moog_program *)calloc(1, sizeof(moog_program));
  if (!p) return MOOG_E_INVAL;
  memcpy(p->hdr, hdr, sizeof(p->hdr));
  p->opt = moog::launch_options_from_env();
  p->hdr[MOOG_H_CMASK_WORDS] = moog::candidate_matrix_words(blob);
  {
    moog::ProgramView pv = moog::view_of(blob);
    for (int l = 0; l < hdr[MOOG_H_N_LAYERS]; ++l) {
      const int a = hdr[MOOG_H_LAYER_OFF + l], b = hdr[MOOG_H_LAYER_OFF + l + 1];
      p->layer_vcap[l] = b > a ? pv.voff[a + 1] - pv.voff[a] : 0;
    }
    if (hdr[MOOG_H_R_ENABLED]) {
      p->n_views = 1 + hdr[MOOG_H_N_VIEWS];
      for (int k = 0; k < p->n_views; ++k) {
        const int32_t *v = k == 0 ? hdr + MOOG_H_R_HEIGHT : pv.ipool + hdr[MOOG_H_VIEWS] + MOOG_VIEW_WORDS * (k - 1);
        memcpy(p->view[k], v, sizeof(p->view[k]));
        p->view_off[k] = (int)(v - hdr);
        p->plan[k] = moog::render_plan(p->hdr, p->view[k]);
      }
    }
    p->n_masks = hdr[MOOG_H_N_MASKS];
    for (int k = 0; k < p->n_masks; ++k) {
      const int32_t *m = pv.ipool + hdr[MOOG_H_MASKS] + MOOG_VIEW_WORDS * k;
      p->mask_off[k] = (int)(m - hdr);
      p->mask_plan[k] = moog::render_plan(p->hdr, m);
    }
  }
  if (moog::env_smem_bytes(p->hdr) > 220 * 1024 || p->hdr[MOOG_H_CMASK_WORDS] > 2048) {
    free(p);
    return MOOG_E_TOO_BIG;
  }
  p->nbytes = nbytes;
  cudaError_t err = cudaMalloc(&p->dev_blob, nbytes);
  if (err == cudaSuccess) err = cudaMemcpy(p->dev_blob, blob, nbytes, cudaMemcpyHostToDevice);
  if (err == cudaSuccess)  // the derived header word, in the device copy too
    err = cudaMemcpy((int32_t *)p->dev_blob + MOOG_H_CMASK_WORDS, &p->hdr[MOOG_H_CMASK_WORDS], sizeof(int32_t),
                     cudaMemcpyHostToDevice);
  if (err == cudaSuccess && hdr[MOOG_H_N_VTX] > 0) {
    moog::ProgramView pv = moog::view_of(blob);
    std::vector<uint16_t> vmap((size_t)hdr[MOOG_H_N_VTX], 0xffffu);
    for (int sl = 0; sl < hdr[MOOG_H_N_SLOTS]; ++sl)
      for (int v = pv.voff[sl]; v < pv.voff[sl + 1] && v < hdr[MOOG_H_N_VTX]; ++v) {
        const int k = v - pv.voff[sl];
        vmap[(size_t)v] = (uint16_t)((sl << 8) | (k < 255 ? k : 255));  // (MOOG_MAX_OUTLINE = 128 < 255)
      }
    err = cudaMalloc((void **)&p->dev_vmap, sizeof(uint16_t) * vmap.size());
    if (err == cudaSuccess)
      err = cudaMemcpy(p->dev_vmap, vmap.data(), sizeof(uint16_t) * vmap.size(), cudaMemcpyHostToDevice);
  }
  if (err != cudaSuccess) {
    if (p->dev_blob) cudaFree(p->dev_blob);
    if (p->dev_vmap) cudaFree(p->dev_vmap);
    free(p);
    return cuda_fail(err);
  }
  *out = p;
  return 0;
}

void moog_program_destroy(moog_program *p) {
  if (!p) return;
  if (p->dev_blob) cudaFree(p->dev_blob);
  if (p->dev_vmap) cudaFree(p->dev_vmap);
  if (p->sched) cudaFree(p->sched);
  if (p->done) cudaFree(p->done);
  for (int k = 0; k < MOOG_MAX_VIEWS; ++k)
    if (p->resample[k]) cudaFree(p->resample[k]);
  free(p);
}

int moog_program_env_smem_bytes(const moog_program *p) { return p ? moog::env_smem_bytes(p->hdr) : MOOG_E_INVAL; }

static int sm_count() {
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return sms;
}

// what moog_env_step with frames does with a batch of n_envs on the current device
static moog::StepPlan env_step_plan(const moog_program *p, int n_envs) {
  return moog::plan_step(p->hdr, moog::MODE_ENV_STEP, n_envs, true, sm_count(), p->opt);
}

int moog_program_set_option(moog_program *p, const char *name, int value) {
  if (!p || !moog::set_launch_option(p->opt, name, value)) return MOOG_E_INVAL;
  return 0;
}

int moog_step_launch_info(const moog_program *p, int n_envs, int *resident_envs_per_sm, int *warps_per_env,
                          int *smem_bytes_per_env) {
  if (!p || n_envs < 0) return MOOG_E_INVAL;
  const moog::StepPlan plan = env_step_plan(p, n_envs);
  if (resident_envs_per_sm) *resident_envs_per_sm = plan.resident;
  if (warps_per_env) *warps_per_env = plan.helper ? 2 : 1;
  if (smem_bytes_per_env) *smem_bytes_per_env = moog::env_smem_bytes(p->hdr, plan.helper);
  return 0;
}

int moog_step_draws_frames(const moog_program *p, int n_envs) {
  if (!p || n_envs < 0) return MOOG_E_INVAL;
  return env_step_plan(p, n_envs).fuse ? 1 : 0;
}

static int render_impl(moog_program *p, const moog_state *st, int n_envs, int view, uint8_t *frames, void *stream,
                       int *done, long long *trace = nullptr);

static int run_step(moog_program *p, const moog_state *st, int n_envs, int mode, const moog_step_io *io,
                    int layer_a, int layer_b, uint8_t *overlap_out, void *stream) {
  if (!p || !valid_state(st) || n_envs < 0) return MOOG_E_INVAL;
  moog::StepArgs a;
  memset(&a, 0, sizeof(a));
  a.blob = p->dev_blob;
  a.vmap = p->dev_vmap;
  a.st = *st;
  a.n_envs = n_envs;
  a.mode = mode;
  if (io) a.io = *io;
  if (a.io.pool) {
    if (!valid_state(a.io.pool) || a.io.pool_size <= 0) return MOOG_E_INVAL;
    a.pool = *a.io.pool;
  }
  a.layer_a = layer_a;
  a.layer_b = layer_b;
  a.overlap_out = overlap_out;
  if (a.io.frames && (mode != moog::MODE_ENV_STEP || !p->hdr[MOOG_H_R_ENABLED] || p->hdr[MOOG_H_R_AA] < 1))
    return MOOG_E_INVAL;
  // a view no chunk size can hold is refused before anything is launched
  if (a.io.frames && !p->plan[0].ok) return MOOG_E_UNSUPPORTED;
  const moog::StepPlan plan = moog::plan_step(p->hdr, mode, n_envs, a.io.frames != nullptr, sm_count(), p->opt);
  int launches = 0;
  cudaError_t err = cudaSuccess;
  if (plan.ordered) {
    if (p->sched_cap < n_envs) {
      if (p->sched) cudaFree(p->sched);
      p->sched = nullptr;
      p->sched_cap = 0;
      err = cudaMalloc((void **)&p->sched, sizeof(int) * 2 * (size_t)n_envs);
      if (err != cudaSuccess) return cuda_fail(err);
      p->sched_cap = n_envs;
      p->sched_state = nullptr;
    }
    int *cost = p->sched, *order = p->sched + p->sched_cap;
    if (p->sched_state != (const void *)st->dyn) {  // another batch: no history yet
      err = cudaMemsetAsync(cost, 0, sizeof(int) * (size_t)n_envs, (cudaStream_t)stream);
      if (err != cudaSuccess) return cuda_fail(err);
      p->sched_state = (const void *)st->dyn;
    }
    err = moog::launch_order(cost, order, n_envs, (cudaStream_t)stream, &launches);
    if (err != cudaSuccess) return cuda_fail(err);
    a.order = order;
    a.cost = cost;
  }
  if (plan.tail) {
    if (p->done_cap < n_envs) {
      if (p->done) cudaFree(p->done);
      p->done = nullptr;
      p->done_cap = 0;
      err = cudaMalloc((void **)&p->done, sizeof(int) * (1 + (size_t)n_envs + moog::kTailExtraInts));
      if (err != cudaSuccess) return cuda_fail(err);
      p->done_cap = n_envs;
    }
    // count, finished list [n_envs], ticket, envs being stepped per SM [256]
    err = cudaMemsetAsync(p->done, 0, sizeof(int) * (1 + (size_t)n_envs + moog::kTailExtraInts), (cudaStream_t)stream);
    if (err != cudaSuccess) return cuda_fail(err);
    a.done = p->done;
    a.sm_active = p->done + 1 + n_envs + 1;
  }
  a.trace = (p->opt.trace_times != 0 && a.io.counters) ? 1 : 0;  // diagnostic: per-env timeline in io.counters
  err = moog::launch_step(a, p->hdr, plan, (cudaStream_t)stream, &launches);
  g_launches += launches;
  if (err != cudaSuccess) return cuda_fail(err);
  if (a.io.frames && !plan.fuse)
    return render_impl(p, st, n_envs, 0, a.io.frames, stream, a.done, a.trace ? (long long *)a.io.counters : nullptr);
  return 0;
}

int moog_env_step(moog_program *p, const moog_state *st, int n_envs, const moog_step_io *io, void *stream) {
  return run_step(p, st, n_envs, moog::MODE_ENV_STEP, io, 0, 0, nullptr, stream);
}

int moog_env_post_reset(moog_program *p, const moog_state *st, int n_envs, const double *rule_noise,
                        void *stream) {
  moog_step_io io;
  memset(&io, 0, sizeof(io));
  io.rule_noise = rule_noise;
  if (p) io.seed = (uint64_t)(uint32_t)p->opt.seed;
  return run_step(p, st, n_envs, moog::MODE_POST_RESET, &io, 0, 0, nullptr, stream);
}

int moog_physics_step(moog_program *p, const moog_state *st, int n_envs, const double *noise, int64_t *counters,
                      void *stream) {
  moog_step_io io;
  memset(&io, 0, sizeof(io));
  io.noise = noise;
  io.counters = counters;
  return run_step(p, st, n_envs, moog::MODE_PHYSICS, &io, 0, 0, nullptr, stream);
}

int moog_overlap_pairs(moog_program *p, const moog_state *st, int n_envs, int layer_a, int layer_b, uint8_t *out,
                       void *stream) {
  if (!p || !out) return MOOG_E_INVAL;
  int L = p->hdr[MOOG_H_N_LAYERS];
  if (layer_a < 0 || layer_a >= L || layer_b < 0 || layer_b >= L) return MOOG_E_INVAL;
  // outlines beyond MOOG_MAX_VERTS are draw-only: the overlap kernels spend one lane per vertex
  if (p->layer_vcap[layer_a] > MOOG_MAX_VERTS || p->layer_vcap[layer_b] > MOOG_MAX_VERTS) return MOOG_E_UNSUPPORTED;
  return run_step(p, st, n_envs, moog::MODE_OVERLAP, nullptr, layer_a, layer_b, out, stream);
}

int moog_render(moog_program *p, const moog_state *st, int n_envs, uint8_t *frames, void *stream) {
  return render_impl(p, st, n_envs, 0, frames, stream, nullptr);
}

int moog_render_view(moog_program *p, const moog_state *st, int n_envs, int view, uint8_t *frames, void *stream) {
  if (!p || !frames || ((uintptr_t)frames & 15) || view < 0 || view >= p->n_views) return MOOG_E_INVAL;
  return render_impl(p, st, n_envs, view, frames, stream, nullptr);
}

static int render_impl(moog_program *p, const moog_state *st, int n_envs, int view, uint8_t *frames, void *stream,
                       int *done, long long *trace) {
  if (!p || !valid_state(st) || !frames || n_envs < 0) return MOOG_E_INVAL;
  if (!p->hdr[MOOG_H_R_ENABLED]) return MOOG_E_INVAL;
  const int32_t *v = p->view[view];
  if (v[MOOG_V_AA] < 1 || !p->plan[view].ok) return MOOG_E_UNSUPPORTED;
  moog::RenderArgs a;
  memset(&a, 0, sizeof(a));
  a.blob = p->dev_blob;
  a.view_off = p->view_off[view];
  a.st = *st;
  a.n_envs = n_envs;
  a.frames = frames;
  a.trace = trace;
  if (v[MOOG_V_AA] > 1) {
    if (!p->resample[view]) {
      const int OH = v[MOOG_V_HEIGHT], OW = v[MOOG_V_WIDTH], aa = v[MOOG_V_AA];
      std::vector<int> table;
      int n = moog::resample_tables(aa * OH, aa * OW, OH, OW, table, &p->ksize_h[view], &p->ksize_v[view]);
      cudaError_t err = cudaMalloc((void **)&p->resample[view], sizeof(int) * (size_t)n);
      if (err == cudaSuccess)
        err = cudaMemcpy(p->resample[view], table.data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice);
      if (err != cudaSuccess) {  // never keep a table that was not filled
        if (p->resample[view]) cudaFree(p->resample[view]);
        p->resample[view] = nullptr;
        return cuda_fail(err);
      }
    }
    a.resample = p->resample[view];
    a.ksize_h = p->ksize_h[view];
    a.ksize_v = p->ksize_v[view];
  }
  int launches = 0;
  cudaError_t err = moog::launch_render(a, p->plan[view], v, (cudaStream_t)stream, &launches, done, n_envs);
  g_launches += launches;
  return err == cudaSuccess ? 0 : cuda_fail(err);
}

int moog_render_mask(moog_program *p, const moog_state *st, int n_envs, int mask, int16_t *out, void *stream) {
  if (!p || !valid_state(st) || !out || n_envs < 0 || ((uintptr_t)out & 15) || mask < 0 || mask >= p->n_masks)
    return MOOG_E_INVAL;
  if (!p->mask_plan[mask].ok) return MOOG_E_UNSUPPORTED;
  moog::RenderArgs a;
  memset(&a, 0, sizeof(a));
  a.blob = p->dev_blob;
  a.view_off = p->mask_off[mask];
  a.st = *st;
  a.n_envs = n_envs;
  a.frames = (uint8_t *)out;
  int launches = 0;
  cudaError_t err = moog::launch_mask(a, p->mask_plan[mask], (cudaStream_t)stream, &launches);
  g_launches += launches;
  return err == cudaSuccess ? 0 : cuda_fail(err);
}

int moog_observe_sprites(moog_program *p, const moog_state *st, int n_envs, float *out, void *stream) {
  if (!p || !valid_state(st) || !out || n_envs < 0 || ((uintptr_t)out & 15)) return MOOG_E_INVAL;
  if (n_envs == 0) return 0;
  moog::ObserveArgs a;
  memset(&a, 0, sizeof(a));
  a.st = *st;
  a.out = out;
  a.n_envs = n_envs;
  a.S = p->hdr[MOOG_H_N_SLOTS];
  a.L = p->hdr[MOOG_H_N_LAYERS];
  memcpy(a.layer_off, &p->hdr[MOOG_H_LAYER_OFF], sizeof(a.layer_off));
  int launches = 0;
  cudaError_t err = moog::launch_observe(a, (cudaStream_t)stream, &launches);
  g_launches += launches;
  return err == cudaSuccess ? 0 : cuda_fail(err);
}

int moog_ray_sensor(moog_program *p, const moog_state *st, int n_envs, const moog_ray_spec *spec, float *out,
                    void *stream) {
  if (!p || !valid_state(st) || !spec || !spec->dirs || !out || n_envs < 0 || ((uintptr_t)out & 15) ||
      ((uintptr_t)spec->dirs & 7))
    return MOOG_E_INVAL;
  const int L = p->hdr[MOOG_H_N_LAYERS];
  if (spec->n_rays < 1 || spec->n_rays > 256 || !isfinite(spec->max_range) || !(spec->max_range > 0.0) ||
      spec->agent_layer < 0 || spec->agent_layer >= L || spec->agent_index < 0 ||
      (L < 32 && (spec->layers >> L) != 0))
    return MOOG_E_INVAL;
  if (n_envs == 0) return 0;
  moog::RayArgs a;
  memset(&a, 0, sizeof(a));
  a.blob = p->dev_blob;
  a.st = *st;
  a.out = out;
  a.dirs = spec->dirs;
  a.max_range = spec->max_range;
  a.n_envs = n_envs;
  a.S = p->hdr[MOOG_H_N_SLOTS];
  a.L = L;
  a.VT = p->hdr[MOOG_H_N_VTX];
  a.n_rays = spec->n_rays;
  a.agent_layer = spec->agent_layer;
  a.agent_index = spec->agent_index;
  a.layers = spec->layers;
  memcpy(a.layer_off, &p->hdr[MOOG_H_LAYER_OFF], sizeof(a.layer_off));
  int launches = 0;
  cudaError_t err = moog::launch_ray_sensor(a, (cudaStream_t)stream, &launches);
  g_launches += launches;
  return err == cudaSuccess ? 0 : cuda_fail(err);
}

const char *moog_strerror(int code) {
  switch (code) {
    case 0: return "ok";
    case MOOG_E_INVAL: return "invalid argument or malformed program blob";
    case MOOG_E_CUDA: return "CUDA runtime error";
    case MOOG_E_TOO_BIG: return "one env record does not fit in shared memory";
    case MOOG_E_UNSUPPORTED: return "configuration not supported by the device path yet";
  }
  return "unknown error";
}

const char *moog_last_cuda_error(void) { return g_cuda_error.c_str(); }

int64_t moog_launch_count(void) { return g_launches.load(); }

}  // extern "C"
