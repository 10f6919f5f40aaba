"""`_directed_collision_vectors` (collisions.py:101-232) on hand-built scenes: the CUDA search
(csrc/moog_step.cu directed_collision_vectors_impl) against the oracle, bit for bit after every
step, with the helper warp (32-vertex tiles) and without it (8-vertex tiles).

The search compacts the crossing (contained vertex, edge) pairs into a list and takes np.argmin per
vertex by a segmented scan over 32 pairs at a time.  Each scene is there for one of the cases that
scan has to get right; `test_scenes_reach_their_cases` checks, with a numpy restatement of the
crossing test, that the scene's first substep really contains it:

    deep30, deep32   more than 32 crossing pairs in one search (30-gon and 32-gon outlines); with
                     slow relative motion the vertices cross varying numbers of edges, so segments
                     straddle passes
    resting          zero relative motion: every edge crosses and the denominator is EPS_INTERP only
    corner_tie       the motion starts exactly on a reflex vertex of the outline: cross_a is 0 on both
                     edges that meet there, equal keys, and the lower edge (whose normal differs from
                     the other's) must win
    wall             a ball against a 4-vertex wall (8 vertices x 4 edges per lane tile)
    overflow         coordinates near 1e155: NaN coefficients (NaN wins np.argmin), and contained
                     vertices without any crossing pair next to ones that have one
"""
import collections

import numpy as np
import pytest

from tests import util

K = 4
STEPS = 6
N_ENVS = 16


def _ngon(n):
    t = np.arange(n) * (2 * np.pi / n)
    return np.stack([0.5 * np.cos(t), 0.5 * np.sin(t)], axis=1)


def _variants(scene):
    """-> list of (sprites of layer a, sprites of layer b), one per pool state."""
    import moog_b200  # noqa: F401  (the MOOG-compatible `moog` package)
    from moog import sprite
    S = sprite.Sprite
    rng = np.random.RandomState(11)
    out = []
    if scene in ('deep30', 'deep32', 'resting'):
        shape = _ngon(32) if scene == 'deep32' else 'circle'
        for k in range(8):
            # a smaller outline almost inside a larger one: every vertex of `a` is contained
            v = 10 ** rng.uniform(-6.5, -2) * (rng.uniform(size=2) - 0.5)
            b_vel = v if scene == 'resting' and k % 2 else np.zeros(2)
            if scene == 'resting' and k % 2 == 0:
                v = np.zeros(2)
            a = S(x=0.5, y=0.5, shape=shape, scale=0.17, angle=rng.uniform(0, 1), x_vel=v[0], y_vel=v[1])
            b = S(x=0.5 + rng.uniform(-0.004, 0.004), y=0.5 + rng.uniform(-0.004, 0.004), shape=shape,
                  scale=0.2, x_vel=b_vel[0], y_vel=b_vel[1])
            out.append(([a], [b]))
    elif scene == 'corner_tie':
        notch = np.array([(0.25, 0.25), (0.75, 0.25), (0.75, 0.75), (0.5, 0.5), (0.25, 0.75)])  # reflex vertex 3
        for d in (2.0 ** -12, 2.0 ** -13, 2.0 ** -10):
            # the tip of `a` is d left of the reflex vertex and moves left by d per substep (dt = 1/4), so the
            # relative trajectory starts exactly on that vertex
            tip = np.array([(0.5 - d, 0.5), (0.55, 0.7), (0.45, 0.7)])
            out.append(([S(x=0, y=0, shape=tip, x_vel=-4 * d)], [S(x=0, y=0, shape=notch)]))
    elif scene == 'wall':
        floor = np.array([[-1, 0.1], [2, 0.1], [2, -1], [-1, -1]])
        for k in range(8):
            v = 10 ** rng.uniform(-6.5, -1.5)
            a = S(x=rng.uniform(0.2, 0.8), y=0.1 + rng.uniform(-0.04, 0.03), shape='circle', scale=0.1,
                  x_vel=rng.uniform(-1, 1) * v, y_vel=-v)
            out.append(([a], [S(x=0, y=0, shape=floor)]))
    elif scene == 'overflow':
        # (scale of the circle `a`, its velocity, position and scale of the square `b`): found with the
        # restatement below; each search has NaN coefficients and contained vertices without a crossing pair
        for sa, va, pb, sb in [
                (2.59385359013712e+155, (6.967826412030912e+152, 5.297583208695557e+152),
                 (5.1494401427452503e+154, -8.551766298432266e+154), 1.233001316581281e+156),
                (2.59385359013712e+155, (-6.967826412030912e+152, 5.297583208695557e+152),
                 (-5.1494401427452503e+154, -8.551766298432266e+154), 1.233001316581281e+156)]:
            with np.errstate(over='ignore'):   # (the inertia and circumradius of such outlines overflow)
                out.append(([S(x=0., y=0., shape='circle', scale=sa, x_vel=va[0], y_vel=va[1])],
                            [S(x=pb[0], y=pb[1], shape='square', scale=sb)]))
    else:
        raise KeyError(scene)
    return out


SCENES = ['deep30', 'deep32', 'resting', 'corner_tie', 'wall', 'overflow']


def _config(scene):
    import moog_b200  # noqa: F401
    from moog import action_spaces, physics as phys, tasks
    variants = _variants(scene)
    states = [collections.OrderedDict(a=a, b=b, agent=[]) for a, b in variants]
    bounce = phys.Collision(elasticity=0.6, symmetric=False, update_angle_vel=False, max_recursion_depth=2)
    cfg = dict(state_initializer=lambda: states[0], physics=phys.Physics((bounce, 'a', ['b']), updates_per_env_step=K),
               task=tasks.CompositeTask(timeout_steps=100), action_space=action_spaces.Grid(action_layers='agent'),
               observers={}, game_rules=())
    return cfg, states


def _crossings(a, b, dt):
    """sprite.py:145-175 / collisions.py:150-180 for the directed search (a's vertices in b) at a's
    current position: [(vertex, [(edge, cross_a) of every crossing pair])] per contained vertex."""
    P0, P1 = a.vertices, b.vertices
    inside = b.contains_points(P0)
    rel = np.array([b.x_vel, b.y_vel]) * dt + (-1.0 * np.array([a.x_vel, a.y_vel]) * dt + 0.0)
    n1 = len(P1)
    out = []
    with np.errstate(all='ignore'):
        for i in np.nonzero(inside)[0]:
            e = P0[i]
            s = e + rel
            d0 = e - s
            rows = []
            for j in range(n1):
                w1, w2 = P1[j], P1[(j + 1) % n1]
                e1, q = w2 - w1, w1 - s
                den = (d0[0] * e1[1] - d0[1] * e1[0]) + 1e-8
                cb = (q[0] * d0[1] - q[1] * d0[0]) / den
                if 0 <= cb <= 1:
                    rows.append((j, (q[0] * e1[1] - q[1] * e1[0]) / den))
            out.append((i, rows))
    return out


def _open_tail_outruns_pass(seg):
    """Some pass of 32 pairs ends inside a segment whose part in that pass is longer than every
    segment that closes in the pass: the scan has to run as long as that open tail."""
    start = np.cumsum([0] + list(seg))[:-1]
    for base in range(0, sum(seg), 32):
        closed = [min(s + n, base + 32) - max(s, base) for s, n in zip(start, seg)
                  if n and s < base + 32 and s + n > base and s + n <= base + 32]
        tail = [base + 32 - max(s, base) for s, n in zip(start, seg) if n and s < base + 32 < s + n]
        if tail and tail[0] > max(closed, default=0):
            return True
    return False


def test_scenes_reach_their_cases():
    seen = collections.defaultdict(int)
    for scene in SCENES:
        for a, b in _variants(scene):
            res = _crossings(a[0], b[0], 1.0 / K)
            seg = [len(r) for _, r in res]
            start = np.cumsum([0] + seg)[:-1]
            if sum(seg) > 32:
                seen[scene, 'more than 32 pairs'] += 1
            if any(s // 32 != (s + n - 1) // 32 for s, n in zip(start, seg) if n):
                seen[scene, 'segment straddles a pass'] += 1
            if _open_tail_outruns_pass(seg):
                seen[scene, 'straddling tail longer than the closed segments of its pass'] += 1
            if a[0].x_vel == b[0].x_vel and a[0].y_vel == b[0].y_vel:
                seen[scene, 'zero relative motion'] += 1
            if len(b[0].vertices) == 4:
                seen[scene, 'E = 4'] += 1
            if 0 in seg and sum(seg):
                seen[scene, 'vertex without a crossing pair'] += 1
            for _, rows in res:
                keys = [-1.0 if np.isnan(A) else abs(1.0 - A) for _, A in rows]
                if any(np.isnan(A) for _, A in rows):
                    seen[scene, 'NaN coefficient'] += 1
                if keys and min(keys) >= 0 and keys.count(min(keys)) > 1:
                    seen[scene, 'equal keys'] += 1
    for case in [('deep30', 'more than 32 pairs'), ('deep30', 'segment straddles a pass'),
                 ('deep32', 'more than 32 pairs'), ('deep32', 'segment straddles a pass'),
                 ('deep32', 'straddling tail longer than the closed segments of its pass'),
                 ('resting', 'zero relative motion'), ('resting', 'segment straddles a pass'),
                 ('corner_tie', 'equal keys'), ('wall', 'E = 4'),
                 ('overflow', 'NaN coefficient'), ('overflow', 'vertex without a crossing pair')]:
        assert seen[case] > 0, case


@pytest.mark.gpu
@pytest.mark.parametrize('helper', ['1', '0'])
@pytest.mark.parametrize('scene', SCENES)
def test_directed_search_matches_oracle(scene, helper, monkeypatch):
    pytest.importorskip('torch')
    from moog_b200.batched_env import BatchedEnvironment
    from oracle.oracle import Oracle
    monkeypatch.setenv('MOOG_HELPER', helper)
    cfg, states = _config(scene)
    env = BatchedEnvironment(**cfg, num_envs=N_ENVS, device='cuda:0', seed=5, initial_states=states)
    env.reset()
    eng, prog = env.engine, env.program
    start = eng.state.download()
    orc = Oracle(prog, {k: start[k] for k in util.STATE_KEYS})
    actions = np.zeros((N_ENVS, 1))
    for t in range(STEPS):
        env.step(actions)
        r_ref, _ = orc.step(actions)
        dev = eng.state.download()
        assert np.array_equal(dev['cnt'], orc.cnt), (scene, t)
        for e in range(N_ENVS):
            live = util.live_mask(prog, orc.cnt[e])
            for k in ('dyn', 'stat'):
                assert util.rel_err(dev[k][e][:, live], getattr(orc, k)[e][:, live]) == 0.0, (scene, t, e, k)
            vlive = util.live_vertex_mask(prog, orc.cnt[e], orc.meta[e])
            assert util.rel_err(dev['vtx'][e][vlive], orc.vtx[e][vlive]) == 0.0, (scene, t, e, 'vtx')
            assert np.array_equal(util.canonical_meta(dev['meta'][e], live),
                                  util.canonical_meta(orc.meta[e], live)), (scene, t, e, 'meta')
        assert np.array_equal(eng.reward.cpu().numpy(), r_ref.astype(np.float32)), (scene, t)


_PROBE_CU = r'''
#include "moog_dcv_argmin.cuh"
#include <cuda_runtime.h>
// stage B alone on one warp: pairs (vertex t, edge ed, cross_a A) in ascending (vertex, edge) order
__global__ void dcv_argmin_probe(const int *t, const int *ed, const double *A, int n, int *out_ed, double *out_a) {
  const int lane = threadIdx.x;
  out_a[lane] = -INFINITY;
  out_ed[lane] = 0;
  __syncwarp();
  moog::DcvCarry carry;
  for (int base = 0; base < n; base += 32) {
    const int k = base + lane;
    const bool act = k < n;
    const int t_after = base + 32 < n ? t[base + 32] : 255;
    int w_ed;
    double w_a;
    if (moog::dcv_argmin_pass(act, t[act ? k : 0], ed[act ? k : 0], A[act ? k : 0], t_after, lane, carry, w_ed, w_a)) {
      out_a[t[k]] = w_a;
      out_ed[t[k]] = w_ed;
    }
  }
}
extern "C" int dcv_argmin_run(const int *t, const int *ed, const double *A, int n, int *out_ed, double *out_a) {
  int *dt, *de, *doe;
  double *da, *doa;
  cudaMalloc(&dt, 4 * (n + 1)); cudaMalloc(&de, 4 * (n + 1)); cudaMalloc(&da, 8 * (n + 1));
  cudaMalloc(&doe, 4 * 32); cudaMalloc(&doa, 8 * 32);
  cudaMemcpy(dt, t, 4 * n, cudaMemcpyHostToDevice);
  cudaMemcpy(de, ed, 4 * n, cudaMemcpyHostToDevice);
  cudaMemcpy(da, A, 8 * n, cudaMemcpyHostToDevice);
  dcv_argmin_probe<<<1, 32>>>(dt, de, da, n, doe, doa);
  cudaMemcpy(out_ed, doe, 4 * 32, cudaMemcpyDeviceToHost);
  cudaMemcpy(out_a, doa, 8 * 32, cudaMemcpyDeviceToHost);
  cudaFree(dt); cudaFree(de); cudaFree(da); cudaFree(doe); cudaFree(doa);
  return (int)cudaGetLastError();
}
'''


@pytest.fixture(scope='module')
def dcv_argmin_probe(tmp_path_factory):
    """Stage B of the search (csrc/moog_dcv_argmin.cuh) compiled on its own, with the library's flags."""
    import ctypes
    import subprocess
    from moog_b200 import build
    d = tmp_path_factory.mktemp('dcv_argmin')
    src, lib = d / 'probe.cu', d / 'probe.so'
    src.write_text(_PROBE_CU)
    subprocess.check_call([build._nvcc()] + build.NVCC_FLAGS + ['-I', build.CSRC, '-shared', '-o', str(lib), str(src)])
    L = ctypes.CDLL(str(lib))
    L.dcv_argmin_run.restype = ctypes.c_int

    def run(t, ed, A):
        t, ed = np.ascontiguousarray(t, dtype=np.int32), np.ascontiguousarray(ed, dtype=np.int32)
        A = np.ascontiguousarray(A, dtype=np.float64)
        oe, oa = np.zeros(32, dtype=np.int32), np.zeros(32, dtype=np.float64)
        ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        assert L.dcv_argmin_run(ptr(t), ptr(ed), ptr(A), len(t), ptr(oe), ptr(oa)) == 0
        return oe, oa
    return run


def _argmin_case(rng, nv, n1, counts, values):
    """Pairs of nv vertices (counts[v] crossing edges of n1 each) with cross_a drawn from `values`."""
    t, ed, A = [], [], []
    for v in range(nv):
        edges = np.sort(rng.choice(n1, size=counts[v], replace=False))
        t += [v] * len(edges)
        ed += edges.tolist()
        A += rng.choice(values, size=len(edges)).tolist()
    return np.array(t, dtype=np.int32), np.array(ed, dtype=np.int32), np.array(A), n1


@pytest.mark.gpu
def test_stage_b_is_np_argmin(dcv_argmin_probe):
    """np.argmin(|1 - row|) of every vertex's row (-inf where an edge does not cross) against stage B,
    edge and cross_a bit for bit, on pair lists of up to 1024 pairs: short closed segments followed by
    a long one that straddles a pass, full rows, NaN, +-inf and tied coefficients."""
    rng = np.random.RandomState(3)
    cases = []
    # 2 pairs, then a vertex with all 32 edges from lane 2 on: its minimum lies in the lanes a scan
    # sized by the closed segments alone would not reach
    A1 = np.full(32, 7.0)
    A1[3] = 0.5
    cases.append((np.array([0, 0] + [1] * 32), np.array([3, 9] + list(range(32))), np.r_[[3.0, 4.0], A1], 32))
    spread = np.r_[rng.normal(0, 5, 50), 1.0, 0.0, -0.0, 2.0, 1.5, 0.5, np.nan, np.inf, -np.inf, 1e300]
    ties = np.array([0.5, 1.5, 3.0, -1.0, 1.0, np.nan, np.inf, -np.inf])
    for k in range(400):
        n1 = int(rng.choice([4, 8, 16, 30, 32]))
        nv = int(rng.randint(1, 33))
        mode = k % 4
        if mode == 0:
            counts = rng.randint(0, 4, size=nv)                       # a line crosses a convex outline twice
        elif mode == 1:
            counts = rng.randint(0, n1 + 1, size=nv)                  # slow motion: any number of edges
        elif mode == 2:
            counts = np.full(nv, n1)                                  # zero relative motion: every edge
        else:
            counts = np.where(rng.uniform(size=nv) < 0.3, n1, rng.randint(0, 3, size=nv))
        cases.append(_argmin_case(rng, nv, n1, counts, ties if k % 3 == 0 else spread))
    for t, ed, A, n1 in cases:
        got_e, got_a = dcv_argmin_probe(t, ed, A)
        for v in range(int(t.max()) + 1 if len(t) else 0):
            row = np.full(n1, -np.inf)
            row[ed[t == v]] = A[t == v]
            with np.errstate(invalid='ignore'):
                i = int(np.argmin(np.abs(1.0 - row)))
            assert got_e[v] == i, (v, n1, len(t))
            assert got_a[v:v + 1].view(np.int64)[0] == row[i:i + 1].view(np.int64)[0], (v, n1, len(t), got_a[v], row[i])
