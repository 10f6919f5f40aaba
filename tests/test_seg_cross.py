"""The outline test's range decision without division (csrc/moog_seg_cross.cuh).

`segments_intersect` (csrc/moog_step.cu) decides matplotlib's four range tests on u = fl(n / den)
-- u > 0 || isclose_(u, 0) and u < 1 || isclose_(u, 1) -- from n and den alone, and divides only
for operands outside that decision's exact regime or inside the bands around its cut-offs
(-1e-13 and 1 + 1e-10).  Here the header is compiled on its own, with the library's flags, and
compared with the division on the same device on operands a few ulps either side of every cut-off
and band edge, across exponents, with +-0, subnormals, +-inf and NaN; then a designed relation puts
a vertex of b at those cut-offs of an edge of a and goes through `moog_overlap_pairs` against the
oracle.
"""
from fractions import Fraction

import numpy as np
import pytest

from tests import test_overlap_random as tor

_PROBE_CU = r'''
#include "moog_seg_cross.cuh"
#include <cuda_runtime.h>
__device__ bool isclose_ref(double a, double b) { return fabs(a - b) <= fmax(1e-10 * fmax(fabs(a), fabs(b)), 1e-13); }
// per operand pair: bit 0 seg_param_in_unit, bit 1 its `exact`, bit 2 the division form,
// bit 3 unit_ratio, bit 4 its `exact`, bit 5 fl(n / d) in [0, 1] by division
__global__ void seg_cross_probe(const double *n, const double *d, int count, int *out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  bool ex, ex2;
  const bool r = moog::seg_param_in_unit(n[i], d[i], ex);
  const double u = n[i] / d[i];
  const bool ref = (u > 0.0 || isclose_ref(u, 0.0)) && (u < 1.0 || isclose_ref(u, 1.0));
  const bool r2 = moog::unit_ratio(n[i], d[i], ex2);
  out[i] = r | ex << 1 | ref << 2 | r2 << 3 | ex2 << 4 | (u >= 0.0 && u <= 1.0) << 5;
}
extern "C" int seg_cross_run(const double *n, const double *d, int count, int *out) {
  double *dn, *dd;
  int *dout;
  cudaMalloc(&dn, 8 * count); cudaMalloc(&dd, 8 * count); cudaMalloc(&dout, 4 * count);
  cudaMemcpy(dn, n, 8 * count, cudaMemcpyHostToDevice);
  cudaMemcpy(dd, d, 8 * count, cudaMemcpyHostToDevice);
  seg_cross_probe<<<(count + 255) / 256, 256>>>(dn, dd, count, dout);
  cudaMemcpy(out, dout, 4 * count, cudaMemcpyDeviceToHost);
  cudaFree(dn); cudaFree(dd); cudaFree(dout);
  return (int)cudaGetLastError();
}
'''


@pytest.fixture(scope='module')
def seg_cross_probe(tmp_path_factory):
    """csrc/moog_seg_cross.cuh compiled on its own, with the library's flags."""
    import ctypes
    import subprocess
    from moog_b200 import build
    d = tmp_path_factory.mktemp('seg_cross')
    src, lib = d / 'probe.cu', d / 'probe.so'
    src.write_text(_PROBE_CU)
    subprocess.check_call([build._nvcc()] + build.NVCC_FLAGS + ['-I', build.CSRC, '-shared', '-o', str(lib), str(src)])
    L = ctypes.CDLL(str(lib))
    L.seg_cross_run.restype = ctypes.c_int

    def run(n, den):
        n, den = np.ascontiguousarray(n, dtype=np.float64), np.ascontiguousarray(den, dtype=np.float64)
        out = np.zeros(len(n), dtype=np.int32)
        ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        assert L.seg_cross_run(ptr(n), ptr(den), len(n), ptr(out)) == 0
        return out
    return run


def _ulps(x, k):
    """x and its k nearest doubles either side."""
    out, lo, hi = [x], x, x
    for _ in range(k):
        lo, hi = np.nextafter(lo, -np.inf), np.nextafter(hi, np.inf)
        out += [lo, hi]
    return out


def operands():
    """(n, den): n a few ulps either side of cut-off * den for every cut-off and band edge, in both signs
    of den, across exponents of den; then the special values against each other."""
    cuts = [0.0, -1e-13, -2.0 ** -44, -2.0 ** -43, 1.0, 1.0 + 1e-10, 1.0 + 2.0 ** -34, 1.0 + 2.0 ** -33, 2.0,
            -0.5, 0.5, 3.0, -3.0, 1e-300, -1e-300, 1e250, -1e250]
    dens = []
    for e in list(range(-60, 40, 3)) + [-44, -43, 33, 60, 200, 900, 1000, 1023]:
        for m in (1.0, 1.3, 1.7, 1.9999999):
            dens.append(np.ldexp(m, e))
    dens += list(_ulps(2.0 ** -44, 2)) + [1e-13]
    n, d = [], []
    with np.errstate(over='ignore'):        # cut-off * den past the largest double: inf, one more special value
        for den, s, c in ((den, s, c) for den in dens for s in (1.0, -1.0) for c in cuts):
            for x in _ulps(c * den * s, 3):
                n.append(x)
                d.append(den * s)
    special = [0.0, -0.0, 5e-324, -5e-324, 2.2250738585072014e-308 / 3, np.inf, -np.inf, np.nan, 1.0, -1.0,
               2.0 ** -959, 2.0 ** 961, np.nextafter(2.0 ** 961, 0), 1.7976931348623157e308]
    for a in special:
        for b in special:
            n.append(a)
            d.append(b)
    return np.array(n), np.array(d)


def _in_band(n, den):
    """Exactly: is n / den inside (-2^-43, -2^-44) or (1 + 2^-34, 1 + 2^-33)?"""
    q = Fraction(float(n)) / Fraction(float(den))
    return -Fraction(1, 2 ** 43) < q < -Fraction(1, 2 ** 44) or 1 + Fraction(1, 2 ** 34) < q < 1 + Fraction(1, 2 ** 33)


@pytest.mark.gpu
def test_decision_matches_division(seg_cross_probe):
    n, d = operands()
    out = seg_cross_probe(n, d)
    r, ex, ref = (out & 1) != 0, (out & 2) != 0, (out & 4) != 0
    assert int((ex & (r != ref)).sum()) == 0, np.argwhere(ex & (r != ref))[:5]
    # the regime: finite n with |n| in [2^-959, 2^961) or 0, |den| in [2^-44, 2^1024)
    an, ad = np.abs(n), np.abs(d)
    regime = ((an == 0) | ((an >= 2.0 ** -959) & (an < 2.0 ** 961))) & (ad >= 2.0 ** -44) & np.isfinite(d)
    assert not ex[~regime].any()
    band = np.array([bool(g) and _in_band(a, b) for g, a, b in zip(regime, n, d)])
    assert band.sum() > 500
    assert not ex[band].any(), 'a band case did not take the division'
    assert ex[regime & ~band].all(), 'the division was taken outside the bands'
    # both answers occur at every cut-off
    assert ref[ex].any() and not ref[ex].all()
    # the crossing test of the directed search shares the regime guard
    r2, ex2, ref2 = (out & 8) != 0, (out & 16) != 0, (out & 32) != 0
    assert int((ex2 & (r2 != ref2)).sum()) == 0


def build_cutoff_batch(cls, n_envs, seed):
    """tests/test_overlap_random.py's batch with every designed pair (a_j, b_j) replaced: a vertex of
    b on the line of an edge of a, at the edge parameter -1e-13 or 1 + 1e-10 (the cut-offs of
    segments_intersect's range tests), a few per cent inside or outside them, or at the edges of
    the bands where the decision hands over to the division."""
    prog, arr, _ = tor.build_batch(cls, n_envs, seed)
    rng = np.random.RandomState(seed + 1)
    voff = tor.util.prog_voff(prog)
    nv = arr['meta'][0, 2]
    lo_a, lo_b = prog.layer_off[prog.layer_index('a')], prog.layer_off[prog.layer_index('b')]
    lams = np.array([-1e-13 * 0.97, -1e-13 * 1.03, -2.0 ** -44, -2.0 ** -43,
                     1 + 1e-10 * 0.97, 1 + 1e-10 * 1.03, 1 + 2.0 ** -34, 1 + 2.0 ** -33])
    e = np.arange(n_envs)
    for j in range(tor.PER_LAYER):
        sa, sb = lo_a + j, lo_b + j
        A = arr['vtx'][:, voff[sa]:voff[sa] + nv[sa]]
        B = arr['vtx'][:, voff[sb]:voff[sb] + nv[sb]]
        ia, ib = rng.randint(0, nv[sa], size=n_envs), rng.randint(0, nv[sb], size=n_envs)
        pa, pa2, qb = A[e, ia], A[e, (ia + 1) % nv[sa]], B[e, ib]
        lam = lams[rng.randint(0, len(lams), size=n_envs)][:, None]
        t = pa + lam * (pa2 - pa) - qb
        B += t[:, None, :]
        arr['dyn'][:, 0:2, sb] += t
    return prog, arr


@pytest.mark.gpu
@pytest.mark.parametrize('cls', ['circle', 'star', 'triangle', 'walls'])
def test_cutoff_vertices_match_oracle(cls):
    from moog_b200.batched_env import Engine
    from oracle.oracle import Oracle
    n_envs = 1024
    prog, arr = build_cutoff_batch(cls, n_envs, seed=77)
    for la, lb in (('a', 'b'), ('b', 'a')):
        ref = Oracle(prog, arr).overlap_pairs(la, lb)
        eng = Engine(prog, n_envs, 'cuda:0')
        eng.state.upload(arr)
        got = eng.overlap_pairs(la, lb).cpu().numpy()
        diag = np.arange(tor.PER_LAYER)
        designed = ref[:, diag, diag]
        print('{} {}{}: {} designed pairs, {} overlapping'.format(cls, la, lb, designed.size, int(designed.sum())))
        assert 0 < designed.sum() < designed.size
        assert int((got != ref).sum()) == 0, (cls, la, lb, np.argwhere(got != ref)[:5])
