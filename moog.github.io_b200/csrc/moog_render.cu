// moog_render.cu -- PILRenderer.__call__ for N envs (moog/observers/pil_renderer.py:88-120).
//
// The reference pastes a background, then for every layer and sprite (z-order,
// back to front) calls Pillow's ImageDraw.polygon with an RGBA fill on an RGB
// canvas, resizes (identity for anti_aliasing=1, which every shipped config
// uses) and flips the rows.  Pillow's fill (src/libImaging/Draw.c,
// polygon_generic + hline32rgba) is an integer-scanline algorithm: vertices are
// truncated to int, every scanline collects the float32 x of the edges it
// touches (non-fused (y-y0)*dx + x0), sorts them and blends the spans; rows never
// interact.  So: one thread per scanline, one canvas per env in shared memory
// (packed RGBX words, row stride W+1 -> conflict-free), sprites walked in
// z-order by every row thread, and the finished canvas is written to HBM once,
// flipped, as coalesced 16-byte stores.
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "moog_render_dev.cuh"

namespace moog {

// blockDim.x = envs_per_block * T, T = threads of one env (>= H, multiple of 32)
__global__ void moog_render_kernel(RenderArgs a, int T, int envs_per_block, int P, int band) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ProgramView pv = view_of(a.blob);
  const int32_t *hdr = pv.hdr;
  const int32_t *view = hdr + a.view_off;
  const int S = hdr[MOOG_H_N_SLOTS], VT = hdr[MOOG_H_N_VTX];
  const int OH = view[MOOG_V_HEIGHT], OW = view[MOOG_V_WIDTH], aa = view[MOOG_V_AA];
  const int g = threadIdx.x / T, t = threadIdx.x - g * T;
  const int n = blockIdx.x * envs_per_block + g;
  const bool live = n < a.n_envs;
  const int C = view[MOOG_V_MODIFIER] == MOOG_PMOD_TORUS ? 9 : 1;
  const RenderLayout lay = render_layout(band > 0 ? band : aa * OH, aa * OW, S * C, (VT > 0 ? VT : 1) * C, OW);
  const size_t row = live ? (size_t)n : 0;
  RenderSrc src;
  src.dyn = a.st.dyn + row * MOOG_DYN_FIELDS * S;
  src.stat = a.st.stat + row * MOOG_STAT_FIELDS * S;
  src.meta = a.st.meta + row * MOOG_META_FIELDS * S;
  src.cnt = a.st.cnt + row * MOOG_MAX_LAYERS;
  src.vtx = (const double2 *)(a.st.vtx + row * 2 * VT);
  src.hdr = hdr;
  src.voff = pv.voff;
  src.view = view;
  render_env(src, lay, smem_raw + (size_t)g * lay.total, nullptr, t, T, P, live,
             a.frames + row * OH * OW * 3, a.resample, a.ksize_h, a.ksize_v, [] { __syncthreads(); }, band);
}

// The same for the envs of a step kernel that is still running (launched behind it with
// programmatic stream serialization: this grid starts once every step CTA is resident or done, so
// its CTAs land on the SMs the step has no more envs for).  CTA b draws the b-th env to finish:
// thread 0 waits for entry b of the step kernel's finished list (acquire; the step kernel releases
// it after the env's record is in HBM).  Every env it could wait for is running or done, so the
// wait is bounded by the step itself; the poll limit only turns a broken launch into an error.
__global__ void moog_render_tail_kernel(RenderArgs a, int T, int P, const int *done, int band) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_env;
  if (threadIdx.x == 0) {
    int v = 0;
    for (unsigned polls = 0;; ++polls) {
      asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(done + 1 + blockIdx.x) : "memory");
      if (v != 0) break;
      if (polls > (1u << 24)) __trap();
      __nanosleep(200);
    }
    s_env = v - 1;
  }
  __syncthreads();
  const int n = s_env;
  ProgramView pv = view_of(a.blob);
  const int32_t *hdr = pv.hdr;
  const int32_t *view = hdr + a.view_off;
  const int S = hdr[MOOG_H_N_SLOTS], VT = hdr[MOOG_H_N_VTX];
  const int OH = view[MOOG_V_HEIGHT], OW = view[MOOG_V_WIDTH], aa = view[MOOG_V_AA];
  const int C = view[MOOG_V_MODIFIER] == MOOG_PMOD_TORUS ? 9 : 1;
  const RenderLayout lay = render_layout(band > 0 ? band : aa * OH, aa * OW, S * C, (VT > 0 ? VT : 1) * C, OW);
  const size_t row = (size_t)n;
  RenderSrc src;
  src.dyn = a.st.dyn + row * MOOG_DYN_FIELDS * S;
  src.stat = a.st.stat + row * MOOG_STAT_FIELDS * S;
  src.meta = a.st.meta + row * MOOG_META_FIELDS * S;
  src.cnt = a.st.cnt + row * MOOG_MAX_LAYERS;
  src.vtx = (const double2 *)(a.st.vtx + row * 2 * VT);
  src.hdr = hdr;
  src.voff = pv.voff;
  src.view = view;
  unsigned long long tr0 = 0;
  if (a.trace) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr0));
  render_env(src, lay, smem_raw, nullptr, (int)threadIdx.x, T, P, true, a.frames + row * OH * OW * 3, a.resample,
             a.ksize_h, a.ksize_v, [] { __syncthreads(); }, band);
  if (a.trace && threadIdx.x == 0) {
    unsigned long long tr1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr1));
    a.trace[MOOG_N_COUNTERS * row + 4] = (long long)tr0;
    a.trace[MOOG_N_COUNTERS * row + 5] = (long long)tr1;
  }
  // this grid must not complete before the step grid has (what follows on the stream waits for
  // this grid only): the CTA that drew the last env to finish waits for the step grid's completion
  if (blockIdx.x == gridDim.x - 1) asm volatile("griddepcontrol.wait;" ::: "memory");
}

// Persistent variant: a few CTAs per SM take tickets for the entries of the finished list, and a
// CTA takes none while its own SM is still stepping envs (sm_active, kept by the step kernel) -- a
// renderer next to a long-running env slows down exactly the env the whole step is waiting for.
// The frames are drawn on the SMs the step has left, the last env's by whichever CTA is free.
__global__ void moog_render_tail_persistent_kernel(RenderArgs a, int T, int P, int *done, int n_done, int busy_thr,
                                                   int band) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_env;
  int *ticket = done + 1 + n_done;
  const int *sm_active = ticket + 1;
  unsigned smid;
  asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
  ProgramView pv = view_of(a.blob);
  const int32_t *hdr = pv.hdr;
  const int32_t *view = hdr + a.view_off;
  const int S = hdr[MOOG_H_N_SLOTS], VT = hdr[MOOG_H_N_VTX];
  const int OH = view[MOOG_V_HEIGHT], OW = view[MOOG_V_WIDTH], aa = view[MOOG_V_AA];
  const int C = view[MOOG_V_MODIFIER] == MOOG_PMOD_TORUS ? 9 : 1;
  const RenderLayout lay = render_layout(band > 0 ? band : aa * OH, aa * OW, S * C, (VT > 0 ? VT : 1) * C, OW);
  bool last = false;
  for (;;) {
    if (threadIdx.x == 0) {
      int env = -1;
      for (unsigned polls = 0;; ++polls) {  // yield while this SM steps envs and tickets remain
        int busy, taken;
        asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(busy) : "l"(sm_active + (smid & 255)) : "memory");
        asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(taken) : "l"(ticket) : "memory");
        if (busy < busy_thr || taken >= n_done) break;
        if (polls > (1u << 24)) __trap();
        __nanosleep(500);
      }
      const int k = atomicAdd(ticket, 1);
      if (k < n_done) {
        int v = 0;
        for (unsigned polls = 0;; ++polls) {
          asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(done + 1 + k) : "memory");
          if (v != 0) break;
          if (polls > (1u << 24)) __trap();
          __nanosleep(200);
        }
        env = v - 1;
        if (k == n_done - 1) env |= 0x40000000;  // the last env to finish
      }
      s_env = env;
    }
    __syncthreads();
    int n = s_env;
    if (n < 0) break;
    last = last || (n & 0x40000000) != 0;
    n &= 0x3fffffff;
    const size_t row = (size_t)n;
    RenderSrc src;
    src.dyn = a.st.dyn + row * MOOG_DYN_FIELDS * S;
    src.stat = a.st.stat + row * MOOG_STAT_FIELDS * S;
    src.meta = a.st.meta + row * MOOG_META_FIELDS * S;
    src.cnt = a.st.cnt + row * MOOG_MAX_LAYERS;
    src.vtx = (const double2 *)(a.st.vtx + row * 2 * VT);
    src.hdr = hdr;
    src.voff = pv.voff;
    src.view = view;
    unsigned long long tr0 = 0;
    if (a.trace) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr0));
    render_env(src, lay, smem_raw, nullptr, (int)threadIdx.x, T, P, true, a.frames + row * OH * OW * 3, a.resample,
               a.ksize_h, a.ksize_v, [] { __syncthreads(); }, band);
    __syncthreads();
    if (a.trace && threadIdx.x == 0) {
      unsigned long long tr1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr1));
      a.trace[MOOG_N_COUNTERS * row + 4] = (long long)tr0;
      a.trace[MOOG_N_COUNTERS * row + 5] = (long long)tr1;
    }
  }
  if (last) asm volatile("griddepcontrol.wait;" ::: "memory");  // see moog_render_tail_kernel
}

// ---------------------------------------------------------------------------
// Resample.c precompute_coeffs + normalize_coeffs_8bpc for the LANCZOS filter
// (SURVEY App. B.6), on the host: the coefficients go through libm's sin() like
// Pillow's, then to 22-bit fixed point.  Layout of the returned table:
//   bounds_h[2*OW] coeff_h[OW*ksize_h] bounds_v[2*OH] coeff_v[OH*ksize_v]
// ---------------------------------------------------------------------------
static double lanczos_weight(double x) {
  if (!(-3.0 <= x && x < 3.0)) return 0.0;
  auto sinc = [](double v) {
    if (v == 0.0) return 1.0;
    v = v * M_PI;
    return sin(v) / v;
  };
  return sinc(x) * sinc(x / 3);
}

static int resample_axis(int in_size, int out_size, std::vector<int> &bounds, std::vector<int> &coeffs) {
  double scale = (double)in_size / out_size, filterscale = scale < 1.0 ? 1.0 : scale;
  double support = 3.0 * filterscale;
  int ksize = (int)ceil(support) * 2 + 1;
  bounds.assign(2 * (size_t)out_size, 0);
  coeffs.assign((size_t)out_size * ksize, 0);
  std::vector<double> k(ksize);
  for (int xx = 0; xx < out_size; ++xx) {
    double center = (xx + 0.5) * scale, ww = 0.0, ss = 1.0 / filterscale;
    int xmin = (int)(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = (int)(center + support + 0.5);
    if (xmax > in_size) xmax = in_size;
    xmax -= xmin;
    for (int x = 0; x < xmax; ++x) {
      k[x] = lanczos_weight((x + xmin - center + 0.5) * ss);
      ww += k[x];
    }
    for (int x = 0; x < xmax; ++x) {
      double w = ww != 0.0 ? k[x] / ww : k[x];
      coeffs[(size_t)xx * ksize + x] = w < 0 ? (int)(-0.5 + w * (1 << 22)) : (int)(0.5 + w * (1 << 22));
    }
    bounds[2 * xx] = xmin;
    bounds[2 * xx + 1] = xmax;
  }
  return ksize;
}

int resample_tables(int H, int W, int OH, int OW, std::vector<int> &table, int *ksize_h, int *ksize_v) {
  std::vector<int> bh, kh, bv, kv;
  *ksize_h = resample_axis(W, OW, bh, kh);
  *ksize_v = resample_axis(H, OH, bv, kv);
  table.clear();
  table.insert(table.end(), bh.begin(), bh.end());
  table.insert(table.end(), kh.begin(), kh.end());
  table.insert(table.end(), bv.begin(), bv.end());
  table.insert(table.end(), kv.begin(), kv.end());
  return (int)table.size();
}

cudaError_t launch_render(const RenderArgs &a, const int32_t *hdr, const int32_t *view, cudaStream_t stream,
                          int *n_launches, int *done, int n_done, int tail_mode, const LaunchOptions &opt) {
  if (a.n_envs <= 0) return cudaSuccess;
  const int OH = view[MOOG_V_HEIGHT], OW = view[MOOG_V_WIDTH], aa = view[MOOG_V_AA];
  const int H = aa * OH, W = aa * OW, S = hdr[MOOG_H_N_SLOTS], VT = hdr[MOOG_H_N_VTX];
  const int C = view[MOOG_V_MODIFIER] == MOOG_PMOD_TORUS ? 9 : 1;  // TorusGeometry: 9 copies per sprite
  // A canvas that does not fit next to the edge lists in one CTA's shared memory is drawn in bands
  // of `band` rows (render_env): the largest band, a multiple of 8 rows, whose layout leaves room
  // for two CTAs per SM.  Anti-aliased canvases are not banded (the Lanczos resize reads across rows).
  int band = 0;
  if (aa == 1 && render_layout(H, W, S * C, (VT > 0 ? VT : 1) * C, OW).total > 110 * 1024) {
    band = H & ~7;
    while (band > 8 && render_layout(band, W, S * C, (VT > 0 ? VT : 1) * C, OW).total > 110 * 1024) band -= 8;
  }
  const int HB = band > 0 ? band : H;
  const int P = (HB <= 128) ? 2 : 1;  // threads per canvas row (they split its columns)
  const int T = (HB * P + 31) & ~31;
  RenderLayout lay = render_layout(HB, W, S * C, (VT > 0 ? VT : 1) * C, OW);
  // envs per CTA: the split that keeps the most envs resident per SM (228 KB of shared
  // memory, 1 KB of it reserved per CTA); ties go to the larger CTA
  int epb = 1;
  {
    int best = 0;
    for (int c = 1; c * T <= 256 || c == 1; ++c) {
      const size_t per_cta = (size_t)lay.total * c + 1024;
      if (per_cta > 228 * 1024) break;
      const int envs = (int)(233472 / per_cta) * c;
      if (envs >= best) { best = envs; epb = c; }
    }
    if (opt.render_epb > 0) epb = opt.render_epb;
  }
  size_t smem = (size_t)lay.total * epb;
  if (smem > 224 * 1024 || T > 1024) return cudaErrorInvalidConfiguration;
  static size_t configured = 0;
  if (smem > 48 * 1024 && smem > configured) {
    cudaError_t err = cudaFuncSetAttribute(moog_render_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    configured = smem;
  }
  if (done) {
    // one env per CTA, in finishing order, overlapping the tail of the step kernel
    smem = (size_t)lay.total;
    static size_t configured_tail = 0;
    if (smem > 48 * 1024 && smem > configured_tail) {
      cudaError_t err =
          cudaFuncSetAttribute(moog_render_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (err != cudaSuccess) return err;
      configured_tail = smem;
    }
    static size_t configured_pers = 0;
    if (tail_mode == 2 && smem > 48 * 1024 && smem > configured_pers) {
      cudaError_t err = cudaFuncSetAttribute(moog_render_tail_persistent_kernel,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (err != cudaSuccess) return err;
      configured_pers = smem;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)a.n_envs);
    cfg.blockDim = dim3((unsigned)T);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t err;
    if (tail_mode == 2) {
      int dev = 0, sms = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
      int per_sm = (int)(233472 / (smem + 1024));
      const int by_threads = 2048 / T;
      if (per_sm > by_threads) per_sm = by_threads;
      if (per_sm < 1) per_sm = 1;
      if (opt.tail_ctas_per_sm > 0 && opt.tail_ctas_per_sm < per_sm) per_sm = opt.tail_ctas_per_sm;
      int grid = sms * per_sm;
      if (grid > n_done) grid = n_done;
      cfg.gridDim = dim3((unsigned)grid);
      const int busy_thr = opt.tail_busy_thr > 0 ? opt.tail_busy_thr : 1;  // envs being stepped on an SM from which its render CTAs stand back
      err = cudaLaunchKernelEx(&cfg, moog_render_tail_persistent_kernel, a, T, P, done, n_done, busy_thr, band);
    } else {
      err = cudaLaunchKernelEx(&cfg, moog_render_tail_kernel, a, T, P, (const int *)done, band);
    }
    if (n_launches) *n_launches += 1;
    return err;
  }
  int blocks = (a.n_envs + epb - 1) / epb;
  moog_render_kernel<<<blocks, epb * T, smem, stream>>>(a, T, epb, P, band);
  if (n_launches) *n_launches += 1;
  return cudaGetLastError();
}

}  // namespace moog
