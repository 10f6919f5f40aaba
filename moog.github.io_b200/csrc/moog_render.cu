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

// One env's frame: render_env (anti_aliasing 1, `rows` rows per band) or render_env_aa (chunks of
// `rows` canvas rows, a ring of `ring` resampled rows), as render_plan chose for the view.
template <bool AA>
__device__ __forceinline__ void draw_env(const RenderArgs &a, const RenderSrc &src, unsigned char *base, int t, int T,
                                         int P, bool live, uint8_t *out, int rows, int ring) {
  const RenderLayout lay = view_layout(src.hdr, src.view, rows, AA ? ring : 0);
  if (AA)
    render_env_aa(src, lay, base, nullptr, t, T, P, live, out, a.resample, a.ksize_h, a.ksize_v,
                  [] { __syncthreads(); }, rows, ring);
  else
    render_env(src, lay, base, nullptr, t, T, P, live, out, [] { __syncthreads(); }, rows);
}

__device__ __forceinline__ RenderSrc env_src(const RenderArgs &a, const ProgramView &pv, const int32_t *view, size_t row) {
  const int S = pv.hdr[MOOG_H_N_SLOTS], VT = pv.hdr[MOOG_H_N_VTX];
  RenderSrc src;
  src.dyn = a.st.dyn + row * MOOG_DYN_FIELDS * S;
  src.stat = a.st.stat + row * MOOG_STAT_FIELDS * S;
  src.meta = a.st.meta + row * MOOG_META_FIELDS * S;
  src.cnt = a.st.cnt + row * MOOG_MAX_LAYERS;
  src.vtx = (const double2 *)(a.st.vtx + row * 2 * VT);
  src.hdr = pv.hdr;
  src.voff = pv.voff;
  src.view = view;
  return src;
}

// blockDim.x = envs_per_block * T, T = threads of one env (render_plan)
template <bool AA>
__global__ void moog_render_kernel(RenderArgs a, int T, int envs_per_block, int P, int rows, int ring) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ProgramView pv = view_of(a.blob);
  const int32_t *view = pv.hdr + a.view_off;
  const int OH = view[MOOG_V_HEIGHT], OW = view[MOOG_V_WIDTH];
  const int g = threadIdx.x / T, t = threadIdx.x - g * T;
  const int n = blockIdx.x * envs_per_block + g;
  const bool live = n < a.n_envs;
  const size_t row = live ? (size_t)n : 0;
  const RenderSrc src = env_src(a, pv, view, row);
  const int env_bytes = view_layout(pv.hdr, view, rows, AA ? ring : 0).total;
  draw_env<AA>(a, src, smem_raw + (size_t)g * env_bytes, t, T, P, live, a.frames + row * OH * OW * 3, rows, ring);
}

// SpriteMask: one env's mask per T threads, as moog_render_kernel<false> draws a frame (a.frames holds
// the int16 masks)
__global__ void moog_render_mask_kernel(RenderArgs a, int T, int envs_per_block, int P, int rows) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ProgramView pv = view_of(a.blob);
  const int32_t *mask = pv.hdr + a.view_off;
  const int OH = mask[MOOG_V_HEIGHT], OW = mask[MOOG_V_WIDTH];
  const int g = threadIdx.x / T, t = threadIdx.x - g * T;
  const int n = blockIdx.x * envs_per_block + g;
  const bool live = n < a.n_envs;
  const size_t row = live ? (size_t)n : 0;
  const RenderSrc src = env_src(a, pv, mask, row);
  const RenderLayout lay = view_layout(pv.hdr, mask, rows, 0);
  mask_env(src, lay, smem_raw + (size_t)g * lay.total, t, T, P, live, (int16_t *)a.frames + row * OH * OW,
           [] { __syncthreads(); }, rows);
}

// The same for the envs of a step kernel that is still running (launched behind it with
// programmatic stream serialization: this grid starts once every step CTA is resident or done, so
// its CTAs land on the SMs the step has no more envs for).  A few CTAs per SM take tickets for the
// entries of the finished list, and a CTA takes none while its own SM is still stepping an env
// (sm_active, kept by the step kernel) -- a renderer next to a long-running env slows down exactly
// the env the whole step is waiting for.  The frames are drawn on the SMs the step has left, the
// last env's by whichever CTA is free.  A ticket's CTA waits for its entry of the finished list
// (acquire; the step kernel releases it after the env's record is in HBM).  Every env it could wait
// for is running or done, so the wait is bounded by the step itself; the poll limit only turns a
// broken launch into an error.
template <bool AA>
__global__ void moog_render_tail_persistent_kernel(RenderArgs a, int T, int P, int *done, int n_done, int busy_thr,
                                                   int rows, int ring) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_env;
  int *ticket = done + 1 + n_done;
  const int *sm_active = ticket + 1;
  unsigned smid;
  asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
  ProgramView pv = view_of(a.blob);
  const int32_t *view = pv.hdr + a.view_off;
  const int OH = view[MOOG_V_HEIGHT], OW = view[MOOG_V_WIDTH];
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
    const RenderSrc src = env_src(a, pv, view, row);
    unsigned long long tr0 = 0;
    if (a.trace) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr0));
    draw_env<AA>(a, src, smem_raw, (int)threadIdx.x, T, P, true, a.frames + row * OH * OW * 3, rows, ring);
    __syncthreads();
    if (a.trace && threadIdx.x == 0) {
      unsigned long long tr1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr1));
      a.trace[MOOG_N_COUNTERS * row + 4] = (long long)tr0;
      a.trace[MOOG_N_COUNTERS * row + 5] = (long long)tr1;
    }
  }
  // this grid must not complete before the step grid has (what follows on the stream waits for
  // this grid only): the CTA that drew the last env to finish waits for the step grid's completion
  if (last) asm volatile("griddepcontrol.wait;" ::: "memory");
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

// Resample.c precompute_coeffs: taps per output pixel, the longest window an output pixel reads
int lanczos_ksize(int in_size, int out_size) {
  double scale = (double)in_size / out_size, filterscale = scale < 1.0 ? 1.0 : scale;
  return (int)ceil(3.0 * filterscale) * 2 + 1;
}

static int resample_axis(int in_size, int out_size, std::vector<int> &bounds, std::vector<int> &coeffs) {
  double scale = (double)in_size / out_size, filterscale = scale < 1.0 ? 1.0 : scale;
  double support = 3.0 * filterscale;
  int ksize = lanczos_ksize(in_size, out_size);
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

// How a view is drawn (see RenderPlan in moog_common.cuh).  anti_aliasing 1: a canvas that does not
// fit next to the edge lists in one CTA's shared memory is drawn in bands: the largest band, a
// multiple of 8 rows, whose layout leaves room for two CTAs per SM.  anti_aliasing > 1: the largest
// chunk (at most 512 rows) whose canvas, edge lists and ring of chunk + ksize_v resampled rows
// leave room for two CTAs per SM, else the largest that fits one CTA; then the chunks are evened out.
RenderPlan render_plan(const int32_t *hdr, const int32_t *view) {
  RenderPlan p;
  memset(&p, 0, sizeof(p));
  const int OH = view[MOOG_V_HEIGHT], OW = view[MOOG_V_WIDTH], aa = view[MOOG_V_AA];
  if (OH < 1 || OW < 1 || aa < 1 || OH > 8192 || OW > 8192 || aa > 16) return p;
  const int H = aa * OH, W = aa * OW;
  const int kBudget2 = 110 * 1024, kBudget1 = 224 * 1024;
  if (4LL * (W + 1) > kBudget1) return p;  // not even one canvas row fits
  if (aa == 1) {
    int band = 0;
    if (view_layout(hdr, view, H, 0).total > kBudget2) {
      band = H & ~7;
      while (band > 8 && view_layout(hdr, view, band, 0).total > kBudget2) band -= 8;
    }
    p.rows = band > 0 ? band : H;
    p.P = (p.rows <= 128) ? 2 : 1;  // threads per canvas row (they split its columns)
  } else {
    const int ks = lanczos_ksize(H, OH);
    for (int budget : {kBudget2, kBudget1}) {
      for (int hc = H < 512 ? H : 512; hc >= 1 && p.rows == 0; --hc) {
        const int ring = hc + ks < H ? hc + ks : H;
        if (view_layout(hdr, view, hc, ring).total <= budget) {
          p.rows = hc;
          p.ring = ring;
        }
      }
      if (p.rows > 0) break;
    }
    if (p.rows == 0) return p;
    if (p.rows < H) {  // the same number of chunks, of even height: no short last chunk
      const int n = (H + p.rows - 1) / p.rows;
      p.rows = (H + n - 1) / n;
      p.ring = p.rows + ks < H ? p.rows + ks : H;
    }
    p.P = p.rows <= 128 ? 2 : 1;
    if (p.rows * p.P < 256) p.P = 256 / p.rows;  // short chunks: more threads share a row
    if (p.P > W / 16) p.P = W / 16 > 1 ? W / 16 : 1;
  }
  p.T = (p.rows * p.P + 31) & ~31;
  p.env_bytes = view_layout(hdr, view, p.rows, p.ring).total;
  p.ok = p.env_bytes <= kBudget1 && p.T <= 1024;
  return p;
}

template <class K>
static cudaError_t allow_smem(K kernel, size_t smem, size_t &configured) {
  if (smem <= 48 * 1024 || smem <= configured) return cudaSuccess;
  cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err == cudaSuccess) configured = smem;
  return err;
}

// envs per CTA: the split that keeps the most envs resident per SM (228 KB of shared
// memory, 1 KB of it reserved per CTA); ties go to the larger CTA
static int envs_per_block(int T, size_t env_bytes) {
  int epb = 1, best = 0;
  for (int c = 1; c * T <= 256 || c == 1; ++c) {
    const size_t per_cta = env_bytes * c + 1024;
    if (per_cta > 228 * 1024) break;
    const int envs = (int)(233472 / per_cta) * c;
    if (envs >= best) { best = envs; epb = c; }
  }
  return epb;
}

template <bool AA>
static cudaError_t launch_render_t(const RenderArgs &a, const RenderPlan &plan, cudaStream_t stream, int *n_launches,
                                   int *done, int n_done) {
  const int T = plan.T, P = plan.P, rows = plan.rows, ring = plan.ring;
  const size_t env_bytes = (size_t)plan.env_bytes;
  const int epb = envs_per_block(T, env_bytes);
  size_t smem = env_bytes * epb;
  if (smem > 224 * 1024) return cudaErrorInvalidConfiguration;
  static size_t configured = 0;
  cudaError_t err = allow_smem(moog_render_kernel<AA>, smem, configured);
  if (err != cudaSuccess) return err;
  if (done) {
    // one env per CTA at a time, in finishing order, overlapping the tail of the step kernel
    smem = env_bytes;
    static size_t configured_tail = 0;
    err = allow_smem(moog_render_tail_persistent_kernel<AA>, smem, configured_tail);
    if (err != cudaSuccess) return err;
    // as many CTAs per SM as its shared memory and threads hold, no more than there are envs
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int per_sm = (int)(233472 / (smem + 1024));
    const int by_threads = 2048 / T;
    if (per_sm > by_threads) per_sm = by_threads;
    if (per_sm < 1) per_sm = 1;
    const int grid = sms * per_sm < n_done ? sms * per_sm : n_done;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)T);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    // busy_thr = 1: no ticket while the SM steps any env (an argument: as a constant in the kernel it
    // costs the anti-aliased variant two registers)
    err = cudaLaunchKernelEx(&cfg, moog_render_tail_persistent_kernel<AA>, a, T, P, done, n_done, 1, rows, ring);
    if (n_launches) *n_launches += 1;
    return err;
  }
  int blocks = (a.n_envs + epb - 1) / epb;
  moog_render_kernel<AA><<<blocks, epb * T, smem, stream>>>(a, T, epb, P, rows, ring);
  if (n_launches) *n_launches += 1;
  return cudaGetLastError();
}

cudaError_t launch_render(const RenderArgs &a, const RenderPlan &plan, const int32_t *view, cudaStream_t stream,
                          int *n_launches, int *done, int n_done) {
  if (a.n_envs <= 0) return cudaSuccess;
  if (!plan.ok) return cudaErrorInvalidConfiguration;  // render_impl refuses such a view before
  return view[MOOG_V_AA] > 1 ? launch_render_t<true>(a, plan, stream, n_launches, done, n_done)
                             : launch_render_t<false>(a, plan, stream, n_launches, done, n_done);
}

cudaError_t launch_mask(const RenderArgs &a, const RenderPlan &plan, cudaStream_t stream, int *n_launches) {
  if (a.n_envs <= 0) return cudaSuccess;
  if (!plan.ok) return cudaErrorInvalidConfiguration;  // mask_impl refuses such a mask before
  const int epb = envs_per_block(plan.T, (size_t)plan.env_bytes);
  const size_t smem = (size_t)plan.env_bytes * epb;
  if (smem > 224 * 1024) return cudaErrorInvalidConfiguration;
  static size_t configured = 0;
  cudaError_t err = allow_smem(moog_render_mask_kernel, smem, configured);
  if (err != cudaSuccess) return err;
  const int blocks = (a.n_envs + epb - 1) / epb;
  moog_render_mask_kernel<<<blocks, epb * plan.T, smem, stream>>>(a, plan.T, epb, plan.P, plan.rows);
  if (n_launches) *n_launches += 1;
  return cudaGetLastError();
}

}  // namespace moog
