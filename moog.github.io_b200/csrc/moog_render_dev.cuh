// moog_render_dev.cuh -- device side of PILRenderer.__call__ (moog/observers/pil_renderer.py:88-120),
// shared by the stand-alone render kernel (moog_render.cu) and the step kernel, which draws the
// frame of the state it leaves an env in while the record is still in shared memory (moog_step.cu).
#pragma once
#include <math.h>

#include "moog_common.cuh"

namespace moog {

#define RENDER_MAXV MOOG_MAX_OUTLINE
#define MAX_XX (2 * RENDER_MAXV + 8)

// C `(int)double` as the reference's host executes it (x86-64 cvttsd2si): NaN and
// out-of-range values give INT_MIN (CUDA's conversion would saturate / give 0)
__device__ __forceinline__ int c_int_cast(double v) {
  return (v > -2147483649.0 && v < 2147483648.0) ? (int)v : (int)0x80000000;
}

// Resample.c clip8: fixed point (22 fractional bits) -> uint8
__device__ __forceinline__ unsigned clip8(int v) {
  v >>= 22;
  return (unsigned)(v < 0 ? 0 : (v > 255 ? 255 : v));
}

__device__ __forceinline__ unsigned div255(unsigned a) { return (((a + 128) >> 8) + (a + 128)) >> 8; }

__device__ __forceinline__ unsigned blend_px(unsigned bg, unsigned ink) {
  unsigned a = ink >> 24;
  unsigned r = div255((bg & 255) * (255 - a) + (ink & 255) * a);
  unsigned g = div255(((bg >> 8) & 255) * (255 - a) + ((ink >> 8) & 255) * a);
  unsigned b = div255(((bg >> 16) & 255) * (255 - a) + ((ink >> 16) & 255) * a);
  return r | (g << 8) | (b << 16);
}

__device__ __forceinline__ int round_up_(float f) { return (int)(f >= 0.0f ? floorf(f + 0.5f) : -floorf(fabsf(f) + 0.5f)); }
__device__ __forceinline__ int round_down_(float f) { return (int)(f >= 0.0f ? ceilf(f - 0.5f) : -ceilf(fabsf(f) - 0.5f)); }

// Draw.c: (y - e->y0) * e->dx + e->x0, float32, no fused multiply-add
__device__ __forceinline__ float edge_x(int x0, int y0, float dx, int y) {
  return __fadd_rn(__fmul_rn((float)(y - y0), dx), (float)x0);
}

// ---------------------------------------------------------------------------
// Pillow's edge list, built ONCE per sprite (ImagingDrawPolygon, Draw.c): the
// consecutive collinear horizontal edges are merged exactly as Pillow merges
// them, dx is divided once.  A row then only reads records.
// ---------------------------------------------------------------------------
struct ERec {
  int x0, y0, ymin, ymax;  // horizontal edge: x0 = xmin, ymin == ymax == y
  float dx;
  int xmax_h;              // horizontal edge: xmax
};

__device__ __forceinline__ ERec make_rec(int2 a, int2 b) {
  ERec r;
  r.ymin = min(a.y, b.y);
  r.ymax = max(a.y, b.y);
  if (a.y == b.y) {
    r.x0 = min(a.x, b.x);
    r.y0 = a.y;
    r.dx = 0.0f;
    r.xmax_h = max(a.x, b.x);
  } else {
    r.x0 = a.x;
    r.y0 = a.y;
    r.dx = __fdiv_rn((float)(b.x - a.x), (float)(b.y - a.y));
    r.xmax_h = 0;
  }
  return r;
}

// returns the number of records written to E (<= count)
__device__ inline int build_edge_list(const int2 *xy, int count, ERec *E, int *has_horizontal) {
  int ne = 0, hz = 0;
  for (int i = 0; i < count - 1; ++i) {
    int2 a = xy[i], b = xy[i + 1];
    if (a.y == b.y) {
      hz = 1;
      if (i != 0 && a.y == xy[i - 1].y) {
        int xp = xy[i - 1].x;
        if (b.x > a.x && a.x > xp) {
          E[ne - 1].xmax_h = b.x;
          continue;
        } else if (b.x < a.x && a.x < xp) {
          E[ne - 1].x0 = b.x;
          continue;
        }
      }
    }
    E[ne++] = make_rec(a, b);
  }
  if (count > 0 && (xy[count - 1].x != xy[0].x || xy[count - 1].y != xy[0].y)) {
    if (xy[count - 1].y == xy[0].y) hz = 1;
    E[ne++] = make_rec(xy[count - 1], xy[0]);
  }
  *has_horizontal = hz;
  return ne;
}

// Where polygon_generic's hline calls go.  BlendSink blends straight into the row
// (hline32rgba); SpanSink records the clipped spans of one (sprite, row) item so
// that the rows can be filled later, in z-order, by another thread.
struct BlendSink {
  unsigned *row;
  int W;
  unsigned ink;
  int xlo, xhi;  // the columns this thread owns
  __device__ __forceinline__ void hline(int x0, int x1) {
    if (x0 < 0) x0 = 0; else if (x0 >= W) return;   // hline32rgba's clipping
    if (x1 < 0) return; else if (x1 >= W) x1 = W - 1;
    x0 = max(x0, xlo);
    x1 = min(x1, xhi);
    for (int x = x0; x <= x1; ++x) row[x] = blend_px(row[x], ink);
  }
};

// BlendSink's counterpart for a sprite mask: the covered pixels of the row take the sprite's slot
struct SlotSink {
  unsigned *row;
  int W;
  unsigned slot;
  int xlo, xhi;
  __device__ __forceinline__ void hline(int x0, int x1) {
    if (x0 < 0) x0 = 0; else if (x0 >= W) return;   // hline32rgba's clipping
    if (x1 < 0) return; else if (x1 >= W) x1 = W - 1;
    x0 = max(x0, xlo);
    x1 = min(x1, xhi);
    for (int x = x0; x <= x1; ++x) row[x] = slot;
  }
};

#define ITEM_SPANS 3          /* spans stored per item; more -> the item is redone directly */
#define ITEM_OVERFLOW 0xffu
struct SpanSink {
  unsigned *item;  // [1 + ITEM_SPANS] words: count, then x0 | x1 << 16
  int W;
  int n;
  __device__ __forceinline__ void hline(int x0, int x1) {
    if (x0 < 0) x0 = 0; else if (x0 >= W) return;   // hline32rgba's clipping
    if (x1 < 0) return; else if (x1 >= W) x1 = W - 1;
    if (x0 > x1) return;
    if (n < ITEM_SPANS) item[1 + n] = (unsigned)x0 | ((unsigned)x1 << 16);
    n++;
  }
};

#define MAX_HROW 8 /* horizontal edges of one polygon on one scanline kept in registers */

// Draw.c draw_horizontal_lines for row y over the horizontal records of that row
// (hrow[0..nh): indices into E, in list order; nh < 0: scan the whole list)
template <class Sink>
__device__ inline void draw_horizontal_lines_rec(const ERec *E, int ne, const unsigned char *hrow, int nh, int y,
                                                 int *x_pos, Sink &sink) {
  const int n = nh >= 0 ? nh : ne;
  for (int q = 0; q < n; ++q) {
    const int i = nh >= 0 ? hrow[q] : q;
    const ERec e = E[i];
    if (e.ymin != e.ymax || e.ymin != y) continue;
    int xmin = e.x0;
    if (*x_pos != -1 && *x_pos < xmin) continue;
    int xmax = e.xmax_h;
    if (*x_pos > xmin) {
      xmin = *x_pos;
      if (xmax < xmin) continue;
    }
    if (xmin <= xmax) sink.hline(xmin, xmax);
    *x_pos = xmax + 1;
  }
}

// Draw.c polygon_generic, the iteration of its scanline loop for row y, on the
// prebuilt edge list.
template <class Sink>
__device__ inline void polygon_row_rec(const ERec *E, int ne, int y, int ymax_c, bool has_horizontal, Sink &sink) {
  float xx[MAX_XX];
  unsigned char hrow[MAX_HROW];
  int j = 0, nh = 0;
  for (int i = 0; i < ne; ++i) {
    const ERec cur = E[i];
    if (cur.ymin == cur.ymax) {  // horizontal edges are deferred when blending
      if (cur.ymin == y) {
        if (nh >= 0 && nh < MAX_HROW) hrow[nh++] = (unsigned char)i; else nh = -1;
      }
      continue;
    }
    if (y >= cur.ymin && y <= cur.ymax) {
      xx[j++] = edge_x(cur.x0, cur.y0, cur.dx, y);
      if (y == cur.ymax && y < ymax_c) {
        xx[j] = xx[j - 1];
        j++;
      } else if ((y == cur.ymin || y == cur.ymax) && cur.dx != 0) {
        for (int k = 0; k < i; ++k) {
          const ERec oth = E[k];
          if (oth.ymin == oth.ymax) continue;
          if ((y != oth.ymin && y != oth.ymax) || oth.dx == 0) continue;
          if (roundf(xx[j - 1]) == roundf(edge_x(oth.x0, oth.y0, oth.dx, y))) {
            int off = (y == ymax_c) ? -1 : 1;
            if (y + off >= oth.ymin && y + off <= oth.ymax) {
              float adj = edge_x(cur.x0, cur.y0, cur.dx, y + off);
              float oadj = edge_x(oth.x0, oth.y0, oth.dx, y + off);
              if (xx[j - 1] > adj + 1 && xx[j - 1] > oadj + 1)
                xx[j - 1] = roundf(fmaxf(adj, oadj)) + 1;
              else if (xx[j - 1] < adj - 1 && xx[j - 1] < oadj - 1)
                xx[j - 1] = roundf(fminf(adj, oadj)) - 1;
              break;
            }
          }
        }
      }
    }
  }
  has_horizontal = has_horizontal && nh != 0;
  // qsort ascending
  for (int a = 1; a < j; ++a) {
    float v = xx[a];
    int b = a;
    while (b > 0 && xx[b - 1] > v) {
      xx[b] = xx[b - 1];
      --b;
    }
    xx[b] = v;
  }
  int x_pos = (j == 0) ? -1 : 0;
  for (int i = 1; i < j; i += 2) {
    int x_end = round_down_(xx[i]);
    if (x_end < x_pos) continue;
    if (has_horizontal) draw_horizontal_lines_rec(E, ne, hrow, nh, y, &x_pos, sink);
    if (x_end < x_pos) continue;
    int x_start = round_up_(xx[i - 1]);
    if (x_pos > x_start) {
      x_start = x_pos;
      if (x_end < x_start) continue;
    }
    if (x_start <= x_end) sink.hline(x_start, x_end);
    x_pos = x_end + 1;
  }
  if (has_horizontal) draw_horizontal_lines_rec(E, ne, hrow, nh, y, &x_pos, sink);
}

// color_maps.py:21-23 (CPython colorsys.hsv_to_rgb, x255, astype(uint8))
__device__ __forceinline__ unsigned to_u8(double v) { return (unsigned)(unsigned char)(long long)v; }

__device__ inline unsigned color_to_ink(int cmap, double c0, double c1, double c2, double opacity) {
  unsigned r8, g8, b8;
  if (cmap != MOOG_CMAP_HSV) {
    r8 = to_u8(c0); g8 = to_u8(c1); b8 = to_u8(c2);
  } else {
    double h = c0, s = c1, v = c2, r, g, b;
    if (s == 0.0) {
      r = g = b = v;
    } else {
      int i = (int)(h * 6.0);
      double f = (h * 6.0) - i;
      double p = v * (1.0 - s);
      double q = v * (1.0 - s * f);
      double t = v * (1.0 - s * (1.0 - f));
      i = ((i % 6) + 6) % 6;
      switch (i) {
        case 0: r = v; g = t; b = p; break;
        case 1: r = q; g = v; b = p; break;
        case 2: r = p; g = v; b = t; break;
        case 3: r = p; g = q; b = v; break;
        case 4: r = t; g = p; b = v; break;
        default: r = v; g = p; b = q; break;
      }
    }
    r8 = to_u8(255 * r); g8 = to_u8(255 * g); b8 = to_u8(255 * b);
  }
  return r8 | (g8 << 8) | (b8 << 16) | (to_u8(opacity) << 24);
}

/* (sprite, row) items whose spans are precomputed, per env: 512, more for scenes with many
   sprites (a pacman maze has ~180), the rest is scan-converted by the row threads directly */
__host__ __device__ inline int item_cap(int S) { return S * 8 < 512 ? 512 : (S * 8 > 2048 ? 2048 : S * 8); }
struct RenderLayout { int canvas, ivtx, erec, items, ink, ymin, ymax, horiz, nedge, ibase, ring, cap, total; };

// H, W: rows and width of the canvas held at once (a band / chunk of the anti_aliasing x image
// size canvas); OW: image width.  ext_items: bytes of a buffer outside this layout that may hold the
// item spans (the step kernel's vertex cache, dead once the int vertices exist); when they fit
// there, L.items = -1.  L.ring: see view_layout.
__host__ __device__ inline RenderLayout render_layout(int H, int W, int S, int VT, int OW, int ext_items = 0) {
  RenderLayout L;
  int o = 0;
  L.canvas = o; o += 4 * H * (W + 1);
  o = (o + 7) & ~7;
  L.erec = o;   o += 24 * VT;
  // the int vertices are dead once the edge lists exist: the item spans reuse their space
  L.ivtx = o;
  L.items = o;
  {
    L.cap = item_cap(S);
    int a = 8 * VT, b = 4 * (1 + ITEM_SPANS) * L.cap;
    if (b <= ext_items) {
      L.items = -1;
      b = 0;
    }
    o += a > b ? a : b;
  }
  L.ink = o;    o += 4 * S;
  L.ymin = o;   o += 4 * S;
  L.ymax = o;   o += 4 * S;
  L.horiz = o;  o += 4 * S;
  L.nedge = o;  o += 4 * S;
  L.ibase = o;  o += 4 * (S + 1);
  L.ring = -1;
  L.total = (o + 15) & ~15;
  return L;
}


// The layout of a view's canvas drawn `rows` rows at a time (render_plan picks them), with
// `ring_rows` rows of OW horizontally resampled RGBX words (anti_aliasing > 1) at L.ring.  While
// chunks follow each other the ring lives behind everything else, like the edge lists; when one chunk
// is the whole canvas, the edge lists and item spans are dead once it is drawn, and the ring reuses
// their space.
__host__ __device__ inline RenderLayout view_layout(const int32_t *hdr, const int32_t *view, int rows, int ring_rows) {
  const int S = hdr[MOOG_H_N_SLOTS], VT = hdr[MOOG_H_N_VTX];
  const int C = view[MOOG_V_MODIFIER] == MOOG_PMOD_TORUS ? 9 : 1;  // TorusGeometry: 9 copies per sprite
  const int OW = view[MOOG_V_WIDTH];
  RenderLayout L = render_layout(rows, view[MOOG_V_AA] * OW, S * C, (VT > 0 ? VT : 1) * C, OW);
  if (ring_rows > 0) {
    L.ring = rows >= view[MOOG_V_AA] * view[MOOG_V_HEIGHT] ? L.erec : L.total;
    const int end = (L.ring + 4 * ring_rows * OW + 15) & ~15;
    if (end > L.total) L.total = end;
  }
  return L;
}

// what render_env reads of one env: the SoA record (global or shared memory) and the program
struct RenderSrc {
  const double *dyn, *stat;
  const int32_t *meta, *cnt;
  const double2 *vtx;
  const int32_t *hdr, *voff;  // program header, slot -> first cached vertex
  const int32_t *view;        // the view's MOOG_VIEW_WORDS settings (view 0: hdr + MOOG_H_R_HEIGHT)
};

// The parts of PILRenderer.__call__ for ONE env that render_env (anti_aliasing 1) and
// render_env_aa share.  Every thread t = 0..T-1 of the CTA group that shares `base` calls them with
// the same arguments; `sync` is a barrier over exactly those threads.
//
// render_prepare: int-truncated canvas vertices, ink, and Pillow's edge list and row extent of every
// (virtual) slot, built once per env; they stay live while the canvas is drawn in bands / chunks.
template <class Sync>
__device__ __forceinline__ void render_prepare(const RenderSrc &src, const RenderLayout &lay, unsigned char *base,
                                               int t, int T, bool live, Sync sync) {
  const int32_t *hdr = src.hdr, *view = src.view;
  const int S = hdr[MOOG_H_N_SLOTS], L = hdr[MOOG_H_N_LAYERS], VT = hdr[MOOG_H_N_VTX];
  // pil_renderer.py:65-66: the canvas is anti_aliasing x the image size
  const int aa = view[MOOG_V_AA], H = aa * view[MOOG_V_HEIGHT], W = aa * view[MOOG_V_WIDTH];
  const int cmap = view[MOOG_V_COLORMAP], pmod = view[MOOG_V_MODIFIER], pml = view[MOOG_V_MOD_LAYER];
  // polygon_modifiers.py:88-96 TorusGeometry: every sprite is drawn as 9 copies shifted by
  // (i, j), i outer / j inner over (-1, 0, 1); copy c of slot s is the virtual slot s * C + c
  // and its vertices live at c * VT + voff[s]
  const int C = pmod == MOOG_PMOD_TORUS ? 9 : 1;
  int2 *ivtx = (int2 *)(base + lay.ivtx);
  unsigned *ink = (unsigned *)(base + lay.ink);
  int *symin = (int *)(base + lay.ymin), *symax = (int *)(base + lay.ymax), *shoriz = (int *)(base + lay.horiz);
  int *snedge = (int *)(base + lay.nedge);
  ERec *erec = (ERec *)(base + lay.erec);
  const double *dyn = src.dyn, *stat = src.stat;
  const int32_t *meta = src.meta, *cnt = src.cnt;
  const double2 *vtx = src.vtx;

  if (live) {
    double ox = 0, oy = 0;
    if (pmod == MOOG_PMOD_FIRST_PERSON) {  // polygon_modifiers.py:54-63
      int s = hdr[MOOG_H_LAYER_OFF + pml];
      ox = 0.5 - dyn[MOOG_D_X * S + s];
      oy = 0.5 - dyn[MOOG_D_Y * S + s];
    }
    // int-truncated canvas vertices (C cast toward zero), per-slot extents and ink
    for (int v = t; v < C * VT; v += T) {
      const int c = v / VT;
      double2 p = vtx[v - c * VT];
      double x = p.x, y = p.y;
      if (pmod == MOOG_PMOD_TORUS) { x = x + (double)(c / 3 - 1); y = y + (double)(c % 3 - 1); }
      else if (pmod != MOOG_PMOD_NONE) { x = x + ox; y = y + oy; }
      ivtx[v] = make_int2(c_int_cast((double)W * x), c_int_cast((double)H * y));
    }
    for (int s = t; s < S; s += T)
      ink[s] = color_to_ink(cmap, stat[MOOG_S_C0 * S + s], stat[MOOG_S_C1 * S + s], stat[MOOG_S_C2 * S + s],
                            stat[MOOG_S_OPACITY * S + s]);
  }
  sync();
  // Draw order = layer order, then list order inside a layer (environment.py:20-25), which is
  // slot order over the LIVE slots (layer l owns the slots [LAYER_OFF[l], LAYER_OFF[l] + cnt[l])).
  // A slot that is not live or has no outline gets an empty row range, so that everything below
  // can walk the slots 0 .. S*C-1 without looking at layers again.
  if (live) {
    for (int vs = t; vs < S * C; vs += T) {
      const int s = vs / C, vo = (vs - s * C) * VT + src.voff[s];
      int nv = meta[MOOG_M_NV * S + s];
      bool drawn = false;
      for (int l = 0; l < L; ++l) {
        const int first = hdr[MOOG_H_LAYER_OFF + l];
        drawn = drawn || (s >= first && s < first + cnt[l]);
      }
      if (!drawn) nv = 0;
      const int2 *xy = ivtx + vo;
      int lo = 0x7fffffff, hi = -0x7fffffff, hz = 0;
      for (int i = 0; i < nv; ++i) {
        lo = min(lo, xy[i].y);
        hi = max(hi, xy[i].y);
      }
      snedge[vs] = nv > 0 ? build_edge_list(xy, nv, erec + vo, &hz) : 0;
      symin[vs] = lo; symax[vs] = hi; shoriz[vs] = hz;
    }
  }
  sync();  // the scan below reads every slot's extents
}

// render_draw_rows: the canvas rows [y0, y1) into the layout's canvas (its row 0 = canvas row y0):
// background, (sprite, row) item spans, then P threads per row fill the sprites in z-order.
// Returns after a barrier: the canvas rows are complete.
// SLOTS (the fill policy): false, the frames: the ink is blended into RGBX words over the view's
// background.  true, a sprite mask: every pixel a sprite with a non-zero ink alpha covers takes its
// slot, over a background of MASK_NONE; the scan conversion is the same.
#define MASK_NONE 0xffffu /* int16 -1 */
template <class Sync, bool SLOTS = false>
__device__ __forceinline__ void render_draw_rows(const RenderSrc &src, const RenderLayout &lay, unsigned char *base,
                                                 unsigned *ext_items, int t, int T, int P, bool live, int y0, int y1,
                                                 Sync sync) {
  const int32_t *view = src.view;
  const int S = src.hdr[MOOG_H_N_SLOTS], VT = src.hdr[MOOG_H_N_VTX];
  const int aa = view[MOOG_V_AA], H = aa * view[MOOG_V_HEIGHT], W = aa * view[MOOG_V_WIDTH];
  const unsigned bgc = SLOTS ? MASK_NONE : (unsigned)view[MOOG_V_BG] & 0xffffffu;
  const int C = view[MOOG_V_MODIFIER] == MOOG_PMOD_TORUS ? 9 : 1;
  unsigned *canvas = (unsigned *)(base + lay.canvas);
  unsigned *ink = (unsigned *)(base + lay.ink);
  int *symin = (int *)(base + lay.ymin), *symax = (int *)(base + lay.ymax), *shoriz = (int *)(base + lay.horiz);
  int *snedge = (int *)(base + lay.nedge), *sibase = (int *)(base + lay.ibase);
  ERec *erec = (ERec *)(base + lay.erec);
  unsigned *items = lay.items >= 0 ? (unsigned *)(base + lay.items) : ext_items;
  const int stride = W + 1;
  if (live)
    for (int i = t; i < (y1 - y0) * stride; i += T) canvas[i] = bgc;
  // (sprite, row) item ranges: exclusive prefix sum of the visible rows per slot by the first
  // warp; when the items do not all fit (lay.cap) thread 0 assigns them greedily instead and
  // the sprites left without a range are scan-converted by the row threads directly
  if (live && t < 32) {
    int acc = 0;
    for (int b = 0; b < S * C; b += 32) {
      const int vs = b + t;
      int rows = 0;
      if (vs < S * C) {
        // Draw.c polygon_generic: ymin = max(ymin, 0); ymax = min(ymax, H); rows >= H are clipped by hline
        const int lo = max(symin[vs], y0), hi = min(symax[vs], y1 - 1);
        rows = hi >= lo ? hi - lo + 1 : 0;
      }
      int x = rows;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, d);
        if (t >= d) x += y;
      }
      if (vs < S * C) sibase[vs] = rows > 0 ? acc + x - rows : -1;
      acc += __shfl_sync(0xffffffffu, x, 31);
    }
    __syncwarp();
    if (t == 0) {
      if (acc > lay.cap) {
        acc = 0;
        for (int s = 0; s < S * C; ++s) {
          const int lo = max(symin[s], y0), hi = min(symax[s], y1 - 1);
          const int rows = hi >= lo ? hi - lo + 1 : 0;
          if (rows > 0 && acc + rows <= lay.cap) {
            sibase[s] = acc;
            acc += rows;
          } else {
            sibase[s] = -1;
          }
        }
      }
      sibase[S * C] = acc;
    }
  }
  sync();
  // phase 1: one (sprite, row) item per thread pass -> clipped spans
  if (live) {
    const int n_items = sibase[S * C];
    int s = 0;  // virtual slot
    for (int it = t; it < n_items; it += T) {
      // items are sprite-major; find the sprite that owns item `it`
      for (;;) {
        int b0 = sibase[s];
        if (b0 >= 0) {
          int lo = max(symin[s], y0), hi = min(symax[s], y1 - 1);
          if (it < b0 + (hi - lo + 1)) break;
        }
        ++s;
      }
      const int lo = max(symin[s], y0);
      const int y = lo + (it - sibase[s]);
      SpanSink sink;
      sink.item = items + (size_t)it * (1 + ITEM_SPANS);
      sink.W = W;
      sink.n = 0;
      polygon_row_rec(erec + (s % C) * VT + src.voff[s / C], snedge[s], y, min(symax[s], H), shoriz[s] != 0, sink);
      sink.item[0] = sink.n <= ITEM_SPANS ? (unsigned)sink.n : ITEM_OVERFLOW;
    }
  }
  sync();
  // phase 2: P threads per row, sprites in z-order
  if (live) {
    const int HBn = y1 - y0;
    for (int w = t; w < HBn * P; w += T) {
      const int part = w / HBn, y = y0 + (w - part * HBn);
      const int xlo = (W * part) / P, xhi = (W * (part + 1)) / P - 1;  // P threads share a row
      unsigned *row = canvas + (y - y0) * stride;
      for (int s = 0; s < S * C; ++s) {
        const int ymin_c = max(symin[s], 0), ymax_c = min(symax[s], H);
        if (y < ymin_c || y > ymax_c) continue;
        const int s0 = C == 1 ? s : s / C;
        const unsigned color = ink[s0];
        if (SLOTS && (color >> 24) == 0u) continue;  // alpha 0: not in the frame, not in the mask
        const int b0 = sibase[s];
        unsigned cntw = ITEM_OVERFLOW;
        const unsigned *item = nullptr;
        if (b0 >= 0) {
          item = items + (size_t)(b0 + (y - max(ymin_c, y0))) * (1 + ITEM_SPANS);
          cntw = item[0];
        }
        if (cntw != ITEM_OVERFLOW) {
          for (unsigned q = 0; q < cntw; ++q) {
            unsigned sp = item[1 + q];
            int x0 = max((int)(sp & 0xffffu), xlo), x1 = min((int)(sp >> 16), xhi);
            if (SLOTS) {
              for (int x = x0; x <= x1; ++x) row[x] = (unsigned)s0;
            } else if ((color >> 24) == 255u) {  // DIV255(fg * 255) == fg: opaque ink overwrites
              for (int x = x0; x <= x1; ++x) row[x] = color & 0xffffffu;
            } else {
              for (int x = x0; x <= x1; ++x) row[x] = blend_px(row[x], color);
            }
          }
        } else if (SLOTS) {
          SlotSink sink;
          sink.row = row;
          sink.W = W;
          sink.slot = (unsigned)s0;
          sink.xlo = xlo;
          sink.xhi = xhi;
          polygon_row_rec(erec + (s - s0 * C) * VT + src.voff[s0], snedge[s], y, ymax_c, shoriz[s] != 0, sink);
        } else {
          BlendSink sink;
          sink.row = row;
          sink.W = W;
          sink.ink = color;
          sink.xlo = xlo;
          sink.xhi = xhi;
          polygon_row_rec(erec + (s - s0 * C) * VT + src.voff[s0], snedge[s], y, ymax_c, shoriz[s] != 0, sink);
        }
      }
    }
  }
  sync();
}

// render_store_rows: pil_renderer.py:118-120, np.flipud -> output row j is image row OH-1-j.  img
// holds the image rows [r0, r1) ([r1 - r0][img_stride] RGBX words); they are the output rows
// [OH - r1, OH - r0) of out ([OH][OW][3] bytes).
__device__ __forceinline__ void render_store_rows(const unsigned *img, int img_stride, unsigned char *out, int OH,
                                                  int OW, int r0, int r1, int t, int T) {
  if ((OW & 15) == 0) {
    // consecutive threads store consecutive 16-byte chunks of the frame (a row is OW * 3 / 16
    // of them); packed word m = 3u + r of a row holds bytes r.. of pixel 4u + r and the first
    // bytes of the next pixel
    uint4 *out4 = (uint4 *)out;
    const int cpr = (OW * 3) >> 4;
    for (int q0 = t; q0 < (r1 - r0) * cpr; q0 += T) {
      const int q = q0 + (OH - r1) * cpr;
      const int j = q / cpr, c = q - j * cpr;
      const unsigned *srcp = img + (OH - 1 - j - r0) * img_stride;
      unsigned w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int m = 4 * c + i, u = m / 3, r = m - 3 * u;
        const unsigned lo = srcp[4 * u + r] & 0xffffffu, hi = srcp[4 * u + r + 1] & 0xffffffu;
        w[i] = (lo >> (8 * r)) | (hi << (24 - 8 * r));
      }
      out4[q] = make_uint4(w[0], w[1], w[2], w[3]);
    }
  } else {
    const int nbytes = (r1 - r0) * OW * 3;
    for (int b0 = t; b0 < nbytes; b0 += T) {
      const int b = b0 + (OH - r1) * OW * 3;
      int p = b / 3, ch = b - 3 * p;
      int j = p / OW, col = p - j * OW;
      out[b] = (unsigned char)((img[(OH - 1 - j - r0) * img_stride + col] >> (8 * ch)) & 255u);
    }
  }
}

// PILRenderer.__call__ with anti_aliasing 1, for ONE env by the T threads t = 0..T-1 of a CTA (every
// thread of the CTA group that shares `base` calls it with the same arguments; `sync` is a barrier
// over exactly those threads).  base: lay.total bytes of shared memory; ext_items: where the item
// spans go when lay.items < 0.  P threads share a canvas row.  out: [OH][OW][3] bytes of this env's
// frame.  HB (0 = the whole canvas): rows per band.  A canvas that does not fit one CTA's shared
// memory (the shipped pacman draws 256 x 256, tests/runtime_benchmark.py up to 1024 x 1024) is drawn
// in bands of HB rows: `lay` is then the layout of an HB-row canvas, the edge lists are built once
// and every band scan-converts, fills and writes out its own rows.
template <class Sync>
__device__ __forceinline__ void render_env(const RenderSrc &src, const RenderLayout &lay, unsigned char *base,
                                           unsigned *ext_items, int t, int T, int P, bool live, unsigned char *out,
                                           Sync sync, int HB = 0) {
  const int OH = src.view[MOOG_V_HEIGHT], OW = src.view[MOOG_V_WIDTH];
  const int H = src.view[MOOG_V_AA] * OH;  // == OH (anti_aliasing 1)
  if (HB <= 0 || HB > H) HB = H;
  render_prepare(src, lay, base, t, T, live, sync);
#pragma unroll 1
  for (int y0 = 0; y0 < H; y0 += HB) {
    const int y1 = min(H, y0 + HB);  // this band: canvas rows [y0, y1)
    render_draw_rows(src, lay, base, ext_items, t, T, P, live, y0, y1, sync);
    if (live) render_store_rows((const unsigned *)(base + lay.canvas), OW + 1, out, OH, OW, y0, y1, t, T);
    if (y0 + HB < H) sync();  // the next band reuses the canvas and the item spans
  }
}

// render_store_rows for a mask: the low 16 bits of the canvas words [r1 - r0][img_stride] of the image
// rows [r0, r1), flipped, into out ([OH][OW] int16).  16-byte stores when a row is a multiple of 16
// bytes (OW % 8 == 0; `out` is then 16-byte aligned wherever an env starts), else one pixel per store.
__device__ __forceinline__ void mask_store_rows(const unsigned *img, int img_stride, int16_t *out, int OH, int OW,
                                                int r0, int r1, int t, int T) {
  if ((OW & 7) == 0) {
    uint4 *out4 = (uint4 *)out;
    const int cpr = OW >> 3;
    for (int q0 = t; q0 < (r1 - r0) * cpr; q0 += T) {
      const int q = q0 + (OH - r1) * cpr;
      const int j = q / cpr, c = q - j * cpr;
      const unsigned *srcp = img + (OH - 1 - j - r0) * img_stride + 8 * c;
      unsigned w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) w[i] = (srcp[2 * i] & 0xffffu) | (srcp[2 * i + 1] << 16);
      out4[q] = make_uint4(w[0], w[1], w[2], w[3]);
    }
  } else {
    const int n = (r1 - r0) * OW;
    for (int i0 = t; i0 < n; i0 += T) {
      const int i = i0 + (OH - r1) * OW;
      const int j = i / OW, col = i - j * OW;
      out[i] = (int16_t)(img[(OH - 1 - j - r0) * img_stride + col] & 0xffffu);
    }
  }
}

// A SpriteMask of ONE env: render_env with the slot fill policy and the int16 store.  The mask row has
// anti_aliasing 1, so `lay` and HB are those of an anti_aliasing 1 frame of the same size.
template <class Sync>
__device__ __forceinline__ void mask_env(const RenderSrc &src, const RenderLayout &lay, unsigned char *base, int t,
                                         int T, int P, bool live, int16_t *out, Sync sync, int HB) {
  const int OH = src.view[MOOG_V_HEIGHT], OW = src.view[MOOG_V_WIDTH];
  if (HB <= 0 || HB > OH) HB = OH;
  render_prepare(src, lay, base, t, T, live, sync);
#pragma unroll 1
  for (int y0 = 0; y0 < OH; y0 += HB) {
    const int y1 = min(OH, y0 + HB);
    render_draw_rows<Sync, true>(src, lay, base, nullptr, t, T, P, live, y0, y1, sync);
    if (live) mask_store_rows((const unsigned *)(base + lay.canvas), OW + 1, out, OH, OW, y0, y1, t, T);
    if (y0 + HB < OH) sync();
  }
}

// Resample.c's inner loop over n taps of 8-bit RGBX pixels p[0], p[step], ... with the fixed-point
// coefficients k, into the channel sums r / g / b (which start at 1 << 21, the rounding term)
__device__ __forceinline__ void lanczos_taps(const unsigned *p, int step, const int *k, int n, int &r, int &g, int &b) {
  for (int y = 0; y < n; ++y) {
    const unsigned px = p[y * step];
    const int c = k[y];
    r += (int)(px & 255u) * c;
    g += (int)((px >> 8) & 255u) * c;
    b += (int)((px >> 16) & 255u) * c;
  }
}

__device__ __forceinline__ unsigned pack_clip8(int r, int g, int b) { return clip8(r) | (clip8(g) << 8) | (clip8(b) << 16); }

// output pixel xx of the horizontal pass over one canvas row
__device__ __forceinline__ unsigned resample_h(const unsigned *row, const int *bh, const int *kh, int ksize_h, int xx) {
  int r = 1 << 21, g = 1 << 21, b = 1 << 21;
  lanczos_taps(row + bh[2 * xx], 1, kh + xx * ksize_h, bh[2 * xx + 1], r, g, b);
  return pack_clip8(r, g, b);
}

// PILRenderer.__call__ with anti_aliasing > 1: Image.resize(LANCZOS) of the aa x canvas (Resample.c,
// 8 bpc: a horizontal pass into an 8-bit intermediate, then a vertical pass, with the fixed-point
// coefficients of resample_tables on the host), streamed so that the canvas never exists whole.
// The canvas is drawn in chunks of HC rows (render_draw_rows, every row exactly once); each chunk is
// resampled horizontally into a ring of R rows of OW RGBX words (lay.ring; canvas row y in ring row
// y % R), after which the next chunk reuses the canvas.  Output row yy needs the intermediate rows
// [bv[2yy], bv[2yy] + bv[2yy+1]); it is resampled vertically into the dead canvas and written out as
// soon as its last row is in the ring.  The windows are monotone in yy and at most ksize_v rows
// long, so R = HC + ksize_v rows keep every row a pending output row still reads.  A canvas that is
// one chunk (HC == H, R == H: the ring is the whole intermediate) takes the straight single pass
// instead, without ring arithmetic.  Same arguments as render_env; `lay` is the layout of an HC-row
// canvas with R ring rows.
template <class Sync>
__device__ __forceinline__ void render_env_aa(const RenderSrc &src, const RenderLayout &lay, unsigned char *base,
                                              unsigned *ext_items, int t, int T, int P, bool live, unsigned char *out,
                                              const int *resample, int ksize_h, int ksize_v, Sync sync, int HC, int R) {
  const int32_t *view = src.view;
  const int OH = view[MOOG_V_HEIGHT], OW = view[MOOG_V_WIDTH], aa = view[MOOG_V_AA];
  const int H = aa * OH, W = aa * OW, stride = W + 1;
  const int *bh = resample, *kh = bh + 2 * OW;
  const int *bv = kh + OW * ksize_h, *kv = bv + 2 * OH;
  unsigned *canvas = (unsigned *)(base + lay.canvas);
  unsigned *ring = (unsigned *)(base + lay.ring);
  render_prepare(src, lay, base, t, T, live, sync);
  if (HC >= H) {  // one chunk
    render_draw_rows(src, lay, base, ext_items, t, T, P, live, 0, H, sync);
    if (live)
      for (int i = t; i < H * OW; i += T) {
        const int yy = i / OW, xx = i - yy * OW;
        ring[i] = resample_h(canvas + yy * stride, bh, kh, ksize_h, xx);
      }
    sync();
    if (live)
      for (int i = t; i < OH * OW; i += T) {
        const int yy = i / OW, xx = i - yy * OW;
        int r = 1 << 21, g = 1 << 21, b = 1 << 21;
        lanczos_taps(ring + bv[2 * yy] * OW + xx, OW, kv + yy * ksize_v, bv[2 * yy + 1], r, g, b);
        canvas[i] = pack_clip8(r, g, b);  // the canvas is dead
      }
    sync();
    if (live) render_store_rows(canvas, OW, out, OH, OW, 0, OH, t, T);
    return;
  }
  // output rows resampled per pass: as many as the dead canvas holds
  const int stage_rows = max(1, (HC * stride) / OW);
  int next = 0;  // first output row not yet written
  int rb = 0;    // ring row of canvas row y0 (y0 % R)
#pragma unroll 1
  for (int y0 = 0; y0 < H; y0 += HC) {
    const int y1 = min(H, y0 + HC);  // this chunk: canvas rows [y0, y1)
    render_draw_rows(src, lay, base, ext_items, t, T, P, live, y0, y1, sync);
    if (live)
      for (int i = t; i < (y1 - y0) * OW; i += T) {
        const int yr = i / OW, xx = i - yr * OW;
        const int q = rb + yr;  // yr < HC <= R
        ring[(q < R ? q : q - R) * OW + xx] = resample_h(canvas + yr * stride, bh, kh, ksize_h, xx);
      }
    rb += y1 - y0;
    if (rb >= R) rb -= R;
    sync();  // the chunk's intermediate rows are in the ring; the canvas is dead
    // output rows [next, last) have their whole window in the ring (every row after the last chunk)
    int last = y1 == H ? OH : next;
    while (last < OH && bv[2 * last] + bv[2 * last + 1] <= y1) ++last;
#pragma unroll 1
    for (int r0 = next; r0 < last; r0 += stage_rows) {
      const int r1 = min(last, r0 + stage_rows);
      if (live)
        for (int i = t; i < (r1 - r0) * OW; i += T) {
          const int yr = i / OW, xx = i - yr * OW, yy = r0 + yr;
          const int ymin = bv[2 * yy], ymax = bv[2 * yy + 1];
          const int *k = kv + yy * ksize_v;
          // the window is ring rows [q, q + ymax) up to the ring's end, then from ring row 0 on
          const int q = ymin % R, n1 = min(ymax, R - q);
          int r = 1 << 21, g = 1 << 21, b = 1 << 21;
          lanczos_taps(ring + q * OW + xx, OW, k, n1, r, g, b);
          lanczos_taps(ring + xx, OW, k + n1, ymax - n1, r, g, b);
          canvas[i] = pack_clip8(r, g, b);
        }
      sync();
      if (live) render_store_rows(canvas, OW, out, OH, OW, r0, r1, t, T);
      if (r1 < OH) sync();  // the canvas is the next pass's (or chunk's) again
    }
    next = last;
  }
}

}  // namespace moog
