// Polygon rasterisation on the lattice: event properties (area-weighted sums) and to_xarray flags.
// Reference: wavebreaking/utils/index_utils.py:35-126 (calculate_properties) and
// wavebreaking/processing/events.py:66-106 (to_xarray); buffer(r)+sjoin(contains) restated as
// "inside (non-zero winding) or on the boundary or closer than r to an edge" (SURVEY.md A.5).
#include <cmath>

#include "wbk_ctx.cuh"

struct RingView {
  const u32* packed;  // packed lattice points (x | y << 16), or
  const int* xy;      // int32 (x, y) pairs, or
  int bx0, by0, bx1, by1;  // a box (n == 4, both pointers NULL): shapely.box(minx, miny, maxx, maxy)
  int n;
  __device__ __forceinline__ void get(int k, int& x, int& y) const {
    if (packed) {
      const u32 p = packed[k];
      x = wbk_px(p);
      y = wbk_py(p);
    } else if (xy) {
      x = xy[2 * k];
      y = xy[2 * k + 1];
    } else {
      x = (k == 0 || k == 1) ? bx1 : bx0;
      y = (k == 1 || k == 2) ? by1 : by0;
    }
  }
};

__device__ __forceinline__ long long ceil_div_ll(long long n, long long d) {  // d != 0
  if (d < 0) {
    n = -n;
    d = -d;
  }
  return n >= 0 ? (n + d - 1) / d : -((-n) / d);
}

__device__ __forceinline__ int ceil_div_i(int n, int d) {  // d != 0
  if (d < 0) {
    n = -n;
    d = -d;
  }
  return n >= 0 ? (n + d - 1) / d : -((-n) / d);
}

// double-double accumulation (error-free TwoSum): the area-weighted sums come out correctly rounded in
// practice, like the compensated (Kahan) group sums of pandas that the reference relies on
// (index_utils.py:94-102) -- the truncated centre-of-mass quotient is sensitive to the last bit.
struct DD {
  double hi, lo;
};
__device__ __forceinline__ void dd_add(DD& a, double v) {
  const double s = __dadd_rn(a.hi, v);
  const double bb = __dsub_rn(s, a.hi);
  const double err = __dadd_rn(__dsub_rn(a.hi, __dsub_rn(s, bb)), __dsub_rn(v, bb));
  a.hi = s;
  a.lo = __dadd_rn(a.lo, err);
}
__device__ __forceinline__ void dd_merge(DD& a, double hi, double lo) {
  dd_add(a, hi);
  a.lo = __dadd_rn(a.lo, lo);
}
// deterministic block-wide double-double sums, six at once (one pair of barriers): out[k] (rounded to double) to
// every thread.
// scratch: >= 6 * 2 * 32 + 6 doubles
__device__ inline void dd_block_sum6(DD (&v)[6], double* scratch, double (&out)[6]) {
  const int lane = wbk_lane(), warp = wbk_warp(), nwarps = wbk_nthreads() >> 5;
#pragma unroll
  for (int k = 0; k < 6; ++k) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      const double oh = __shfl_xor_sync(WBK_FULL, v[k].hi, d), ol = __shfl_xor_sync(WBK_FULL, v[k].lo, d);
      dd_merge(v[k], oh, ol);
    }
  }
  __syncthreads();
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      scratch[(k * 32 + warp) * 2] = v[k].hi;
      scratch[(k * 32 + warp) * 2 + 1] = v[k].lo;
    }
  }
  __syncthreads();
  if (warp < 6) {  // warp k reduces sum k (fixed lane order: deterministic)
    DD w;
    w.hi = lane < nwarps ? scratch[(warp * 32 + lane) * 2] : 0.0;
    w.lo = lane < nwarps ? scratch[(warp * 32 + lane) * 2 + 1] : 0.0;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      const double oh = __shfl_xor_sync(WBK_FULL, w.hi, d), ol = __shfl_xor_sync(WBK_FULL, w.lo, d);
      dd_merge(w, oh, ol);
    }
    if (lane == 0) scratch[384 + warp] = __dadd_rn(w.hi, w.lo);
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 6; ++k) out[k] = scratch[384 + k];
}

// column of the extended grid -> column of the real grid (x % nlon without the division: W < a few nlon)
__device__ __forceinline__ int fold_x(int px, int nlon) {
  while (px >= nlon) px -= nlon;
  return px;
}

// The to_xarray buffer (events.py:75-79) on a grid with dlon : dlat = p : q (reduced): r = (dlon + dlat) / 4
// degrees.  In index units a lattice point at (ex, ey) from an edge (dx, dy) is closer than r (in degrees) to the
// edge's interior iff 16 p^2 q^2 C^2 < (p + q)^2 L, with C = dx ey - dy ex, L = p^2 dx^2 + q^2 dy^2 and the foot of
// the perpendicular inside the edge (0 < D < L, D = p^2 ex dx + q^2 ey dy); closer than r to a vertex iff
// 16 (p^2 ex^2 + q^2 ey^2) < (p + q)^2.  Below aspect 3 the vertex discs hold no lattice point but the vertex itself
// (the host refuses other grids: grid_ratio), so GEOS's polygonal arcs cannot matter (SURVEY.md A.5).
struct FlagMetric {
  long long p2, q2;  // p^2, q^2 (p, q <= 64)
  long long kc, kl;  // 16 p^2 q^2, (p + q)^2
  int unit_ok;       // no lattice point off a diagonal unit step lies in the band: kc >= kl (p^2 + q^2)
};

__device__ __forceinline__ bool metric_near(const FlagMetric& m, long long ex, long long ey, long long dx, long long dy) {
  const long long D = m.p2 * ex * dx + m.q2 * ey * dy, L = m.p2 * dx * dx + m.q2 * dy * dy;
  if (D <= 0) return 16 * (m.p2 * ex * ex + m.q2 * ey * ey) < m.kl;
  if (D >= L) {
    const long long fx = ex - dx, fy = ey - dy;
    return 16 * (m.p2 * fx * fx + m.q2 * fy * fy) < m.kl;
  }
  const long long C = dx * ey - dy * ex;
  // kc C^2 reaches 2^94 for |C| < 2^33: exact in 128 bits
  return C == 0 || (__int128)m.kc * C * C < (__int128)m.kl * L;
}

// Warp-cooperative scan of lattice row y over columns [bx0, bx0 + bw): on return acc[i] is the winding number
// of (bx0 + i, y) (for points not on the boundary) and flg[i] has bit 0 / bit 1 set if the point is on the
// boundary or closer than sqrt(r2a) / sqrt(r2b) to an edge.  ANISO: bit 1 is the to_xarray rule of `fm` instead
// of sqrt(r2b).  rmax >= every radius in index units (for ANISO: >= r / min(dlon, dlat)), R = floor(rmax).
template <bool ANISO>
__device__ inline void raster_scan_row(const RingView& rv, int y, int bx0, int bw, int* acc, u32* flg, double r2a,
                                       double r2b, double rmax, int R, const FlagMetric& fm,
                                       const unsigned short* elist = nullptr, int ecount = 0) {
  const int lane = wbk_lane();
  for (int i = lane; i < bw; i += 32) {
    acc[i] = 0;
    flg[i] = 0;
  }
  __syncwarp();
  const int n = rv.n;
  const int nscan = elist ? ecount : n;  // with a row bucket only the edges that can touch this row are visited
  for (int e0 = 0; e0 < nscan; e0 += 32) {
    const int q = e0 + lane;
    if (q < nscan) {
      const int e = elist ? (int)elist[q] : q;
      int xa, ya, xb, yb;
      rv.get(e, xa, ya);
      rv.get(e + 1 == n ? 0 : e + 1, xb, yb);
      const int dx = xb - xa, dy = yb - ya;
      if (dx != 0 || dy != 0) {
        const int lo = min(ya, yb), hi = max(ya, yb);
        // winding contribution: lattice points strictly left of the crossing get +-1
        if (dy != 0 && lo <= y && y < hi) {
          const int s = dy > 0 ? 1 : -1;
          // |dx|, |y - ya| < 2^15 on grids below 32768 points per axis: the product fits an int
          const bool small = (dx < 32768 && dx > -32768 && dy < 32768 && dy > -32768);
          const long long cx = small ? (long long)(xa + ceil_div_i(dx * (y - ya), dy))
                                     : (long long)xa + ceil_div_ll((long long)dx * (y - ya), (long long)dy);
          const long long idx = cx - bx0;
          if (idx > 0) {
            atomicAdd(&acc[0], s);
            if (idx < bw) atomicAdd(&acc[(int)idx], -s);
          }
        }
        // boundary / near-edge candidates of this row
        if (y >= lo - R && y <= hi + R) {
          const long long len2 = (long long)dx * dx + (long long)dy * dy;
          if (len2 <= 2 && (ANISO ? r2a <= 0.5 && fm.unit_ok : rmax * rmax <= 0.5)) {
            // unit step of a contour ring with radii <= sqrt(1/2): every lattice point off the edge is at least
            // 1/sqrt(2) away, so only the end points qualify; the start vertex is marked here, the end vertex is the
            // start of the next edge.  (ANISO: a diagonal step's off-edge neighbours stay out of the band while
            // 16 p^2 q^2 >= (p + q)^2 (p^2 + q^2), i.e. up to aspect ~2.76.)
            const int idx = xa - bx0;
            if (ya == y && idx >= 0 && idx < bw) atomicOr(&flg[idx], 3u);
            continue;
          }
          int cl, ch;
          if (dy == 0) {
            cl = min(xa, xb) - R;
            ch = max(xa, xb) + R;
          } else {
            // candidate columns around the edge's abscissa on this row (float with a generous margin: every
            // candidate is tested exactly below)
            const float ady = fabsf((float)dy);
            const float xc = (float)xa + (float)dx * (float)(y - ya) / (float)dy;
            const float hw = (float)rmax * sqrtf((float)len2) / ady + (float)rmax + 1.0f + 1e-3f * fabsf(xc);
            cl = max((int)floorf(xc - hw), min(xa, xb) - R - 1);
            ch = min((int)ceilf(xc + hw), max(xa, xb) + R + 1);
          }
          cl = max(cl, bx0);
          ch = min(ch, bx0 + bw - 1);
          for (int px = cl; px <= ch; ++px) {
            const long long ex = px - xa, ey = y - ya;
            const long long dot = ex * dx + ey * dy;
            u32 bits = 0;
            if (dot <= 0) {
              const double d2 = (double)(ex * ex + ey * ey);
              bits = (d2 < r2a ? 1u : 0u) | (d2 < r2b ? 2u : 0u);
              if (ex == 0 && ey == 0) bits = 3u;
            } else if (dot >= len2) {
              const long long fx = px - xb, fy = y - yb;
              const double d2 = (double)(fx * fx + fy * fy);
              bits = (d2 < r2a ? 1u : 0u) | (d2 < r2b ? 2u : 0u);
              if (fx == 0 && fy == 0) bits = 3u;
            } else {
              const long long cross = (long long)dx * ey - (long long)dy * ex;
              if (cross == 0) {
                bits = 3u;
              } else {
                const double c2 = (double)cross * (double)cross, l2 = (double)len2;
                bits = (c2 < r2a * l2 ? 1u : 0u) | (c2 < r2b * l2 ? 2u : 0u);
              }
            }
            if (ANISO) bits = (bits & 1u) | (metric_near(fm, ex, ey, dx, dy) ? 2u : 0u);
            if (bits) atomicOr(&flg[px - bx0], bits);
          }
        }
      }
    }
  }
  __syncwarp();
  // inclusive prefix sum of the winding differences along the row
  int carry = 0;
  for (int i0 = 0; i0 < bw; i0 += 32) {
    const int i = i0 + lane;
    int v = i < bw ? acc[i] : 0;
    int incl = wbk_warp_incl_scan(v);
    if (i < bw) acc[i] = incl + carry;
    carry += __shfl_sync(WBK_FULL, incl, 31);
  }
  __syncwarp();
}

// ------------------------------------------------------------------------------------------ event list
__global__ void __launch_bounds__(1024) event_list_kernel(WbkIdx x, int J, int njobs) {
  __shared__ int sscan[40];
  const int n = 3 * njobs;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int kind = i / njobs, job = i - kind * njobs;
    x.ev_off[i] = x.ev_count[kind * J + job];
  }
  __syncthreads();
  const int total = wbk_block_excl_scan(x.ev_off, n, sscan);
  if (threadIdx.x == 0) {
    x.ev_off[n] = total;
    x.total[1] = total;
  }
}

#define RS_THREADS 256
#define RS_EVENT_ROWCAP 512  // row-buffer columns of the event rasteriser (wider events are scanned in chunks)
#define RS_RING_CAP 4096     // ring vertices staged in shared memory per event
#define RS_ROWS_CAP 1024     // lattice rows of an event's bounding box that get an edge bucket
#define RS_EDGE_CAP 8192     // edge incidences in the row buckets
#define RS_PRE 4             // 32-column groups of a row whose field values are prefetched before the scan
#define RS_NO_INTENSITY (-1)  // events_raster_kernel without an intensity field

// how the intensity is stored: flip bit 0 / bit 1 = latitudes / longitudes descending; for packed int16 the CF packing
// value = float64(s) * scale + offset (two roundings), s == fill -> NaN (fill outside the int16 range: no fill value)
struct RsInten {
  int flip, fill;
  double scale, offset;
};

// r2_flag: the squared flag radius in cells (dlon == dlat), or with ANISO the squared extent r / min(dlon, dlat) of
// fm's band, which is below one cell: R and the margins below are those of r2_prop wherever that is >= 1 cell.
// IT: the intensity's dtype (WBK_F32 / WBK_F64 / WBK_I16), or RS_NO_INTENSITY (its sum stays 0 and `intensity` is not
// read).  The intensity is read in its stored orientation (ist.flip) and widened to double, or decoded for WBK_I16, so
// the sums equal those of a converted (decoded), re-oriented copy bit for bit.
template <typename T, bool ANISO, int IT>
__global__ void __launch_bounds__(RS_THREADS, 3)
events_raster_kernel(WbkDev d, WbkIdx x, const int* __restrict__ job_off, const int* __restrict__ pt_off,
                     const u32* __restrict__ pts, const double* __restrict__ area, const T* __restrict__ data,
                     const void* __restrict__ intensity, RsInten ist, int8_t* __restrict__ flags, int ntime, int nlevels,
                     int J, int njobs, double r2_prop, double r2_flag, FlagMetric fm, int rowcap) {
  WBK_DYN_SMEM(int, sm);
  __shared__ int s_box[5];
  __shared__ int s_scan[40];
  const int tid = threadIdx.x, lane = wbk_lane(), warp = wbk_warp(), nwarps = blockDim.x >> 5;
  int* acc = sm + (size_t)warp * 2 * rowcap;
  u32* flg = reinterpret_cast<u32*>(acc + rowcap);
  const int nlat = d.nlat, nlon = d.nlon, W = d.W;
  const double rmax = sqrt(r2_prop > r2_flag ? r2_prop : r2_flag);
  const int R = (int)floor(rmax);
  const int nlist = 3 * njobs;
  const int total = x.ev_off[nlist];
  (void)job_off;
  for (int w = blockIdx.x; w < total; w += gridDim.x) {
    int lo = 0, hi = nlist - 1;
    while (lo < hi) {
      int mid = (lo + hi + 1) >> 1;
      if (x.ev_off[mid] <= w) lo = mid; else hi = mid - 1;
    }
    const int kind = lo / njobs, job = lo - kind * njobs, e = w - x.ev_off[lo];
    int* ev = x.ev_int + (((size_t)kind * J + job) * x.EC + e) * WBK_EV_INTS;
    double* evf = x.ev_f64 + (((size_t)kind * J + job) * x.EC + e) * WBK_EV_F64;
    const int t = job / nlevels;
    RingView rv;
    rv.xy = nullptr;
    if (kind == WBK_EV_OVERTURNING) {
      rv.packed = nullptr;
      rv.bx0 = ev[3]; rv.by0 = ev[4]; rv.bx1 = ev[5]; rv.by1 = ev[6];
      rv.n = 4;
    } else {
      rv.packed = pts + pt_off[ev[0]] + ev[1];
      rv.n = ev[2] - ev[1] + 1;
      rv.bx0 = rv.by0 = rv.bx1 = rv.by1 = 0;
    }
    // bounding box of the vertices (rings that fit are staged in shared memory: every row scans all edges)
    if (tid == 0) {
      s_box[0] = 0x7fffffff; s_box[1] = 0x7fffffff; s_box[2] = -1; s_box[3] = -1;
    }
    __syncthreads();
    {
      u32* sring = reinterpret_cast<u32*>(sm + (size_t)nwarps * 2 * rowcap);
      const bool stage = rv.packed != nullptr && rv.n <= RS_RING_CAP;
      int x0 = 0x7fffffff, y0 = 0x7fffffff, x1 = -1, y1 = -1;
      for (int k = tid; k < rv.n; k += blockDim.x) {
        int vx, vy;
        rv.get(k, vx, vy);
        if (stage) sring[k] = rv.packed[k];
        x0 = min(x0, vx); x1 = max(x1, vx); y0 = min(y0, vy); y1 = max(y1, vy);
      }
      x0 = wbk_warp_min(x0); y0 = wbk_warp_min(y0); x1 = wbk_warp_max(x1); y1 = wbk_warp_max(y1);
      if (lane == 0) {
        atomicMin(&s_box[0], x0); atomicMin(&s_box[1], y0); atomicMax(&s_box[2], x1); atomicMax(&s_box[3], y1);
      }
      if (stage) rv.packed = sring;
    }
    __syncthreads();
    const int vx0 = s_box[0], vy0 = s_box[1], vx1 = s_box[2], vy1 = s_box[3];
    // 0: all vertices on the real grid, 1: straddles the last meridian (host clips), 2: entirely in the extension
    const int split = vx1 < nlon ? 0 : (vx0 >= nlon ? 2 : 1);
    const int shift = split == 2 ? nlon : 0;
    // overturning boxes with radii below one cell: the members are exactly the lattice points of the closed box
    // (every other lattice point is at least one cell away), no winding / near-edge scan needed
    const bool boxfast = kind == WBK_EV_OVERTURNING && rmax < 1.0;
    const int mrg = boxfast ? 0 : R + 1;
    const int bx0 = max(vx0 - mrg, 0), bx1 = min(vx1 + mrg, W - 1);
    const int by0 = max(vy0 - mrg, 0), by1 = min(vy1 + mrg, nlat - 1);
    const int bw = bx1 - bx0 + 1;
    // row buckets: edge e is listed under every lattice row it can touch (its y-span widened by R), so a row
    // visits a handful of edges instead of the whole ring
    const int nrows = by1 - by0 + 1;
    int* rcount = reinterpret_cast<int*>(sm + (size_t)nwarps * 2 * rowcap + RS_RING_CAP);  // [RS_ROWS_CAP + 1]
    int* rcur = rcount + RS_ROWS_CAP + 1;                                                   // [RS_ROWS_CAP]
    unsigned short* redge = reinterpret_cast<unsigned short*>(rcur + RS_ROWS_CAP);          // [RS_EDGE_CAP]
    bool bucketed = rv.n <= 65535 && nrows <= RS_ROWS_CAP && rv.n > 64;
    if (bucketed) {
      for (int i = tid; i <= nrows; i += blockDim.x) rcount[i] = 0;
      __syncthreads();
      for (int e = tid; e < rv.n; e += blockDim.x) {
        int xa, ya, xb, yb;
        rv.get(e, xa, ya);
        rv.get(e + 1 == rv.n ? 0 : e + 1, xb, yb);
        const int lo = max(min(ya, yb) - R, by0), hi = min(max(ya, yb) + R, by1);
        for (int y = lo; y <= hi; ++y) atomicAdd(&rcount[y - by0], 1);
      }
      __syncthreads();
      const int ninc = wbk_block_excl_scan(rcount, nrows, s_scan);
      if (tid == 0) rcount[nrows] = ninc;
      for (int i = tid; i < nrows; i += blockDim.x) rcur[i] = rcount[i];
      __syncthreads();
      bucketed = rcount[nrows] <= RS_EDGE_CAP;  // uniform
      if (bucketed) {
        for (int e = tid; e < rv.n; e += blockDim.x) {
          int xa, ya, xb, yb;
          rv.get(e, xa, ya);
          rv.get(e + 1 == rv.n ? 0 : e + 1, xb, yb);
          const int lo = max(min(ya, yb) - R, by0), hi = min(max(ya, yb) + R, by1);
          for (int y = lo; y <= hi; ++y) redge[atomicAdd(&rcur[y - by0], 1)] = (unsigned short)e;
        }
      }
      __syncthreads();
    }
    DD s_a = {0, 0}, s_v = {0, 0}, s_i = {0, 0}, s_x = {0, 0}, s_y = {0, 0}, s_n = {0, 0};
    for (int y = by0 + warp; y <= by1; y += nwarps) {
     const unsigned short* elist = bucketed ? redge + rcount[y - by0] : nullptr;
     const int ecount = bucketed ? rcount[y - by0 + 1] - rcount[y - by0] : 0;
     for (int cx0 = bx0; cx0 <= bx1; cx0 += rowcap) {  // wide events: the row is scanned in column chunks
      const int cw = min(rowcap, bx1 - cx0 + 1);
      const size_t rowbase = ((size_t)t * nlat + y) * nlon;
      // the field values of the row's first RS_PRE * 32 columns are requested before the scan, so their DRAM latency
      // hides behind it (otherwise every 32-column step of the member loop waits for a load on its own)
      T dpre[RS_PRE];
#pragma unroll
      for (int k = 0; k < RS_PRE; ++k) {
        dpre[k] = (T)0;
        if (32 * k < cw) {  // warp-uniform
          const int px = cx0 + lane + 32 * k;
          if (lane + 32 * k < cw) dpre[k] = data[rowbase + fold_x(px, nlon)];
        }
      }
      int8_t* frow = flags ? flags + (((size_t)kind * ntime + t) * nlat + y) * nlon : nullptr;
      if (!boxfast) raster_scan_row<ANISO>(rv, y, cx0, cw, acc, flg, r2_prop, r2_flag, rmax, R, fm, elist, ecount);
      const double a = area[y];
      int row_members = 0;
      auto visit = [&](int i, double dv) {
        const bool in = boxfast || acc[i] != 0;
        const u32 f = boxfast ? 3u : flg[i];
        const int px = cx0 + i;
        if (in || (f & 1u)) {
          const int xf = fold_x(px, nlon);
          // sum(a) and sum(y * a) have one value per row: counted here, added once per row below
          dd_add(s_v, __dmul_rn(a, dv));
          if (IT != RS_NO_INTENSITY) {
            const int ys = (ist.flip & 1) ? nlat - 1 - y : y, xs = (ist.flip & 2) ? nlon - 1 - xf : xf;
            const size_t k = ((size_t)t * nlat + ys) * nlon + xs;
            double iv;
            if (IT == WBK_I16) {
              const short s = static_cast<const short*>(intensity)[k];
              iv = (int)s == ist.fill ? __longlong_as_double(0x7ff8000000000000LL)
                                      : __dadd_rn(__dmul_rn((double)s, ist.scale), ist.offset);
            } else {
              iv = IT == WBK_F32 ? (double)static_cast<const float*>(intensity)[k]
                                 : static_cast<const double*>(intensity)[k];
            }
            dd_add(s_i, __dmul_rn(a, iv));
          }
          dd_add(s_x, __dmul_rn((double)px, a));
          ++row_members;
        }
        if (frow && split != 1 && (in || (f & 2u))) {
          const int xf = px - shift;
          if (xf >= 0 && xf < nlon) frow[xf] = 1;
        }
      };
#pragma unroll
      for (int k = 0; k < RS_PRE; ++k)
        if (lane + 32 * k < cw) visit(lane + 32 * k, (double)dpre[k]);
      for (int i = lane + 32 * RS_PRE; i < cw; i += 32) {
        const int px = cx0 + i;
        const int xf = fold_x(px, nlon);
        visit(i, (double)data[rowbase + xf]);
      }
      if (row_members) {
        // n identical addends: n * value is exact in double-double (two-product by FMA), like adding them one by one
        const double nrm = (double)row_members;
        const double ya = __dmul_rn((double)y, a);
        const double pa = __dmul_rn(nrm, a), pa_lo = __fma_rn(nrm, a, -pa);
        const double py = __dmul_rn(nrm, ya), py_lo = __fma_rn(nrm, ya, -py);
        dd_merge(s_a, pa, pa_lo);
        dd_merge(s_y, py, py_lo);
        dd_add(s_n, nrm);
      }
      __syncwarp();
     }
    }
    DD sums6[6] = {s_a, s_v, s_i, s_x, s_y, s_n};
    double tot6[6];
    dd_block_sum6(sums6, reinterpret_cast<double*>(sm), tot6);  // the row buffers are free by now
    if (tid == 0) {
      evf[0] = tot6[0]; evf[1] = tot6[1]; evf[2] = tot6[2]; evf[3] = tot6[3]; evf[4] = tot6[4]; evf[5] = tot6[5];
      if (kind != WBK_EV_OVERTURNING) {
        ev[3] = vx0; ev[4] = vy0; ev[5] = vx1; ev[6] = vy1;
      }
      ev[8] = split;
      if (split == 1) {  // work list of the meridian split
        const int pos = atomicAdd(&x.split_count[3], 1);
        if (pos < x.SPR) x.split_list[pos] = w;
        else atomicOr(&x.split_count[2], 1);
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------ meridian split
// utils/index_utils.py:148-173 for the events that have vertices on both sides of the last meridian: the faces
// of the ring left of x = nlon-1 and right of x = nlon are kept as separate pieces (no bridge edges between
// faces: crossings on the cut line are sorted and paired, every chain of kept vertices is linked from its exit
// crossing to the paired entry crossing), cut vertices are truncated to ints and x is folded with % nlon.
// One thread per event (the work is sequential and tiny); pieces go to a vertex pool + ring list that
// split_raster_kernel then rasterises into the flag grids.
#define SPLIT_MAX_CHAINS 24

struct SplitChain {
  int off, cnt;            // vertices in the pool (chain scratch)
  long long yin_n, yin_d;  // entry / exit ordinates on the cut line as exact fractions (den > 0)
  long long yout_n, yout_d;
};

__device__ __forceinline__ bool frac_less(long long an, long long ad, long long bn, long long bd) {
  return an * bd < bn * ad;
}
__device__ __forceinline__ bool frac_eq(long long an, long long ad, long long bn, long long bd) {
  return an * bd == bn * ad;
}

// clip one ring against x = c keeping x <= c (keep_le) or x >= c; appends pieces to the ring list
__device__ void split_clip_side(const RingView& rv, int c, bool keep_le, int nlon, int t, int kind, int ev, WbkIdx& x) {
  const int n = rv.n;
  int nin = 0;
  for (int k = 0; k < n; ++k) {
    int vx, vy;
    rv.get(k, vx, vy);
    nin += (keep_le ? vx < c : vx > c) ? 1 : 0;
  }
  if (nin == 0) return;
  SplitChain ch[SPLIT_MAX_CHAINS];
  int nch = 0;
  // scratch space for the chains: at most n + 2 * chains vertices
  const int scratch_cap = n + 2 * SPLIT_MAX_CHAINS;
  const int sbase = atomicAdd(&x.split_count[0], scratch_cap);
  if (sbase + scratch_cap > x.SPV) {
    atomicOr(&x.split_count[2], 1);
    return;
  }
  int* sxy = x.split_xy + 2 * (size_t)sbase;
  int sp = 0;
  // A chain is a maximal run of vertices STRICTLY beyond the line; it is entered and left through a crossing point on
  // the line: the neighbouring ring vertex if that one lies on the line, else the exact intersection of the edge.
  // Ring edges that run along the line belong to no chain -- whether they bound a face is decided by the pairing of
  // the crossings below, as in the overlay + polygonize of the reference (index_utils.py:158-163): no vertex on the
  // line sticks out of a face as a zero-area antenna, parts that only meet along the line stay separate faces.
  auto inside = [&](int k) {
    int vx, vy;
    rv.get(k, vx, vy);
    return keep_le ? vx < c : vx > c;
  };
  if (nin == n) {
    ch[0].off = 0;
    ch[0].cnt = n;
    for (int k = 0; k < n; ++k) {
      int vx, vy;
      rv.get(k, vx, vy);
      sxy[2 * k] = vx;
      sxy[2 * k + 1] = vy;
    }
    nch = -1;  // whole ring
  } else {
    int start = 0;
    for (int k = 0; k < n; ++k)
      if (inside(k) && !inside(k == 0 ? n - 1 : k - 1)) {
        start = k;
        break;
      }
    int k = start, visited = 0;
    while (visited < n) {
      const int prev = k == 0 ? n - 1 : k - 1;
      if (inside(k) && !inside(prev)) {
        if (nch >= SPLIT_MAX_CHAINS) {
          atomicOr(&x.split_count[2], 2);  // not a capacity the host can raise: reported as WBK_ST_SPLIT_CHAINS
          return;
        }
        SplitChain& cc = ch[nch];
        cc.off = sp;
        int kx, ky, px, py;
        rv.get(k, kx, ky);
        rv.get(prev, px, py);
        if (px != c) {  // entry crossing strictly inside the edge prev -> k
          long long den = (long long)kx - px, num = (long long)py * den + (long long)(c - px) * (ky - py);
          if (den < 0) { den = -den; num = -num; }
          cc.yin_n = num; cc.yin_d = den;
          sxy[2 * sp] = c;
          sxy[2 * sp + 1] = (int)(num >= 0 ? num / den : -((-num) / den));  // astype(int): truncation
          ++sp;
        } else {  // the ring vertex before the chain lies on the line: it is the crossing point
          cc.yin_n = py; cc.yin_d = 1;
          sxy[2 * sp] = c;
          sxy[2 * sp + 1] = py;
          ++sp;
        }
        int j = k;
        while (inside(j)) {
          int jx, jy;
          rv.get(j, jx, jy);
          sxy[2 * sp] = jx;
          sxy[2 * sp + 1] = jy;
          ++sp;
          j = j + 1 == n ? 0 : j + 1;
          ++visited;
        }
        const int last = j == 0 ? n - 1 : j - 1;
        int lx, ly, jx, jy;
        rv.get(last, lx, ly);
        rv.get(j, jx, jy);
        if (jx != c) {
          long long den = (long long)jx - lx, num = (long long)ly * den + (long long)(c - lx) * (jy - ly);
          if (den < 0) { den = -den; num = -num; }
          cc.yout_n = num; cc.yout_d = den;
          sxy[2 * sp] = c;
          sxy[2 * sp + 1] = (int)(num >= 0 ? num / den : -((-num) / den));
          ++sp;
        } else {  // the ring vertex after the chain lies on the line
          cc.yout_n = jy; cc.yout_d = 1;
          sxy[2 * sp] = c;
          sxy[2 * sp + 1] = jy;
          ++sp;
        }
        cc.cnt = sp - cc.off;
        ++nch;
        k = j;
      } else {
        k = k + 1 == n ? 0 : k + 1;
        ++visited;
      }
    }
  }
  // pair the crossings along the cut line (sorted by ordinate; ties: chain id, entry before exit)
  int partner[SPLIT_MAX_CHAINS];
  const int nchains = nch < 0 ? 1 : nch;
  if (nch < 0) {
    partner[0] = 0;
  } else {
    int ord[2 * SPLIT_MAX_CHAINS];  // crossing id = 2 * chain + type (0 entry, 1 exit)
    const int nc = 2 * nch;
    for (int i = 0; i < nc; ++i) {
      const int id = i;
      const long long yn = (id & 1) ? ch[id >> 1].yout_n : ch[id >> 1].yin_n;
      const long long yd = (id & 1) ? ch[id >> 1].yout_d : ch[id >> 1].yin_d;
      int pos = i;
      while (pos > 0) {
        const int o = ord[pos - 1];
        const long long on = (o & 1) ? ch[o >> 1].yout_n : ch[o >> 1].yin_n;
        const long long od = (o & 1) ? ch[o >> 1].yout_d : ch[o >> 1].yin_d;
        bool less = frac_less(yn, yd, on, od);
        if (!less && frac_eq(yn, yd, on, od)) less = id < o;  // (chain, type) order == id order
        if (!less) break;
        ord[pos] = o;
        --pos;
      }
      ord[pos] = id;
    }
    bool ok = true;
    for (int i = 0; i < nch; ++i) partner[i] = i;
    for (int i = 0; i + 1 < nc; i += 2) {
      const int a0 = ord[i], a1 = ord[i + 1];
      if ((a0 & 1) == 1 && (a1 & 1) == 0) partner[a0 >> 1] = a1 >> 1;
      else if ((a0 & 1) == 0 && (a1 & 1) == 1) partner[a1 >> 1] = a0 >> 1;
      else { ok = false; break; }
    }
    if (!ok)
      for (int i = 0; i < nch; ++i) partner[i] = i;  // non-simple ring: close every chain on itself
  }
  // faces
  bool used[SPLIT_MAX_CHAINS];
  for (int i = 0; i < nchains; ++i) used[i] = false;
  for (int f0 = 0; f0 < nchains; ++f0) {
    if (used[f0]) continue;
    // pass 1: vertex count and exact-enough doubled area (cut ordinates as double fractions)
    int cnt = 0;
    double area2 = 0.0, fx = 0, fy = 0, px = 0, py = 0;
    bool first = true;
    int cur = f0;
    int guard = 0;
    while (guard++ <= nchains) {
      for (int i = 0; i < ch[cur].cnt; ++i) {
        double vx = (double)sxy[2 * (ch[cur].off + i)], vy = (double)sxy[2 * (ch[cur].off + i) + 1];
        if (nch >= 0) {
          if (i == 0 && ch[cur].yin_d != 1) vy = (double)ch[cur].yin_n / (double)ch[cur].yin_d;
          if (i == ch[cur].cnt - 1 && ch[cur].yout_d != 1) vy = (double)ch[cur].yout_n / (double)ch[cur].yout_d;
        }
        if (first) { fx = vx; fy = vy; first = false; } else area2 += px * vy - vx * py;
        px = vx; py = vy;
        ++cnt;
      }
      cur = partner[cur];
      if (cur == f0) break;
    }
    area2 += px * fy - fx * py;
    // mark used
    cur = f0;
    guard = 0;
    while (guard++ <= nchains) {
      used[cur] = true;
      cur = partner[cur];
      if (cur == f0) break;
    }
    if (cnt < 3 || fabs(area2) < 1e-9) continue;
    // pass 2: emit (fold x, drop consecutive repeats and a closing repeat)
    const int obase = atomicAdd(&x.split_count[0], cnt);
    const int ridx = atomicAdd(&x.split_count[1], 1);
    if (obase + cnt > x.SPV || ridx >= x.SPR) {
      atomicOr(&x.split_count[2], 1);
      return;
    }
    int* oxy = x.split_xy + 2 * (size_t)obase;
    int m = 0;
    cur = f0;
    guard = 0;
    while (guard++ <= nchains) {
      for (int i = 0; i < ch[cur].cnt; ++i) {
        const int vx = sxy[2 * (ch[cur].off + i)] % nlon, vy = sxy[2 * (ch[cur].off + i) + 1];
        if (m > 0 && oxy[2 * (m - 1)] == vx && oxy[2 * (m - 1) + 1] == vy) continue;
        oxy[2 * m] = vx;
        oxy[2 * m + 1] = vy;
        ++m;
      }
      cur = partner[cur];
      if (cur == f0) break;
    }
    if (m > 1 && oxy[0] == oxy[2 * (m - 1)] && oxy[1] == oxy[2 * (m - 1) + 1]) --m;
    int* rr = x.split_ring + 4 * (size_t)ridx;
    rr[0] = obase; rr[1] = m; rr[2] = t; rr[3] = kind | (ev << 2);  // ev: index of the event in gather order
  }
}

// One warp per listed event: the lanes stage the ring in shared memory, lane 0 runs the (sequential, tiny) clipping.
#define SPLIT_WARPS 4
#define SPLIT_STAGE 2048  // ring vertices staged per warp
__global__ void __launch_bounds__(32 * SPLIT_WARPS)
split_events_kernel(WbkDev d, WbkIdx x, const int* __restrict__ pt_off, const u32* __restrict__ pts, int nlevels, int J,
                    int njobs) {
  __shared__ u32 sring[SPLIT_WARPS][SPLIT_STAGE];
  const int lane = wbk_lane(), warp = wbk_warp();
  const int nlist = 3 * njobs;
  const int count = min(x.split_count[3], x.SPR);
  for (int q = blockIdx.x * SPLIT_WARPS + warp; q < count; q += gridDim.x * SPLIT_WARPS) {
    const int w = x.split_list[q];
    int lo = 0, hi = nlist - 1;
    while (lo < hi) {
      int mid = (lo + hi + 1) >> 1;
      if (x.ev_off[mid] <= w) lo = mid; else hi = mid - 1;
    }
    const int kind = lo / njobs, job = lo - kind * njobs, e = w - x.ev_off[lo];
    const int* ev = x.ev_int + (((size_t)kind * J + job) * x.EC + e) * WBK_EV_INTS;
    RingView rv;
    rv.xy = nullptr;
    if (kind == WBK_EV_OVERTURNING) {
      rv.packed = nullptr;
      rv.bx0 = ev[3]; rv.by0 = ev[4]; rv.bx1 = ev[5]; rv.by1 = ev[6];
      rv.n = 4;
    } else {
      rv.packed = pts + pt_off[ev[0]] + ev[1];
      rv.n = ev[2] - ev[1] + 1;
      rv.bx0 = rv.by0 = rv.bx1 = rv.by1 = 0;
      __syncwarp();
      if (rv.n <= SPLIT_STAGE) {
        for (int k = lane; k < rv.n; k += 32) sring[warp][k] = rv.packed[k];
        rv.packed = sring[warp];
      }
      __syncwarp();
    }
    if (lane == 0) {
      const int t = job / nlevels;
      split_clip_side(rv, d.nlon - 1, true, d.nlon, t, kind, w, x);
      split_clip_side(rv, d.nlon, false, d.nlon, t, kind, w, x);
    }
  }
}

// rasterise the split pieces (real grid, r = 1/2 cell or with ANISO the rule of fm: processing/events.py:75-79) into
// the flag grids; rf: r / min(dlon, dlat) in cells (< 1)
template <bool ANISO>
__global__ void __launch_bounds__(RS_THREADS)
split_raster_kernel(WbkIdx x, int nlat, int nlon, int ntime, int8_t* __restrict__ flags, int rowcap, int* status,
                    FlagMetric fm, double rf) {
  WBK_DYN_SMEM(int, sm);
  __shared__ int s_box[4];
  const int tid = threadIdx.x, lane = wbk_lane(), warp = wbk_warp(), nwarps = blockDim.x >> 5;
  // the work list, the vertex pool or the ring list of the clipper overflowed: some straddling event is missing from
  // the flag grids -> the host regrows event_cap (which sizes these arenas) and re-runs the batch
  if (blockIdx.x == 0 && tid == 0) {
    if (x.split_count[2] & 1) atomicOr(&status[0], (int)WBK_ST_EVENT_OVERFLOW);
    if (x.split_count[2] & 2) atomicOr(&status[0], (int)WBK_ST_SPLIT_CHAINS);
  }
  int* acc = sm + (size_t)warp * 2 * rowcap;
  u32* flg = reinterpret_cast<u32*>(acc + rowcap);
  const int nrings = min(x.split_count[1], x.SPR);
  for (int r = blockIdx.x; r < nrings; r += gridDim.x) {
    const int* rr = x.split_ring + 4 * (size_t)r;
    RingView rv;
    rv.packed = nullptr;
    rv.xy = x.split_xy + 2 * (size_t)rr[0];
    rv.n = rr[1];
    rv.bx0 = rv.by0 = rv.bx1 = rv.by1 = 0;
    const int t = rr[2], kind = rr[3] & 3;
    if (tid == 0) {
      s_box[0] = 0x7fffffff; s_box[1] = 0x7fffffff; s_box[2] = -1; s_box[3] = -1;
    }
    __syncthreads();
    {
      int x0 = 0x7fffffff, y0 = 0x7fffffff, x1 = -1, y1 = -1;
      for (int k = tid; k < rv.n; k += blockDim.x) {
        int vx, vy;
        rv.get(k, vx, vy);
        x0 = min(x0, vx); x1 = max(x1, vx); y0 = min(y0, vy); y1 = max(y1, vy);
      }
      x0 = wbk_warp_min(x0); y0 = wbk_warp_min(y0); x1 = wbk_warp_max(x1); y1 = wbk_warp_max(y1);
      if (lane == 0) {
        atomicMin(&s_box[0], x0); atomicMin(&s_box[1], y0); atomicMax(&s_box[2], x1); atomicMax(&s_box[3], y1);
      }
    }
    __syncthreads();
    const int bx0 = max(s_box[0] - 1, 0), bx1 = min(s_box[2] + 1, nlon - 1);
    const int by0 = max(s_box[1] - 1, 0), by1 = min(s_box[3] + 1, nlat - 1);
    const int bw = bx1 - bx0 + 1;
    if (rv.n > 0 && bw > 0) {
      for (int y = by0 + warp; y <= by1; y += nwarps) {
        if (ANISO) raster_scan_row<true>(rv, y, bx0, bw, acc, flg, rf * rf, rf * rf, rf, 0, fm);
        else raster_scan_row<false>(rv, y, bx0, bw, acc, flg, 0.25, 0.25, 0.5, 0, fm);
        for (int i = lane; i < bw; i += 32)
          if (acc[i] != 0 || (flg[i] & (ANISO ? 2u : 1u))) flags[(((size_t)kind * ntime + t) * nlat + y) * nlon + (bx0 + i)] = 1;
        __syncwarp();
      }
    }
    __syncthreads();
  }
}

static int raster_rowcap(int W) { return (W + 2 + 31) & ~31; }

// dlon : dlat as the reduced ratio p : q of the to_xarray metric (FlagMetric).  Spacings within 1e-9 (relative) of
// each other are the isotropic grid p = q = 1 (fm->p2 == 0: the radius-in-cells path).  Otherwise the ratio of the two
// doubles must be exactly p / q with p, q <= 64 (so the products of metric_near stay exact) and max / min < 3 (vertex
// discs without lattice points); anything else sets the error (prefixed with `who`) and returns WBK_ERR_INVALID.
static int grid_ratio(const char* who, double dlon, double dlat, FlagMetric* fm) {
  *fm = FlagMetric{0, 0, 0, 0, 0};
  if (!(dlon > 0) || !(dlat > 0) || !std::isfinite(dlon) || !std::isfinite(dlat)) {
    wbk_set_error("%s: grid spacings dlon=%.17g, dlat=%.17g must be positive and finite", who, dlon, dlat);
    return WBK_ERR_INVALID;
  }
  if (fabs(dlon - dlat) <= 1e-9 * fabs(dlon)) return WBK_OK;
  // dlon / dlat = (a / b) * 2^k with a, b odd integers (53-bit significands)
  int ea, eb;
  unsigned long long a = (unsigned long long)ldexp(frexp(dlon, &ea), 53);
  unsigned long long b = (unsigned long long)ldexp(frexp(dlat, &eb), 53);
  int k = ea - eb;
  while (!(a & 1)) { a >>= 1; ++k; }
  while (!(b & 1)) { b >>= 1; --k; }
  unsigned long long g = a, h = b;
  while (h) { const unsigned long long t = g % h; g = h; h = t; }
  a /= g;
  b /= g;
  while (k > 0 && a <= 64) { a <<= 1; --k; }
  while (k < 0 && b <= 64) { b <<= 1; ++k; }
  if (k != 0 || a > 64 || b > 64) {
    wbk_set_error("%s: dlon=%.17g / dlat=%.17g is not a ratio p/q of integers <= 64", who, dlon, dlat);
    return WBK_ERR_INVALID;
  }
  const long long p = (long long)a, q = (long long)b;
  if (p >= 3 * q || q >= 3 * p) {
    wbk_set_error("%s: dlon=%.17g, dlat=%.17g: flag grids need an aspect ratio max(dlon, dlat) / min(dlon, dlat) < 3",
                  who, dlon, dlat);
    return WBK_ERR_INVALID;
  }
  fm->p2 = p * p;
  fm->q2 = q * q;
  fm->kc = 16 * p * p * q * q;
  fm->kl = (p + q) * (p + q);
  fm->unit_ok = fm->kc >= fm->kl * (fm->p2 + fm->q2);
  return WBK_OK;
}


// one instantiation per (anisotropic metric, intensity dtype or none) of the data type T
template <typename T>
static int launch_events_raster(bool aniso, int it, size_t smem, cudaStream_t st, int grid, const WbkDev& d,
                                const WbkIdx& x, const int* d_job_off, const int* d_pt_off, const uint32_t* d_pts,
                                const double* area, const T* data, const void* intensity, const RsInten& ist,
                                int8_t* d_flags,
                                int ntime, int nlevels, int J, int njobs, double r2_prop, double r2_flag,
                                const FlagMetric& fm, int rowcap) {
  decltype(&events_raster_kernel<T, false, RS_NO_INTENSITY>) kern;
  if (it == WBK_F32)
    kern = aniso ? events_raster_kernel<T, true, WBK_F32> : events_raster_kernel<T, false, WBK_F32>;
  else if (it == WBK_F64)
    kern = aniso ? events_raster_kernel<T, true, WBK_F64> : events_raster_kernel<T, false, WBK_F64>;
  else if (it == WBK_I16)
    kern = aniso ? events_raster_kernel<T, true, WBK_I16> : events_raster_kernel<T, false, WBK_I16>;
  else
    kern = aniso ? events_raster_kernel<T, true, RS_NO_INTENSITY> : events_raster_kernel<T, false, RS_NO_INTENSITY>;
  WBK_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  WBK_LAUNCH(KID_EVENTS_RASTER, kern, dim3(grid), dim3(RS_THREADS), smem, st, d, x, d_job_off, d_pt_off,
             (const u32*)d_pts, area, data, intensity, ist, d_flags, ntime, nlevels, J, njobs, r2_prop, r2_flag, fm,
             rowcap);
  WBK_LAUNCH_CHECK();
  return WBK_OK;
}

extern "C" int wbk_events_raster(wbk_ctx* ctx, const int* d_job_off, const int* d_pt_off, const uint32_t* d_pts,
                                 const double* d_coords, const void* d_data, int dtype, const void* d_intensity,
                                 int intensity_dtype, const wbk_smooth_opts* intensity_opts, int ntime,
                                 int8_t* d_flags, const wbk_index_params* prm, void* stream) {
  if (!ctx || !d_job_off || !d_pt_off || !d_coords || !d_data || !prm || ntime < 0) {
    wbk_set_error("wbk_events_raster: invalid argument");
    return WBK_ERR_INVALID;
  }
  if (dtype != WBK_F32 && dtype != WBK_F64) {
    wbk_set_error("wbk_events_raster: unsupported dtype");
    return WBK_ERR_INVALID;
  }
  if (d_intensity && intensity_dtype != WBK_F32 && intensity_dtype != WBK_F64 && intensity_dtype != WBK_I16) {
    wbk_set_error("wbk_events_raster: unsupported intensity dtype %d", intensity_dtype);
    return WBK_ERR_INVALID;
  }
  if (d_intensity && intensity_dtype == WBK_I16 && !intensity_opts) {
    wbk_set_error("wbk_events_raster: a packed int16 intensity needs its packing (intensity_opts)");
    return WBK_ERR_INVALID;
  }
  FlagMetric fm;
  if (d_flags) {
    const int rc = grid_ratio("wbk_events_raster", prm->dlon, prm->dlat, &fm);
    if (rc != WBK_OK) return rc;
  } else {
    fm = FlagMetric{0, 0, 0, 0, 0};
  }
  const bool aniso = fm.p2 != 0;
  cudaStream_t st = (cudaStream_t)stream;
  WbkDev& d = ctx->d;
  const int njobs = ctx->njobs, J = ctx->caps.max_jobs;
  if (d_flags && ntime > 0)
    WBK_CUDA_CHECK(cudaMemsetAsync(d_flags, 0, (size_t)3 * ntime * d.nlat * d.nlon, st));
  if (njobs == 0) return WBK_OK;
  WBK_CUDA_CHECK(cudaMemsetAsync(ctx->x.split_count, 0, 16, st));  // cursors of the meridian split (filled by the rasteriser)
  WBK_LAUNCH(KID_EVENT_LIST, event_list_kernel, dim3(1), dim3(1024), 0, st, ctx->x, J, njobs);
  WBK_LAUNCH_CHECK();
  const double r_prop = (prm->dlon + prm->dlat) / 2.0 / 2.0;  // index units (index_utils.py:47-50)
  // degrees -> cells (anisotropic: the larger of the band's two extents, r / dlon and r / dlat)
  const double r_flag = !d_flags ? r_prop : r_prop / (aniso ? fmin(prm->dlon, prm->dlat) : prm->dlon);
  const int rowcap = raster_rowcap(d.W) < RS_EVENT_ROWCAP ? raster_rowcap(d.W) : RS_EVENT_ROWCAP;
  int nwarps = RS_THREADS / 32;
  const size_t smem = (size_t)nwarps * 2 * rowcap * sizeof(int) + (size_t)RS_RING_CAP * sizeof(u32) +
                      (size_t)(2 * RS_ROWS_CAP + 1) * sizeof(int) + (size_t)RS_EDGE_CAP * sizeof(unsigned short);
  const double* area = d_coords + 3 * (size_t)d.nlat;
  const int grid = 148 * 9;
  const int it = d_intensity ? intensity_dtype : RS_NO_INTENSITY;
  RsInten ist{0, 0x7fffffff, 1.0, 0.0};
  if (intensity_opts) {
    ist.flip = (intensity_opts->flip_lat ? 1 : 0) | (intensity_opts->flip_lon ? 2 : 0);
    if (intensity_dtype == WBK_I16) {
      ist.fill = intensity_opts->has_fill ? intensity_opts->fill : 0x7fffffff;
      ist.scale = intensity_opts->scale;
      ist.offset = intensity_opts->offset;
    }
  }
  int rc;
  if (dtype == WBK_F32)
    rc = launch_events_raster<float>(aniso, it, smem, st, grid, d, ctx->x, d_job_off, d_pt_off, d_pts, area,
                                     (const float*)d_data, d_intensity, ist, d_flags, ntime, ctx->nlevels, J, njobs,
                                     r_prop * r_prop, r_flag * r_flag, fm, rowcap);
  else
    rc = launch_events_raster<double>(aniso, it, smem, st, grid, d, ctx->x, d_job_off, d_pt_off, d_pts, area,
                                      (const double*)d_data, d_intensity, ist, d_flags, ntime, ctx->nlevels, J, njobs,
                                      r_prop * r_prop, r_flag * r_flag, fm, rowcap);
  if (rc != WBK_OK) return rc;
  ctx->split_clipped = d_flags != nullptr;
  if (d_flags) {
    // events straddling the last meridian: clip on the device, rasterise the pieces
    WBK_LAUNCH(KID_SPLIT, split_events_kernel, dim3(148 * 2), dim3(32 * SPLIT_WARPS), 0, st, d, ctx->x, d_pt_off,
               (const u32*)d_pts, ctx->nlevels, J, njobs);
    WBK_LAUNCH_CHECK();
    const int rc2 = raster_rowcap(d.nlon);
    const size_t smem2 = (size_t)(RS_THREADS / 32) * 2 * rc2 * sizeof(int);
    auto split_raster = aniso ? split_raster_kernel<true> : split_raster_kernel<false>;
    WBK_CUDA_CHECK(cudaFuncSetAttribute(split_raster, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
    WBK_LAUNCH(KID_SPLIT_RASTER, split_raster, dim3(148 * 2), dim3(RS_THREADS), smem2, st, ctx->x, d.nlat, d.nlon,
               ntime, d_flags, rc2, d.status, fm, r_flag);
    WBK_LAUNCH_CHECK();
  }
  return WBK_OK;
}

// The clipper alone, for callers that want the pieces of the straddling events (wbk_split_fetch) but no flag grids
extern "C" int wbk_split_clip(wbk_ctx* ctx, const int* d_pt_off, const uint32_t* d_pts, void* stream) {
  if (!ctx || !d_pt_off) {
    wbk_set_error("wbk_split_clip: invalid argument");
    return WBK_ERR_INVALID;
  }
  if (ctx->split_clipped || ctx->njobs == 0) return WBK_OK;  // wbk_events_raster already did it for its flag grids
  cudaStream_t st = (cudaStream_t)stream;
  WBK_LAUNCH(KID_SPLIT, split_events_kernel, dim3(148 * 2), dim3(32 * SPLIT_WARPS), 0, st, ctx->d, ctx->x, d_pt_off,
             (const u32*)d_pts, ctx->nlevels, ctx->caps.max_jobs, ctx->njobs);
  WBK_LAUNCH_CHECK();
  ctx->split_clipped = 1;
  return WBK_OK;
}

// ------------------------------------------------------------------------------------------ generic rings
// r2: squared radius in cells, or with ANISO the squared extent of fm's band (r / min(dlon, dlat))^2
template <bool ANISO>
__global__ void __launch_bounds__(RS_THREADS)
rings_raster_kernel(const int* __restrict__ xy, const int* __restrict__ ring_off, const int* __restrict__ ring_t,
                    int nrings, int nlat, int nlon, int ntime, double r2, int8_t* out_i8, int* owner, int rowcap,
                    FlagMetric fm) {
  WBK_DYN_SMEM(int, sm);
  __shared__ int s_box[4];
  const int tid = threadIdx.x, lane = wbk_lane(), warp = wbk_warp(), nwarps = blockDim.x >> 5;
  int* acc = sm + (size_t)warp * 2 * rowcap;
  u32* flg = reinterpret_cast<u32*>(acc + rowcap);
  const double rmax = sqrt(r2);
  const int R = (int)floor(rmax);
  for (int r = blockIdx.x; r < nrings; r += gridDim.x) {
    RingView rv;
    rv.packed = nullptr;
    rv.xy = xy + 2 * (size_t)ring_off[r];
    rv.n = ring_off[r + 1] - ring_off[r];
    rv.bx0 = rv.by0 = rv.bx1 = rv.by1 = 0;
    const int t = ring_t[r];
    if (tid == 0) {
      s_box[0] = 0x7fffffff; s_box[1] = 0x7fffffff; s_box[2] = -0x7fffffff; s_box[3] = -0x7fffffff;
    }
    __syncthreads();
    {
      int x0 = 0x7fffffff, y0 = 0x7fffffff, x1 = -0x7fffffff, y1 = -0x7fffffff;
      for (int k = tid; k < rv.n; k += blockDim.x) {
        int vx, vy;
        rv.get(k, vx, vy);
        x0 = min(x0, vx); x1 = max(x1, vx); y0 = min(y0, vy); y1 = max(y1, vy);
      }
      x0 = wbk_warp_min(x0); y0 = wbk_warp_min(y0); x1 = wbk_warp_max(x1); y1 = wbk_warp_max(y1);
      if (lane == 0) {
        atomicMin(&s_box[0], x0); atomicMin(&s_box[1], y0); atomicMax(&s_box[2], x1); atomicMax(&s_box[3], y1);
      }
    }
    __syncthreads();
    const int bx0 = max(s_box[0] - R - 1, 0), bx1 = min(s_box[2] + R + 1, nlon - 1);
    const int by0 = max(s_box[1] - R - 1, 0), by1 = min(s_box[3] + R + 1, nlat - 1);
    const int bw = bx1 - bx0 + 1;
    if (rv.n > 0 && bw > 0 && t >= 0 && t < ntime) {
      for (int y = by0 + warp; y <= by1; y += nwarps) {
        raster_scan_row<ANISO>(rv, y, bx0, bw, acc, flg, r2, r2, rmax, R, fm);
        for (int i = lane; i < bw; i += 32) {
          if (acc[i] != 0 || (flg[i] & (ANISO ? 2u : 1u))) {
            const size_t o = ((size_t)t * nlat + y) * nlon + (bx0 + i);
            if (out_i8) out_i8[o] = 1;
            if (owner) atomicMax(&owner[o], r);
          }
        }
        __syncwarp();
      }
    }
    __syncthreads();
  }
}

__global__ void owner_fill_kernel(int* owner, size_t n, int v) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) owner[i] = v;
}
__global__ void owner_apply_kernel(const int* __restrict__ owner, const double* __restrict__ val, double* __restrict__ out, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int r = owner[i];
    if (r >= 0) out[i] = val[r];
  }
}

// r2: squared radius in cells (fm.p2 == 0), or the squared extent of fm's band
static int rasterize_rings(const char* who, const int* d_xy, const int* d_ring_off, const int* d_ring_t,
                           const double* d_ring_val, int nrings, int nlat, int nlon, int ntime, double r2,
                           const FlagMetric& fm, int8_t* d_out_i8, double* d_out_f64, int* d_owner, void* stream) {
  if (nrings < 0 || nlat < 1 || nlon < 1 || ntime < 0 || !(r2 >= 0) || (!d_out_i8 && !d_out_f64) ||
      (d_out_f64 && (!d_owner || !d_ring_val)) || (nrings > 0 && (!d_xy || !d_ring_off || !d_ring_t))) {
    wbk_set_error("%s: invalid argument", who);
    return WBK_ERR_INVALID;
  }
  if (nrings == 0 || ntime == 0) return WBK_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int rowcap = raster_rowcap(nlon);
  const size_t smem = (size_t)(RS_THREADS / 32) * 2 * rowcap * sizeof(int);
  if (smem > 200 * 1024) {
    wbk_set_error("%s: grid width %d too large for the row buffers", who, nlon);
    return WBK_ERR_CAPACITY;
  }
  const size_t ncell = (size_t)ntime * nlat * nlon;
  if (d_out_f64) {
    WBK_LAUNCH(KID_OWNER, owner_fill_kernel, dim3(592), dim3(256), 0, st, d_owner, ncell, -1);
    WBK_LAUNCH_CHECK();
  }
  auto kern = fm.p2 != 0 ? rings_raster_kernel<true> : rings_raster_kernel<false>;
  WBK_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int grid = nrings < 148 * 4 ? nrings : 148 * 4;
  WBK_LAUNCH(KID_RINGS_RASTER, kern, dim3(grid), dim3(RS_THREADS), smem, st, d_xy, d_ring_off, d_ring_t, nrings, nlat,
             nlon, ntime, r2, d_out_i8, d_out_f64 ? d_owner : (int*)nullptr, rowcap, fm);
  WBK_LAUNCH_CHECK();
  if (d_out_f64) {
    WBK_LAUNCH(KID_OWNER, owner_apply_kernel, dim3(592), dim3(256), 0, st, (const int*)d_owner, d_ring_val, d_out_f64, ncell);
    WBK_LAUNCH_CHECK();
  }
  return WBK_OK;
}

extern "C" int wbk_rasterize_rings(const int* d_xy, const int* d_ring_off, const int* d_ring_t,
                                   const double* d_ring_val, int nrings, int nlat, int nlon, int ntime, double r2,
                                   int8_t* d_out_i8, double* d_out_f64, int* d_owner, void* stream) {
  return rasterize_rings("wbk_rasterize_rings", d_xy, d_ring_off, d_ring_t, d_ring_val, nrings, nlat, nlon, ntime, r2,
                         FlagMetric{0, 0, 0, 0, 0}, d_out_i8, d_out_f64, d_owner, stream);
}

extern "C" int wbk_rasterize_rings_grid(const int* d_xy, const int* d_ring_off, const int* d_ring_t,
                                        const double* d_ring_val, int nrings, int nlat, int nlon, int ntime,
                                        double dlon, double dlat, int8_t* d_out_i8, double* d_out_f64, int* d_owner,
                                        void* stream) {
  FlagMetric fm;
  const int rc = grid_ratio("wbk_rasterize_rings_grid", dlon, dlat, &fm);
  if (rc != WBK_OK) return rc;
  // isotropic: r = (dlon + dlat) / 4 degrees is half a cell; otherwise the band reaches r / min(dlon, dlat) cells
  const double rcell = fm.p2 == 0 ? 0.5 : (dlon + dlat) / 4.0 / fmin(dlon, dlat);
  return rasterize_rings("wbk_rasterize_rings_grid", d_xy, d_ring_off, d_ring_t, d_ring_val, nrings, nlat, nlon, ntime,
                         rcell * rcell, fm, d_out_i8, d_out_f64, d_owner, stream);
}
