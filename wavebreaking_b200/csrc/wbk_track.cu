// Event tracking: exact polygon-overlap areas for the by_overlap method.
// Reference: wavebreaking/processing/events.py:205-214 (geopandas intersection(...).area of event pairs).
//
// area(A n B) is evaluated without clipping A against B: every polygon is the signed sum of the triangles
// (O, v_i, v_i+1) spanned by its edges and a common origin O, so
//     area(A n B) = sum_a sum_b sign_a sign_b area(T_a n T_b)
// and each triangle-triangle intersection is a tiny convex clip.  One CTA per event pair, threads over the
// (edge of A) x (edge of B) products, fp64, deterministic block reduction.
#include "wbk_common.cuh"

#define TRK_THREADS 256

struct TrkPoly {
  const double* xy;      // all vertices (x, y pairs)
  const int* ring_off;   // ring r = vertices [ring_off[r], ring_off[r+1])
  const int* poly_off;   // polygon p = rings [poly_off[p], poly_off[p+1])
};

// signed doubled area and CCW-ordered copy of triangle (o, a, b)
__device__ __forceinline__ double tri_ccw(double ox, double oy, double ax, double ay, double bx, double by, double* t) {
  const double c = (ax - ox) * (by - oy) - (ay - oy) * (bx - ox);
  t[0] = ox; t[1] = oy;
  if (c >= 0) { t[2] = ax; t[3] = ay; t[4] = bx; t[5] = by; }
  else        { t[2] = bx; t[3] = by; t[4] = ax; t[5] = ay; }
  return c;
}

// area of (convex CCW triangle p) n (convex CCW triangle q): Sutherland-Hodgman, at most 7 vertices
__device__ inline double tri_tri_area(const double* p, const double* q) {
  double poly[16], tmp[16];
  int n = 3;
  for (int i = 0; i < 6; ++i) poly[i] = q[i];
  for (int e = 0; e < 3 && n > 0; ++e) {
    const double ex0 = p[2 * e], ey0 = p[2 * e + 1];
    const double ex1 = p[2 * ((e + 1) % 3)], ey1 = p[2 * ((e + 1) % 3) + 1];
    const double dx = ex1 - ex0, dy = ey1 - ey0;
    int m = 0;
    for (int i = 0; i < n; ++i) {
      const double cx = poly[2 * i], cy = poly[2 * i + 1];
      const int j = i + 1 == n ? 0 : i + 1;
      const double nx = poly[2 * j], ny = poly[2 * j + 1];
      const double sc = dx * (cy - ey0) - dy * (cx - ex0);  // >= 0: inside (left of the edge)
      const double sn = dx * (ny - ey0) - dy * (nx - ex0);
      if (sc >= 0) {
        tmp[2 * m] = cx; tmp[2 * m + 1] = cy; ++m;
      }
      if ((sc > 0 && sn < 0) || (sc < 0 && sn > 0)) {
        const double t = sc / (sc - sn);
        tmp[2 * m] = cx + t * (nx - cx); tmp[2 * m + 1] = cy + t * (ny - cy); ++m;
      }
    }
    n = m;
    for (int i = 0; i < 2 * n; ++i) poly[i] = tmp[i];
  }
  if (n < 3) return 0.0;
  double a2 = 0.0;
  for (int i = 0; i < n; ++i) {
    const int j = i + 1 == n ? 0 : i + 1;
    a2 += poly[2 * i] * poly[2 * j + 1] - poly[2 * j] * poly[2 * i + 1];
  }
  return a2 > 0 ? 0.5 * a2 : 0.0;
}

// edge k (0-based over all rings of polygon p) -> its two end points
__device__ __forceinline__ void trk_edge(const TrkPoly& P, int p, int k, double& ax, double& ay, double& bx, double& by) {
  int r = P.poly_off[p];
  while (k >= P.ring_off[r + 1] - P.ring_off[r]) {
    k -= P.ring_off[r + 1] - P.ring_off[r];
    ++r;
  }
  const int s = P.ring_off[r], n = P.ring_off[r + 1] - s;
  const int k2 = k + 1 == n ? 0 : k + 1;
  ax = P.xy[2 * (s + k)]; ay = P.xy[2 * (s + k) + 1];
  bx = P.xy[2 * (s + k2)]; by = P.xy[2 * (s + k2) + 1];
}

__device__ __forceinline__ int trk_nedges(const TrkPoly& P, int p) {
  return P.ring_off[P.poly_off[p + 1]] - P.ring_off[P.poly_off[p]];
}

// out[3 * pair + {0,1,2}] = area(A), area(B), area(A n B)
__global__ void __launch_bounds__(TRK_THREADS) track_overlap_kernel(TrkPoly P, const int* __restrict__ pairs, int npairs,
                                                                    double* __restrict__ out) {
  __shared__ double red[40];
  for (int w = blockIdx.x; w < npairs; w += gridDim.x) {
    const int pa = pairs[2 * w], pb = pairs[2 * w + 1];
    const int na = trk_nedges(P, pa), nb = trk_nedges(P, pb);
    // common origin: first vertex of A (keeps the triangle areas small)
    const int sa = P.ring_off[P.poly_off[pa]];
    const double ox = na > 0 ? P.xy[2 * sa] : 0.0, oy = na > 0 ? P.xy[2 * sa + 1] : 0.0;
    double area_a = 0, area_b = 0, inter = 0;
    for (int k = threadIdx.x; k < na; k += TRK_THREADS) {
      double ax, ay, bx, by;
      trk_edge(P, pa, k, ax, ay, bx, by);
      area_a += (ax - ox) * (by - oy) - (ay - oy) * (bx - ox);
    }
    for (int k = threadIdx.x; k < nb; k += TRK_THREADS) {
      double ax, ay, bx, by;
      trk_edge(P, pb, k, ax, ay, bx, by);
      area_b += (ax - ox) * (by - oy) - (ay - oy) * (bx - ox);
    }
    const long long nprod = (long long)na * nb;
    for (long long q = threadIdx.x; q < nprod; q += TRK_THREADS) {
      const int ka = (int)(q / nb), kb = (int)(q - (long long)ka * nb);
      double a0x, a0y, a1x, a1y, b0x, b0y, b1x, b1y, ta[6], tb[6];
      trk_edge(P, pa, ka, a0x, a0y, a1x, a1y);
      trk_edge(P, pb, kb, b0x, b0y, b1x, b1y);
      const double ca = tri_ccw(ox, oy, a0x, a0y, a1x, a1y, ta);
      const double cb = tri_ccw(ox, oy, b0x, b0y, b1x, b1y, tb);
      if (ca == 0.0 || cb == 0.0) continue;
      // quick reject on bounding boxes
      const double axmin = fmin(ox, fmin(a0x, a1x)), axmax = fmax(ox, fmax(a0x, a1x));
      const double bxmin = fmin(ox, fmin(b0x, b1x)), bxmax = fmax(ox, fmax(b0x, b1x));
      const double aymin = fmin(oy, fmin(a0y, a1y)), aymax = fmax(oy, fmax(a0y, a1y));
      const double bymin = fmin(oy, fmin(b0y, b1y)), bymax = fmax(oy, fmax(b0y, b1y));
      if (axmax <= bxmin || bxmax <= axmin || aymax <= bymin || bymax <= aymin) continue;
      const double s = ((ca > 0) == (cb > 0)) ? 1.0 : -1.0;
      inter += s * tri_tri_area(ta, tb);
    }
    area_a = wbk_block_sum_f64(area_a, red);
    area_b = wbk_block_sum_f64(area_b, red);
    inter = wbk_block_sum_f64(inter, red);
    if (threadIdx.x == 0) {
      // orientation of the rings does not matter: |area|, and the product of winding signs for the overlap
      const double sgn = ((area_a > 0) == (area_b > 0)) ? 1.0 : -1.0;
      out[3 * w + 0] = fabs(0.5 * area_a);
      out[3 * w + 1] = fabs(0.5 * area_b);
      out[3 * w + 2] = sgn * inter;
    }
    __syncthreads();
  }
}

extern "C" int wbk_track_overlap(const double* d_xy, const int* d_ring_off, const int* d_poly_off, const int* d_pairs,
                                 int npairs, double* d_out, void* stream) {
  if (npairs < 0 || (npairs > 0 && (!d_xy || !d_ring_off || !d_poly_off || !d_pairs || !d_out))) {
    wbk_set_error("wbk_track_overlap: invalid argument");
    return WBK_ERR_INVALID;
  }
  if (npairs == 0) return WBK_OK;
  TrkPoly P{d_xy, d_ring_off, d_poly_off};
  const int grid = npairs < 148 * 8 ? npairs : 148 * 8;
  WBK_LAUNCH(KID_TRACK_OVERLAP, track_overlap_kernel, dim3(grid), dim3(TRK_THREADS), 0, (cudaStream_t)stream, P, d_pairs,
             npairs, d_out);
  WBK_LAUNCH_CHECK();
  return WBK_OK;
}

// ------------------------------------------------------------------------------------------------------------
// Candidate pairs (events.py:160-181).  The events are sorted by date; for event i the host supplies the index window
// [lo[i], hi[i]) of the events j with 0 < date_j - date_i <= time_range (two vectorised searches).  One warp per
// event expands its window, drops the pairs whose bounding boxes are disjoint (their intersection is empty, so
// `inter.area / union.area` is 0) and appends the rest with one warp-aggregated atomic per 32 candidates.
// d_bbox may be NULL (by_distance: every pair of the window is a candidate).
__global__ void __launch_bounds__(256) track_candidates_kernel(const int* __restrict__ lo, const int* __restrict__ hi,
                                                               const int* __restrict__ bbox, int n, int* __restrict__ pairs,
                                                               int cap, int* __restrict__ count) {
  const int lane = wbk_lane();
  const int wpb = blockDim.x >> 5;
  for (int i = blockIdx.x * wpb + wbk_warp(); i < n; i += gridDim.x * wpb) {
    const int a = lo[i], b = hi[i];
    int bx0 = 0, by0 = 0, bx1 = 0, by1 = 0;
    if (bbox) {
      bx0 = bbox[4 * i]; by0 = bbox[4 * i + 1]; bx1 = bbox[4 * i + 2]; by1 = bbox[4 * i + 3];
    }
    for (int j0 = a; j0 < b; j0 += 32) {
      const int j = j0 + lane;
      bool keep = j < b;
      if (keep && bbox) {
        const int cx0 = bbox[4 * j], cy0 = bbox[4 * j + 1], cx1 = bbox[4 * j + 2], cy1 = bbox[4 * j + 3];
        keep = !(bx1 < cx0 || cx1 < bx0 || by1 < cy0 || cy1 < by0) && bx0 <= bx1 && cx0 <= cx1;  // empty boxes never match
      }
      const u32 m = __ballot_sync(WBK_FULL, keep);
      if (m == 0) continue;
      int base = 0;
      if (lane == 0) base = atomicAdd(count, __popc(m));
      base = __shfl_sync(WBK_FULL, base, 0);
      if (keep) {
        const int slot = base + __popc(m & ((1u << lane) - 1u));
        if (slot < cap) {
          pairs[2 * slot] = i;
          pairs[2 * slot + 1] = j;
        }
      }
    }
  }
}

extern "C" int wbk_track_candidates(const int* d_lo, const int* d_hi, const int* d_bbox, int n, int* d_pairs, int cap,
                                    int* d_count, void* stream) {
  if (n < 0 || cap < 0 || !d_count || (n > 0 && (!d_lo || !d_hi)) || (cap > 0 && !d_pairs)) {
    wbk_set_error("wbk_track_candidates: invalid argument");
    return WBK_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  WBK_CUDA_CHECK(cudaMemsetAsync(d_count, 0, sizeof(int), st));
  if (n == 0) return WBK_OK;
  const int blocks = (n + 7) / 8 < 148 * 8 ? (n + 7) / 8 : 148 * 8;
  WBK_LAUNCH(KID_TRACK_PAIRS, track_candidates_kernel, dim3(blocks), dim3(256), 0, st, d_lo, d_hi, d_bbox, n, d_pairs, cap,
             d_count);
  WBK_LAUNCH_CHECK();
  return WBK_OK;
}

// ------------------------------------------------------------------------------------------------------------
// Exact "do the two lattice polygons overlap in a region of positive area?" (events.py:205-214 with overlap = 0:
// `inter.area / union.area > 0`; GEOS returns an empty / lower-dimensional intersection, area 0.0, for polygons
// that merely touch).  All vertices are integers below 2^12, so every predicate is exact in int64:
//   1. a proper (transversal, interior-interior) crossing of an edge of A with an edge of B  => overlap;
//   2. no edge of A meets an edge of B at all  => the boundaries are disjoint: overlap iff the first vertex of a ring
//      of one polygon lies inside the other (non-zero winding);
//   3. the boundaries touch but never cross properly: the touch points cut each boundary into arcs that lie
//      entirely inside, outside or on the other boundary.  Every edge that takes part in a touch is cut at the other
//      polygon's vertices on it; the midpoint of each piece is classified exactly (coordinates scaled by twice the
//      squared edge length): strictly inside => overlap; on the other boundary (collinear pieces) => overlap iff
//      both interiors lie on the same side of the shared piece (ring orientation signs).  Rings without a touched
//      edge are covered by rule 2.
// Polygon p = vertices [poly_voff[p], poly_voff[p+1]) of the edge table (x0, y0, x1, y1 per vertex: the edge from
// that vertex to the next one of its ring); vsign = orientation of the vertex's ring (+1 counter-clockwise).
// result: 0 / 1, | 2 when rule 3 decided.
#define TRX_THREADS 128
#define TRX_MAXTOUCH 96

__device__ __forceinline__ long long trx_cross(long long ax, long long ay, long long bx, long long by) { return ax * by - ay * bx; }

// winding number contribution of edge (x0,y0)->(x1,y1) for the point (px,py), all in the same (scaled) units;
// *on is set when the point lies on the closed edge
__device__ __forceinline__ int trx_wind(long long x0, long long y0, long long x1, long long y1, long long px, long long py, bool* on) {
  const long long cr = trx_cross(x1 - x0, y1 - y0, px - x0, py - y0);
  if (cr == 0 && px >= min(x0, x1) && px <= max(x0, x1) && py >= min(y0, y1) && py <= max(y0, y1)) *on = true;
  if (y0 <= py && py < y1) return cr > 0 ? 1 : 0;
  if (y1 <= py && py < y0) return cr < 0 ? -1 : 0;
  return 0;
}

__global__ void __launch_bounds__(TRX_THREADS) track_exact_kernel(const int4* __restrict__ edges, const int* __restrict__ vsign,
                                                                  const int* __restrict__ ring_off, const int* __restrict__ poly_off,
                                                                  const int* __restrict__ pairs, int npairs, int* __restrict__ result) {
  __shared__ int s_flag[4];                 // [0] proper crossing, [1] any touch, [2] touch list overflow
  __shared__ int s_ntouch[2];
  __shared__ int s_touch[2][TRX_MAXTOUCH];  // touched edges of A / of B (vertex indices; duplicates allowed)
  __shared__ int s_w, s_on;
  __shared__ long long s_next;
  const int tid = threadIdx.x;
  for (int w = blockIdx.x; w < npairs; w += gridDim.x) {
    const int pa = pairs[2 * w], pb = pairs[2 * w + 1];
    const int a0 = ring_off[poly_off[pa]], a1 = ring_off[poly_off[pa + 1]];
    const int b0 = ring_off[poly_off[pb]], b1 = ring_off[poly_off[pb + 1]];
    const int nA = a1 - a0, nB = b1 - b0;
    if (tid < 4) s_flag[tid] = 0;
    if (tid < 2) s_ntouch[tid] = 0;
    __syncthreads();
    // ---- rule 1: all edge pairs (thread: one edge of A against every edge of B, uniform broadcast reads)
    for (int at = 0; at < nA; at += TRX_THREADS) {
      const int ia = at + tid;
      if (ia < nA) {
        const int4 e = edges[a0 + ia];
        const int exmin = min(e.x, e.z), exmax = max(e.x, e.z), eymin = min(e.y, e.w), eymax = max(e.y, e.w);
        bool proper = false, touched = false;
        for (int ib = 0; ib < nB; ++ib) {
          const int4 f = edges[b0 + ib];
          if (exmax < min(f.x, f.z) || max(f.x, f.z) < exmin || eymax < min(f.y, f.w) || max(f.y, f.w) < eymin) continue;
          const long long d1 = trx_cross(f.z - f.x, f.w - f.y, e.x - f.x, e.y - f.y);
          const long long d2 = trx_cross(f.z - f.x, f.w - f.y, e.z - f.x, e.w - f.y);
          const long long d3 = trx_cross(e.z - e.x, e.w - e.y, f.x - e.x, f.y - e.y);
          const long long d4 = trx_cross(e.z - e.x, e.w - e.y, f.z - e.x, f.w - e.y);
          if (((d1 > 0 && d2 < 0) || (d1 < 0 && d2 > 0)) && ((d3 > 0 && d4 < 0) || (d3 < 0 && d4 > 0))) {
            proper = true;
            break;
          }
          const bool meet = !((d1 > 0 && d2 > 0) || (d1 < 0 && d2 < 0) || (d3 > 0 && d4 > 0) || (d3 < 0 && d4 < 0));
          if (meet) {  // closed segments share a point (collinear ones: their boxes intersect, checked above)
            touched = true;
            const int k = atomicAdd(&s_ntouch[1], 1);
            if (k < TRX_MAXTOUCH) s_touch[1][k] = b0 + ib;
            else s_flag[2] = 1;
          }
        }
        if (proper) s_flag[0] = 1;
        if (touched) {
          s_flag[1] = 1;
          const int k = atomicAdd(&s_ntouch[0], 1);
          if (k < TRX_MAXTOUCH) s_touch[0][k] = a0 + ia;
          else s_flag[2] = 1;
        }
      }
      __syncthreads();
      if (s_flag[0]) break;  // block-uniform
    }
    int res = s_flag[0] ? 1 : 0;
    const bool touch = s_flag[1] != 0, overflow = s_flag[2] != 0;
    __syncthreads();
    if (!res && nA > 0 && nB > 0) {
      // ---- rule 2: first vertex of every ring against the other polygon (skipped when it lies on the boundary)
      for (int side = 0; side < 2 && !res; ++side) {
        const int pr0 = side == 0 ? poly_off[pa] : poly_off[pb], pr1 = side == 0 ? poly_off[pa + 1] : poly_off[pb + 1];
        const int o0 = side == 0 ? b0 : a0, o1 = side == 0 ? b1 : a1;
        for (int r = pr0; r < pr1 && !res; ++r) {
          if (ring_off[r + 1] == ring_off[r]) continue;
          const int4 v = edges[ring_off[r]];
          if (tid == 0) { s_w = 0; s_on = 0; }
          __syncthreads();
          int wsum = 0;
          bool on = false;
          for (int i = o0 + tid; i < o1; i += TRX_THREADS) {
            const int4 f = edges[i];
            wsum += trx_wind(f.x, f.y, f.z, f.w, v.x, v.y, &on);
          }
          if (wsum) atomicAdd(&s_w, wsum);
          if (on) s_on = 1;
          __syncthreads();
          if (!s_on && s_w != 0) res = 1;  // block-uniform
          __syncthreads();
        }
      }
    }
    if (!res && touch) {
      // ---- rule 3: the pieces of the touched edges (all edges when the touch lists overflowed)
      res |= 2;
      for (int side = 0; side < 2 && !(res & 1); ++side) {
        const int s0 = side == 0 ? a0 : b0, s1 = side == 0 ? a1 : b1;  // subject polygon
        const int o0 = side == 0 ? b0 : a0, o1 = side == 0 ? b1 : a1;  // the other one
        const int nlist = overflow ? s1 - s0 : min(s_ntouch[side], TRX_MAXTOUCH);
        for (int li = 0; li < nlist && !(res & 1); ++li) {
          const int ei = overflow ? s0 + li : s_touch[side][li];
          const int4 e = edges[ei];
          const long long dx = e.z - e.x, dy = e.w - e.y;
          const long long L2 = dx * dx + dy * dy, S = 2 * L2;
          if (L2 == 0) continue;
          long long s = 0;
          while (s < L2 && !(res & 1)) {  // block-uniform loop
            if (tid == 0) { s_next = L2; s_w = 0; s_on = -1; }
            __syncthreads();
            // next cut: the smallest parameter > s of a vertex of the other polygon on the open edge
            long long best = L2;
            for (int i = o0 + tid; i < o1; i += TRX_THREADS) {
              const int4 f = edges[i];
              if (trx_cross(dx, dy, f.x - e.x, f.y - e.y) == 0) {
                const long long tv = (f.x - e.x) * dx + (f.y - e.y) * dy;
                if (tv > s && tv < best) best = tv;
              }
            }
            if (best < L2) atomicMin((unsigned long long*)&s_next, (unsigned long long)best);
            __syncthreads();
            const long long nxt = s_next;
            // midpoint of the piece (s, nxt), scaled by S = 2 L2
            const long long mx = (long long)e.x * S + dx * (s + nxt), my = (long long)e.y * S + dy * (s + nxt);
            int wsum = 0;
            for (int i = o0 + tid; i < o1; i += TRX_THREADS) {
              const int4 f = edges[i];
              bool on = false;
              wsum += trx_wind((long long)f.x * S, (long long)f.y * S, (long long)f.z * S, (long long)f.w * S, mx, my, &on);
              if (on) atomicMax(&s_on, i);
            }
            if (wsum) atomicAdd(&s_w, wsum);
            __syncthreads();
            if (s_on >= 0) {
              if (side == 0) {  // shared boundary piece: same side?
                const int4 f = edges[s_on];
                const long long dot = dx * (f.z - f.x) + dy * (f.w - f.y);
                const int sa = vsign[ei], sb = vsign[s_on] * (dot > 0 ? 1 : (dot < 0 ? -1 : 0));
                if (sa != 0 && sa == sb) res |= 1;
              }
            } else if (s_w != 0) {
              res |= 1;
            }
            __syncthreads();
            s = nxt;
          }
        }
      }
    }
    if (tid == 0) result[w] = res;
    __syncthreads();
  }
}

extern "C" int wbk_track_overlap_exact(const int* d_edges, const int* d_vsign, const int* d_ring_off, const int* d_poly_off,
                                       const int* d_pairs, int npairs, int* d_result, void* stream) {
  if (npairs < 0 || (npairs > 0 && (!d_edges || !d_vsign || !d_ring_off || !d_poly_off || !d_pairs || !d_result))) {
    wbk_set_error("wbk_track_overlap_exact: invalid argument");
    return WBK_ERR_INVALID;
  }
  if (npairs == 0) return WBK_OK;
  const int grid = npairs < 148 * 16 ? npairs : 148 * 16;
  WBK_LAUNCH(KID_TRACK_EXACT, track_exact_kernel, dim3(grid), dim3(TRX_THREADS), 0, (cudaStream_t)stream,
             (const int4*)d_edges, d_vsign, d_ring_off, d_poly_off, d_pairs, npairs, d_result);
  WBK_LAUNCH_CHECK();
  return WBK_OK;
}

// ------------------------------------------------------------------------------------------------------------
// by_distance (events.py:187-201): sklearn's haversine of the two centres of mass of every pair, evaluated in the
// operand order of sklearn/metrics/_dist_metrics.pyx.tp:2641-2656 (x1 = first event, x2 = second).  CUDA's sin /
// asin differ from glibc's by <= 2 ulp, so the caller re-evaluates with libm the pairs whose distance lies within
// 1e-9 (relative) of the threshold.  d_rad: [n][2] radians exactly as the reference feeds them.
__global__ void track_distance_kernel(const double* __restrict__ rad, const int* __restrict__ pairs, int npairs,
                                      double* __restrict__ out) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < npairs; k += gridDim.x * blockDim.x) {
    const int a = pairs[2 * k], b = pairs[2 * k + 1];
    const double a0 = rad[2 * a], a1 = rad[2 * a + 1], b0 = rad[2 * b], b1 = rad[2 * b + 1];
    const double s0 = sin(__dmul_rn(0.5, __dsub_rn(a0, b0))), s1 = sin(__dmul_rn(0.5, __dsub_rn(a1, b1)));
    const double h = __dadd_rn(__dmul_rn(s0, s0), __dmul_rn(__dmul_rn(__dmul_rn(cos(a0), cos(b0)), s1), s1));
    out[k] = __dmul_rn(2.0, asin(sqrt(h)));
  }
}

extern "C" int wbk_track_distance(const double* d_rad, const int* d_pairs, int npairs, double* d_out, void* stream) {
  if (npairs < 0 || (npairs > 0 && (!d_rad || !d_pairs || !d_out))) {
    wbk_set_error("wbk_track_distance: invalid argument");
    return WBK_ERR_INVALID;
  }
  if (npairs == 0) return WBK_OK;
  const int grid = (npairs + 255) / 256 < 148 * 8 ? (npairs + 255) / 256 : 148 * 8;
  WBK_LAUNCH(KID_TRACK_DIST, track_distance_kernel, dim3(grid), dim3(256), 0, (cudaStream_t)stream, d_rad, d_pairs, npairs,
             d_out);
  WBK_LAUNCH_CHECK();
  return WBK_OK;
}

// ------------------------------------------------------------------------------------------------------------
// Tracking polygons of one kind of one collected batch, appended to a device window in the layout that
// wbk_track_candidates / wbk_track_overlap_exact read (utils/index_utils.py:129-184 transform_polygons, as
// pipeline.events_soup builds it on the host): x folded with x % nlon, an event with split == 1 replaced by its
// device-clipper pieces (in piece order), an overturning = its box (x1, y0), (x1, y1), (x0, y1), (x0, y0).
// count -> exclusive scan (one CTA) -> fill (one warp per event).
#define TAP_THREADS 1024
#define TAP_SPLIT_COL 8
#define TAP_BOX_COL 3

struct TapIn {
  const int* ev_int;       // [rows][WBK_EV_INTS] of the batch (kind-major gather)
  const int* ring_off;     // [rows + 1] ring vertices of every row in ring_pts
  const u32* ring_pts;     // packed lattice points (x low 16 bits, y high 16 bits)
  const int* sp_ev;        // [npieces] row of every piece
  const int* sp_off;       // [npieces + 1]
  const int* sp_xy;        // [..][2] folded piece vertices
  int npieces, first, n, is_box, nlon;
};

struct TapOut {
  int4* edges;
  int* vsign;
  int* ring_off;
  int* poly_off;
  int4* bbox;
  int v0, r0, p0;          // where this batch starts in the window
  int cap_v, cap_r, cap_p;  // window capacities (writes beyond them are dropped)
};

__device__ __forceinline__ int2 tap_i2(int x, int y) {
  int2 r;
  r.x = x; r.y = y;
  return r;
}
__device__ __forceinline__ int4 tap_i4(int x, int y, int z, int w) {
  int4 r;
  r.x = x; r.y = y; r.z = z; r.w = w;
  return r;
}

__device__ __forceinline__ bool tap_split(const TapIn& in, int e) {
  return in.ev_int[(size_t)(in.first + e) * WBK_EV_INTS + TAP_SPLIT_COL] == 1;
}

// one warp: the k-th piece (in piece order) of row `row`, for k = 0, 1, ...: f(k, piece)
template <typename F>
__device__ __forceinline__ void tap_pieces(const TapIn& in, int row, F f) {
  const int lane = wbk_lane();
  int k = 0;
  for (int b = 0; b < in.npieces; b += 32) {
    const int r = b + lane;
    u32 m = __ballot_sync(WBK_FULL, r < in.npieces && in.sp_ev[r] == row);
    while (m) {
      const int bit = __ffs(m) - 1;
      m &= m - 1;
      f(k++, b + bit);
    }
  }
}

__global__ void __launch_bounds__(TAP_THREADS) track_append_scan_kernel(TapIn in, TapOut out) {
  __shared__ int sscan[40];
  const int lane = wbk_lane(), nw = blockDim.x >> 5;
  int* nr = out.poly_off + out.p0;  // rings per event, scanned in place into the polygon offsets
  for (int e = wbk_warp(); e < in.n; e += nw) {
    int cnt = 1;
    if (tap_split(in, e)) {
      cnt = 0;
      tap_pieces(in, in.first + e, [&](int, int) { ++cnt; });
    }
    if (lane == 0) nr[e] = cnt;
  }
  __syncthreads();
  const int nrings = wbk_block_excl_scan(nr, in.n, sscan);
  if ((long long)out.r0 + nrings + 1 > out.cap_r) return;  // (the caller sized the window from the same tables)
  for (int e = threadIdx.x; e < in.n; e += blockDim.x) nr[e] += out.r0;
  if (threadIdx.x == 0) nr[in.n] = out.r0 + nrings;
  __syncthreads();
  int* nv = out.ring_off + out.r0;  // vertices per ring, scanned in place into the ring offsets
  for (int e = wbk_warp(); e < in.n; e += nw) {
    const int R = nr[e] - out.r0;
    if (tap_split(in, e)) {
      tap_pieces(in, in.first + e, [&](int k, int r) {
        if (lane == 0) nv[R + k] = in.sp_off[r + 1] - in.sp_off[r];
      });
    } else if (lane == 0) {
      nv[R] = in.is_box ? 4 : in.ring_off[in.first + e + 1] - in.ring_off[in.first + e];
    }
  }
  __syncthreads();
  const int nverts = wbk_block_excl_scan(nv, nrings, sscan);
  for (int r = threadIdx.x; r < nrings; r += blockDim.x) nv[r] += out.v0;
  if (threadIdx.x == 0) nv[nrings] = out.v0 + nverts;
}

// one warp writes the edges of ring [s, s + len) of the window and its orientation sign; vertex k = xy(k)
template <typename XY>
__device__ __forceinline__ void tap_ring(const TapOut& out, int s, int len, XY xy, int4& box) {
  const int lane = wbk_lane();
  long long a2 = 0;
  for (int k = lane; k < len; k += 32) {
    const int2 p = xy(k), q = xy(k + 1 == len ? 0 : k + 1);
    if (s + k < out.cap_v) out.edges[s + k] = tap_i4(p.x, p.y, q.x, q.y);
    a2 += (long long)p.x * q.y - (long long)q.x * p.y;
    box.x = min(box.x, p.x); box.y = min(box.y, p.y); box.z = max(box.z, p.x); box.w = max(box.w, p.y);
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) a2 += __shfl_xor_sync(WBK_FULL, a2, d);
  const int sg = a2 > 0 ? 1 : (a2 < 0 ? -1 : 0);
  for (int k = lane; k < len && s + k < out.cap_v; k += 32) out.vsign[s + k] = sg;
}

__global__ void __launch_bounds__(256) track_append_fill_kernel(TapIn in, TapOut out) {
  const int lane = wbk_lane(), wpb = blockDim.x >> 5;
  for (int e = blockIdx.x * wpb + wbk_warp(); e < in.n; e += gridDim.x * wpb) {
    const int row = in.first + e, nlon = in.nlon;
    int4 box = tap_i4(0x7fffffff, 0x7fffffff, -0x7fffffff - 1, -0x7fffffff - 1);
    const int R = out.poly_off[out.p0 + e];
    if (tap_split(in, e)) {
      tap_pieces(in, row, [&](int k, int r) {
        const int a = in.sp_off[r];
        const int2* pxy = reinterpret_cast<const int2*>(in.sp_xy);
        tap_ring(out, out.ring_off[R + k], in.sp_off[r + 1] - a, [&](int i) { return pxy[a + i]; }, box);
      });
    } else if (in.is_box) {
      const int* b = in.ev_int + (size_t)row * WBK_EV_INTS + TAP_BOX_COL;
      const int x0 = ((b[0] % nlon) + nlon) % nlon, y0 = b[1], x1 = ((b[2] % nlon) + nlon) % nlon, y1 = b[3];
      tap_ring(out, out.ring_off[R], 4, [&](int i) {
        return i == 0 ? tap_i2(x1, y0) : i == 1 ? tap_i2(x1, y1) : i == 2 ? tap_i2(x0, y1) : tap_i2(x0, y0);
      }, box);
    } else {
      const int a = in.ring_off[row];
      tap_ring(out, out.ring_off[R], in.ring_off[row + 1] - a, [&](int i) {
        const u32 p = in.ring_pts[a + i];
        return tap_i2((int)(p & 0xffffu) % nlon, (int)(p >> 16));
      }, box);
    }
    box.x = wbk_warp_min(box.x); box.y = wbk_warp_min(box.y);
    box.z = wbk_warp_max(box.z); box.w = wbk_warp_max(box.w);
    if (box.x > box.z) box = tap_i4(1, 1, 0, 0);  // no vertex: an empty box (PolygonSoup.bounds)
    if (lane == 0 && out.p0 + e < out.cap_p) out.bbox[out.p0 + e] = box;
  }
}

extern "C" int wbk_track_append(const int* d_ev_int, const int* d_ring_off, const uint32_t* d_ring_pts, const int* d_sp_ev,
                                const int* d_sp_off, const int* d_sp_xy, int npieces, int first, int n, int is_box,
                                int nlon, long long nrings, long long nverts, int* d_edges, int* d_vsign,
                                int* d_win_ring_off, int* d_win_poly_off, int* d_bbox, long long v0, long long r0,
                                long long p0, long long cap_v, long long cap_r, long long cap_p, void* stream) {
  const long long lim = 2147483647LL;
  if (n < 0 || first < 0 || npieces < 0 || nlon < 1 || nrings < 0 || nverts < 0 || v0 < 0 || r0 < 0 || p0 < 0) {
    wbk_set_error("wbk_track_append: invalid argument (n %d, first %d, npieces %d, nlon %d)", n, first, npieces, nlon);
    return WBK_ERR_INVALID;
  }
  if (v0 + nverts > lim || r0 + nrings + 1 > lim || p0 + n + 1 > lim) {
    wbk_set_error("wbk_track_append: the window would hold %lld vertices, %lld rings and %lld polygons; its 32-bit "
                  "offsets allow at most 2^31 - 1", v0 + nverts, r0 + nrings, p0 + n);
    return WBK_ERR_INVALID;
  }
  if (v0 + nverts > cap_v || r0 + nrings + 1 > cap_r || p0 + n + 1 > cap_p) {
    wbk_set_error("wbk_track_append: the window is too small (%lld / %lld vertices, %lld / %lld ring offsets, "
                  "%lld / %lld polygon offsets)", v0 + nverts, cap_v, r0 + nrings + 1, cap_r, p0 + n + 1, cap_p);
    return WBK_ERR_INVALID;
  }
  if (n == 0) return WBK_OK;
  if (!d_ev_int || (!is_box && (!d_ring_off || !d_ring_pts)) || (npieces > 0 && (!d_sp_ev || !d_sp_off || !d_sp_xy)) ||
      !d_edges || !d_vsign || !d_win_ring_off || !d_win_poly_off || !d_bbox) {
    wbk_set_error("wbk_track_append: invalid argument (null pointer)");
    return WBK_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const TapIn in{d_ev_int, d_ring_off, d_ring_pts, d_sp_ev, d_sp_off, d_sp_xy, npieces, first, n, is_box, nlon};
  const TapOut out{(int4*)d_edges, d_vsign, d_win_ring_off, d_win_poly_off, (int4*)d_bbox, (int)v0, (int)r0, (int)p0,
                   (int)(cap_v < lim ? cap_v : lim), (int)(cap_r < lim ? cap_r : lim), (int)(cap_p < lim ? cap_p : lim)};
  WBK_LAUNCH(KID_TRACK_APPEND, track_append_scan_kernel, dim3(1), dim3(TAP_THREADS), 0, st, in, out);
  WBK_LAUNCH_CHECK();
  const int blocks = (n + 7) / 8 < 148 * 8 ? (n + 7) / 8 : 148 * 8;
  WBK_LAUNCH(KID_TRACK_APPEND, track_append_fill_kernel, dim3(blocks), dim3(256), 0, st, in, out);
  WBK_LAUNCH_CHECK();
  return WBK_OK;
}
