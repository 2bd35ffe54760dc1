// Streamer / overturning / cutoff indices on a packed, device-resident contour set.
// Reference: wavebreaking/indices/streamer_index.py:100-275, overturning_index.py:99-215,
// cutoff_index.py:83-98.
#include "wbk_ctx.cuh"

// ------------------------------------------------------------------------------------------ arenas
#define PT_HOST 32   // == PT, the pair-scan tile edge
size_t wbk_index_layout(struct wbk_ctx* ctx, unsigned char* base, size_t off) {
  WbkIdx& x = ctx->x;
  const wbk_caps& c = ctx->caps;
  x.PC = (int)wbk_pow2_ceil((u32)c.pair_cap);
  x.EC = c.event_cap;
  x.SC = c.sel_cap;
  const size_t J = c.max_jobs, PC = x.PC, EC = x.EC, SC = x.SC;
  size_t o = off;
  auto take = [&](size_t bytes) -> unsigned char* {
    o = (o + 255) & ~(size_t)255;
    unsigned char* p = base ? base + o : nullptr;
    o += bytes;
    return p;
  };
  x.sel = (int*)take(J * SC * 4);
  x.nsel = (int*)take(J * 4);
  x.pairs = (u64*)take(J * SC * PC * 8);
  x.pair_count = (int*)take(J * SC * 4);
  x.tile_off = (int*)take((J * SC + 1) * 4);
  x.pairs_b = (u64*)take(J * PC * 8);
  x.flag = (int*)take(J * SC * PC * 4);
  x.scanb = (int*)take(J * PC * 4);
  x.label = (int*)take(J * PC * 4);
  x.hk = (u64*)take(J * SC * 2 * PC * 8);
  x.hv1 = (u32*)take(J * 2 * PC * 4);
  x.hv2 = (u32*)take(J * 2 * PC * 4);
  x.TLC = (int)(J * SC * 256 > (size_t)1 << 24 ? (size_t)1 << 24 : J * SC * 256);
  if ((size_t)x.TLC < J * (PC / 16)) x.TLC = (int)(J * (PC / 16));
  x.tile_list = (u64*)take((size_t)x.TLC * 8);
  x.hm1 = (u64*)take(J * SC * 2 * PC * 8);
  x.hm2 = (u64*)take(J * SC * 2 * PC * 8);
  x.pairs2 = (u64*)take(J * SC * PC * 8);
  x.cnt1 = (int*)take(J * SC * 4);
  x.touch_off = (int*)take((J * SC + 1) * 4);
  x.ev_int = (int*)take(3 * J * EC * WBK_EV_INTS * 4);
  x.ev_f64 = (double*)take(3 * J * EC * WBK_EV_F64 * 8);
  x.ev_count = (int*)take(3 * J * 4);
  x.ev_off = (int*)take((3 * J + 1) * 4);
  x.total = (int*)take(64);
  x.NB = (c.seg_cap + c.contour_cap + PT_HOST - 1) / PT_HOST;
  x.blk_x = (int*)take(J * SC * (size_t)x.NB * 4 * 4);
  x.blk_pf = (double*)take(J * SC * (size_t)x.NB * 2 * 8);
  // meridian-split arenas grow with event_cap: their overflow is reported as WBK_ST_EVENT_OVERFLOW (wbk_raster.cu)
  const size_t spv_job = EC * 32 > 4096 ? EC * 32 : 4096, spr_job = EC / 2 > 32 ? EC / 2 : 32;
  x.SPV = (int)(J * spv_job < (size_t)1 << 26 ? J * spv_job : (size_t)1 << 26);
  x.SPR = (int)(J * spr_job < (size_t)1 << 24 ? J * spr_job : (size_t)1 << 24);
  x.split_xy = (int*)take((size_t)x.SPV * 2 * 4);
  x.split_ring = (int*)take((size_t)x.SPR * 4 * 4);
  x.split_count = (int*)take(64);
  x.split_list = (int*)take((size_t)x.SPR * 4);
  x.NRC = WBK_NEAR_CAP;
  x.near_rec = (int*)take((size_t)x.NRC * 4 * sizeof(int));
  x.near_cnt = (int*)take(64);
  return (o + 255) & ~(size_t)255;
}

struct PackedSet {
  const int* job_off;
  const int* pt_off;
  const int* meta;
  const u32* pts;
  int njobs, nlevels, ncontours, npoints;
};

struct CoordTabs {
  const double *lat_deg, *lat_rad, *cos_lat, *area, *lon_rad;
};

__host__ __device__ inline CoordTabs make_coords(const double* c, int nlat) {
  CoordTabs t;
  t.lat_deg = c;
  t.lat_rad = c + nlat;
  t.cos_lat = c + 2 * nlat;
  t.area = c + 3 * nlat;
  t.lon_rad = c + 4 * nlat;
  return t;
}

__device__ __forceinline__ int* ev_int_ptr(const WbkIdx& x, int J, int kind, int job, int e) {
  return x.ev_int + (((size_t)kind * J + job) * x.EC + e) * WBK_EV_INTS;
}

// ------------------------------------------------------------------------------------------ selection + cutoffs
// One warp per job: ordered compaction of the full-width contours (exp_lon == max) and of the cutoffs
// (closed, exp_lon < max, exp_lon >= min_exp: cutoff_index.py:89-93).
__global__ void select_kernel(WbkDev d, WbkIdx x, PackedSet ps, wbk_index_params prm, int J) {
  const int job = blockIdx.x * (blockDim.x >> 5) + wbk_warp();
  if (job >= ps.njobs) return;
  const int lane = wbk_lane();
  const int c0 = ps.job_off[job], c1 = ps.job_off[job + 1];
  const int gmax = prm.gmax_nx >= 0 ? prm.gmax_nx : *d.max_nx;  // < 0: the batch maximum found by wbk_contours
  int nsel = 0, ncut = 0;
  for (int cb = c0; cb < c1; cb += 32) {
    const int c = cb + lane;
    int is_sel = 0, is_cut = 0, npts = 0;
    if (c < c1) {
      const int closed = ps.meta[4 * c + 0], nx = ps.meta[4 * c + 1];
      npts = ps.pt_off[c + 1] - ps.pt_off[c];
      is_sel = nx == gmax;
      is_cut = prm.do_cutoffs && closed && nx < gmax && ((double)nx * prm.dlon >= prm.co_min_exp);
    }
    const u32 bs = __ballot_sync(WBK_FULL, is_sel), bc = __ballot_sync(WBK_FULL, is_cut);
    const u32 below = (1u << lane) - 1u;
    if (is_sel) {
      int k = nsel + __popc(bs & below);
      if (k < x.SC) x.sel[(size_t)job * x.SC + k] = c;
    }
    if (is_cut) {
      int k = ncut + __popc(bc & below);
      if (k < x.EC) {
        int* ev = ev_int_ptr(x, J, WBK_EV_CUTOFF, job, k);
        ev[0] = c; ev[1] = 0; ev[2] = npts - 1;
        for (int q = 3; q < WBK_EV_INTS; ++q) ev[q] = 0;
      }
    }
    nsel += __popc(bs);
    ncut += __popc(bc);
  }
  if (lane == 0) {
    if (nsel > x.SC) {
      atomicOr(&d.status[job], (int)WBK_ST_SEL_OVERFLOW);
      nsel = x.SC;
    }
    if (ncut > x.EC) {
      atomicOr(&d.status[job], (int)WBK_ST_EVENT_OVERFLOW);
      ncut = x.EC;
    }
    x.nsel[job] = nsel;
    x.ev_count[WBK_EV_CUTOFF * J + job] = ncut;
    x.ev_count[WBK_EV_STREAMER * J + job] = 0;
    x.ev_count[WBK_EV_OVERTURNING * J + job] = 0;
    for (int s = 0; s < x.SC; ++s) x.pair_count[(size_t)job * x.SC + s] = 0;
  }
}

// ------------------------------------------------------------------------------------------ overturnings
#define OT_THREADS 256
#define OT_GMAX 512

__device__ __forceinline__ bool arc_subset(int min_i, int max_i, int min_j, int max_j, int nlon) {
  // set(range(min_i, max_i + 1) % nlon) subset of set(range(min_j, max_j + 1) % nlon)
  const int li = max_i - min_i + 1, lj = max_j - min_j + 1;
  if (lj >= nlon) return true;
  if (li >= nlon) return false;
  int a = min_i % nlon, b = min_j % nlon;
  int off = a - b;
  if (off < 0) off += nlon;
  return off + li <= lj;
}

__global__ void __launch_bounds__(OT_THREADS) overturning_kernel(WbkDev d, WbkIdx x, PackedSet ps, CoordTabs ct,
                                                                 wbk_index_params prm, int J) {
  const int job = blockIdx.x;
  if (job >= ps.njobs) return;
  WBK_DYN_SMEM(int, sm);
  const int W = d.W, tid = threadIdx.x, nt = blockDim.x;
  int* cnt = sm;            // [W] crossings per column
  int* ymin = sm + W;       // [W]
  int* ymax = sm + 2 * W;   // [W]
  int* first = sm + 3 * W;  // [W] first contour position with this column
  int* last = sm + 4 * W;   // [W] last contour position with this column
  int* tmp = sm + 5 * W;    // [W] scan buffer
  __shared__ int sscan[40];
  __shared__ int g_min[OT_GMAX], g_max[OT_GMAX], g_keep[OT_GMAX], g_pos[OT_GMAX];
  __shared__ int s_ng, s_nev;
  if (tid == 0) s_nev = 0;
  __syncthreads();
  const double rg = prm.range_group / prm.dlon, mexp = prm.ot_min_exp / prm.dlon;

  const int nsel = x.nsel[job];
  for (int si = 0; si < nsel; ++si) {
    const int c = x.sel[(size_t)job * x.SC + si];
    const int base = ps.pt_off[c], n = ps.pt_off[c + 1] - base;
    for (int i = tid; i < W; i += nt) {
      cnt[i] = 0;
      ymin[i] = 0x7fffffff;
      ymax[i] = -1;
      first[i] = 0x7fffffff;
      last[i] = -1;
    }
    __syncthreads();
    for (int k = tid; k < n; k += nt) {
      const u32 p = ps.pts[base + k];
      const int px = wbk_px(p), py = wbk_py(p);
      atomicAdd(&cnt[px], 1);
      atomicMin(&ymin[px], py);
      atomicMax(&ymax[px], py);
      atomicMin(&first[px], k);
      atomicMax(&last[px], k);
    }
    __syncthreads();
    // previous overturning longitude of every column (running max of "column if count >= 3")
    for (int i = tid; i < W; i += nt) tmp[i] = cnt[i] >= 3 ? i : -1;
    __syncthreads();
    wbk_block_incl_max_scan(tmp, W, sscan);
    // group starts (overturning_index.py:129): first ot longitude, or gap > range_group / dlon
    if (tid == 0) s_ng = 0;
    __syncthreads();
    // start flags into `first`-independent buffer: reuse tmp after reading prev values -> two passes
    // the start flag is kept in bit 30 of cnt
    for (int i = tid; i < W; i += nt) {
      if (cnt[i] >= 3) {
        const int prev = i > 0 ? tmp[i - 1] : -1;
        const bool start = prev < 0 || ((double)(i - prev) > rg);
        if (start) cnt[i] |= (1 << 30);
      }
    }
    __syncthreads();
    for (int i = tid; i < W; i += nt) tmp[i] = (cnt[i] >> 30) & 1;
    __syncthreads();
    const int ng = wbk_block_excl_scan(tmp, W, sscan);  // tmp[i] = number of starts before column i
    if (ng > OT_GMAX) {
      if (tid == 0) atomicOr(&d.status[job], (int)WBK_ST_EVENT_OVERFLOW);
      __syncthreads();
      continue;
    }
    for (int g = tid; g < ng; g += nt) g_max[g] = -1;
    __syncthreads();
    for (int i = tid; i < W; i += nt) {
      const int cv = cnt[i];
      if ((cv & 0x3fffffff) >= 3) {
        const bool start = (cv >> 30) & 1;
        const int g = tmp[i] + (start ? 1 : 0) - 1;  // group id of this column
        if (start) g_min[g] = i;
        atomicMax(&g_max[g], i);
      }
    }
    __syncthreads();
    // check_duplicates (overturning_index.py:136-162)
    for (int g = tid; g < ng; g += nt) g_keep[g] = 1;
    __syncthreads();
    for (int q = tid; q < ng * ng; q += nt) {
      const int a = q / ng, b = q % ng;
      if (a == b) continue;
      if (arc_subset(g_min[a], g_max[a], g_min[b], g_max[b], d.nlon)) {
        const int la = g_max[a] - g_min[a] + 1, lb = g_max[b] - g_min[b] + 1;
        const int drop = (la == lb) ? (a > b ? a : b) : (la < lb ? a : b);
        g_keep[drop] = 0;
      }
    }
    __syncthreads();
    // check_expansion (:164-166) runs only if something is left (it is a filter, so order is irrelevant)
    for (int g = tid; g < ng; g += nt)
      if (g_keep[g] && !((double)(g_max[g] - g_min[g]) >= mexp)) g_keep[g] = 0;
    __syncthreads();
    // ordered compaction -> events
    for (int g = tid; g < ng; g += nt) g_pos[g] = g_keep[g];
    __syncthreads();
    const int nkeep = wbk_block_excl_scan(g_pos, ng, sscan);
    const int ev_base = s_nev;
    __syncthreads();
    for (int g = tid; g < ng; g += nt) {
      if (!g_keep[g]) continue;
      const int e = ev_base + g_pos[g];
      if (e >= x.EC) continue;
      int lo = 0x7fffffff, hi = -1;
      for (int cx = g_min[g]; cx <= g_max[g]; ++cx) {
        if ((cnt[cx] & 0x3fffffff) > 0) {
          lo = min(lo, ymin[cx]);
          hi = max(hi, ymax[cx]);
        }
      }
      // orientation (:191-202): first point with x == min_lon vs last point with x == max_lon
      const int yw = wbk_py(ps.pts[base + first[g_min[g]]]);
      const int ye = wbk_py(ps.pts[base + last[g_max[g]]]);
      const int anti = fabs(ct.lat_deg[yw]) <= fabs(ct.lat_deg[ye]) ? 0 : 1;
      int* ev = ev_int_ptr(x, J, WBK_EV_OVERTURNING, job, e);
      ev[0] = c; ev[1] = 0; ev[2] = 0;
      ev[3] = g_min[g]; ev[4] = lo; ev[5] = g_max[g]; ev[6] = hi;
      ev[7] = anti; ev[8] = 0; ev[9] = 0;
    }
    __syncthreads();
    if (tid == 0) s_nev = ev_base + nkeep;
    __syncthreads();
  }
  if (tid == 0) {
    int nev = s_nev;
    if (nev > x.EC) {
      atomicOr(&d.status[job], (int)WBK_ST_EVENT_OVERFLOW);
      nev = x.EC;
    }
    x.ev_count[WBK_EV_OVERTURNING * J + job] = nev;
  }
}

// ------------------------------------------------------------------------------------------ streamers
#ifndef ST_THREADS
#define ST_THREADS 1024
#endif
#define PT 32            // pair-scan tile edge (one point per lane)
#define CS_SORT 16384    // surviving pairs sorted in shared memory
#define CS_SMEM ((size_t)CS_SORT * 8)
#define PS_THREADS 256
#define EARTH_R 6371.0

// sklearn DistanceMetric("haversine") between X[a] and X[b] (radians), times 6371 (streamer_index.py:130)
__device__ __forceinline__ double hav_km(double la1, double lo1, double c1, double la2, double lo2, double c2) {
  const double s0 = sin(__dmul_rn(0.5, __dsub_rn(la1, la2)));
  const double s1 = sin(__dmul_rn(0.5, __dsub_rn(lo1, lo2)));
  const double t = __dmul_rn(__dmul_rn(__dmul_rn(c1, c2), s1), s1);
  const double h = __dadd_rn(__dmul_rn(s0, s0), t);
  return __dmul_rn(__dmul_rn(2.0, asin(sqrt(h))), EARTH_R);
}

// inclusive prefix sum of doubles over data[0..n), in place
__device__ inline void block_incl_scan_f64(double* data, int n, double* scratch /* >= 34 */) {
  const int tid = wbk_tid(), nt = wbk_nthreads(), lane = wbk_lane(), warp = wbk_warp(), nwarps = nt >> 5;
  const int chunk = (n + nt - 1) / nt;
  const int b = min(n, tid * chunk), e = min(n, b + chunk);
  double s = 0.0;
  for (int i = b; i < e; ++i) s += data[i];
  double incl = s;
#pragma unroll
  for (int dd = 1; dd < 32; dd <<= 1) {
    double t = __shfl_up_sync(WBK_FULL, incl, dd);
    if (lane >= dd) incl += t;
  }
  if (lane == 31) scratch[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    double w = lane < nwarps ? scratch[lane] : 0.0;
    double wi = w;
#pragma unroll
    for (int dd = 1; dd < 32; dd <<= 1) {
      double t = __shfl_up_sync(WBK_FULL, wi, dd);
      if (lane >= dd) wi += t;
    }
    if (lane < nwarps) scratch[lane] = wi - w;
  }
  __syncthreads();
  double run = scratch[warp] + (incl - s);
  for (int i = b; i < e; ++i) {
    run += data[i];
    data[i] = run;
  }
  __syncthreads();
}

// along-contour distances on[k] and their prefix sums for every full-width contour; tile counts
__global__ void __launch_bounds__(ST_THREADS) streamer_prep_kernel(WbkDev d, WbkIdx x, PackedSet ps, CoordTabs ct,
                                                                   double* on, double* pfx, double prm_dlon,
                                                                   double geo_dis, double cont_dis) {
  const int job = blockIdx.x;
  if (job >= ps.njobs) return;
  __shared__ double sscan[40];
  const int tid = threadIdx.x, nt = blockDim.x, nlon = d.nlon;
  const int nsel = x.nsel[job];
  for (int si = 0; si < x.SC; ++si) {
    if (si >= nsel) {
      if (tid == 0) x.tile_off[(size_t)job * x.SC + si] = 0;
      continue;
    }
    const int c = x.sel[(size_t)job * x.SC + si];
    const int base = ps.pt_off[c], n = ps.pt_off[c + 1] - base;
    for (int k = tid; k < n; k += nt) {
      double v = 0.0;
      if (k > 0) {
        const u32 p0 = ps.pts[base + k - 1], p1 = ps.pts[base + k];
        const int y0 = wbk_py(p0), x0 = wbk_px(p0) % nlon, y1 = wbk_py(p1), x1 = wbk_px(p1) % nlon;
        v = hav_km(ct.lat_rad[y0], ct.lon_rad[x0], ct.cos_lat[y0], ct.lat_rad[y1], ct.lon_rad[x1], ct.cos_lat[y1]);
      }
      on[base + k] = v;
      pfx[base + k] = v;
    }
    __syncthreads();
    block_incl_scan_f64(pfx + base, n, sscan);
    // twin of every point: the point of this contour with the same y whose x differs by nlon (its periodic copy),
    // -1 if there is none.  Rows that are equal after x % nlon (check_duplicates, streamer_index.py:160-183) can only
    // pair a point with itself or its twin, so the pair scan resolves duplicate groups on the fly.
    {
      const int slot = job * x.SC + si;
      int* tw = x.flag + (size_t)slot * x.PC;
      // fp32 record of every point for the pair scan (packed point bits, lat, lon, cos lat): one coalesced 16-byte
      // load per lane and tile instead of a chain of dependent table lookups; lives in the (not yet used) pair arena
      float4* rec = reinterpret_cast<float4*>(x.pairs + (size_t)slot * x.PC);
      if (n > x.PC / 2) {
        if (tid == 0) atomicOr(&d.status[job], (int)WBK_ST_PAIR_OVERFLOW);
        for (int k = tid; k < min(n, x.PC / 2); k += nt) {
          tw[k] = -1;
          rec[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      } else {
        for (int k = tid; k < n; k += nt) {
          const u32 p = ps.pts[base + k];
          const int py = wbk_py(p);
          rec[k] = make_float4(__uint_as_float(p), (float)ct.lat_rad[py], (float)ct.lon_rad[wbk_px(p) % nlon],
                               (float)ct.cos_lat[py]);
        }
        const u32 cap = wbk_pow2_ceil((u32)(2 * n));
        u32* hkeys = reinterpret_cast<u32*>(x.hk + (size_t)slot * 2 * x.PC);
        u32* hvals = hkeys + cap;
        for (u32 i = tid; i < cap; i += nt) hkeys[i] = WBK_NONE;
        __syncthreads();
        for (int k = tid; k < n; k += nt) wbk_hash_insert32(hkeys, hvals, cap, ps.pts[base + k], (u32)k);
        __syncthreads();
        for (int k = tid; k < n; k += nt) {
          const u32 p = ps.pts[base + k];
          const int px = wbk_px(p), py = wbk_py(p);
          u32 t = WBK_NONE;
          if (px + nlon < 65536) t = wbk_hash_find32(hkeys, hvals, cap, wbk_pack_xy(px + nlon, py));
          if (t == WBK_NONE && px >= nlon) t = wbk_hash_find32(hkeys, hvals, cap, wbk_pack_xy(px - nlon, py));
          tw[k] = t == WBK_NONE ? -1 : (int)t;
        }
      }
    }
    const int T = (n + PT - 1) / PT;
    // column / row range and along-contour prefix range of every PT-point block (tile skipping in the pair scan)
    for (int b = wbk_warp(); b < T; b += (nt >> 5)) {
      int mn = 0x7fffffff, mx = -1, yn = 0x7fffffff, yx = -1;
      double pmin = 1e300, pmax = -1e300;
      for (int k = b * PT + wbk_lane(); k < min(n, (b + 1) * PT); k += 32) {
        const u32 pp = ps.pts[base + k];
        mn = min(mn, wbk_px(pp));
        mx = max(mx, wbk_px(pp));
        yn = min(yn, wbk_py(pp));
        yx = max(yx, wbk_py(pp));
        const double pf = pfx[base + k];
        pmin = fmin(pmin, pf);
        pmax = fmax(pmax, pf);
      }
      mn = wbk_warp_min(mn);
      mx = wbk_warp_max(mx);
      yn = wbk_warp_min(yn);
      yx = wbk_warp_max(yx);
#pragma unroll
      for (int dd = 16; dd > 0; dd >>= 1) {
        pmin = fmin(pmin, __shfl_xor_sync(WBK_FULL, pmin, dd));
        pmax = fmax(pmax, __shfl_xor_sync(WBK_FULL, pmax, dd));
      }
      if (wbk_lane() == 0 && b < x.NB) {
        int* bx = x.blk_x + ((size_t)job * x.SC + si) * x.NB * 4;
        bx[4 * b] = mn;
        bx[4 * b + 1] = mx;
        bx[4 * b + 2] = yn;
        bx[4 * b + 3] = yx;
        double* bp = x.blk_pf + ((size_t)job * x.SC + si) * x.NB * 2;
        bp[2 * b] = pmin;
        bp[2 * b + 1] = pmax;
      }
    }
    __syncthreads();  // block ranges are read below
    // active tiles (bi <= bj): column ranges at most 120 apart (streamer_index.py:157), some pair further than
    // cont_dis along the contour, bounding boxes within geo_dis; appended to the batch-wide work list of the pair
    // scan as slot << 40 | bi << 20 | bj
    {
      const int slot = job * x.SC + si;
      const int* bx = x.blk_x + (size_t)slot * x.NB * 4;
      const double* bp = x.blk_pf + (size_t)slot * x.NB * 2;
      const double d2r = 0.017453292519943295;
      const double dlat_deg = fabs(ct.lat_deg[1] - ct.lat_deg[0]);
      const long long nsq = (long long)T * T;
      for (long long q = tid; q < nsq; q += nt) {
        const int bi = (int)(q / T), bj = (int)(q - (long long)bi * T);
        if (bj < bi) continue;
        const int xgap = max(max(bx[4 * bj] - bx[4 * bi + 1], bx[4 * bi] - bx[4 * bj + 1]), 0);
        if (xgap > 120) continue;  // |x1 - x2| <= 120 can not hold (streamer_index.py:157)
        // cont(i, j) = pfx[j] - pfx[i] <= max pfx(bj) - min pfx(bi) (the rounded subtraction is monotone)
        if (!(__dsub_rn(bp[2 * bj + 1], bp[2 * bi]) > cont_dis * (1.0 - 2e-9))) continue;  // keeps the tolerance band
        // lower bound of the great-circle distance between the two blocks' bounding boxes: the latitude gap, and
        // the longitude gap at the most poleward latitude (h >= cos^2(lat_max) min sin^2(dlon/2) over the blocks'
        // column gaps [xgap, xgap_max]); tiles that cannot reach geo_dis are left out (1e-6 relative slack).  The
        // reference measures longitudes after x % nlon, so a column gap g is the longitude gap g * dlon folded
        // into a circle: while g * dlon < 180 degrees sin(dlon/2) grows with g and the smallest gap bounds it;
        // past 180 degrees (coarse grids, or the pole-ward ends of 2.5-degree grids) it shrinks again and is 0 at
        // g = nlon (a point and its periodic copy), so the minimum over the whole range is taken.
        const int ygap = max(max(bx[4 * bj + 2] - bx[4 * bi + 3], bx[4 * bi + 2] - bx[4 * bj + 3]), 0);
        if (EARTH_R * (dlat_deg * ygap * d2r) > geo_dis * 1.000001) continue;
        if (xgap > 0) {
          const double lat_lo = ct.lat_deg[min(bx[4 * bi + 2], bx[4 * bj + 2])], lat_hi = ct.lat_deg[max(bx[4 * bi + 3], bx[4 * bj + 3])];
          const double amax = fmax(fabs(lat_lo), fabs(lat_hi));
          const int xgap_max = max(bx[4 * bj + 1] - bx[4 * bi], bx[4 * bi + 1] - bx[4 * bj]);
          const double dlon = prm_dlon * xgap * d2r;
          double s_lon;
          if (prm_dlon * xgap_max < 180.0) {
            s_lon = sin(fmin(0.5 * dlon, 1.5707963267948966));
          } else if (xgap_max / nlon > (xgap - 1) / nlon) {
            s_lon = 0.0;  // some gap in the range is a whole number of turns
          } else {
            // |sin(g dlon / 2)| is concave between two of its zeros: its minimum over the range is at an end
            s_lon = fmin(fabs(sin(0.5 * dlon)), fabs(sin(0.5 * (prm_dlon * xgap_max * d2r))));
          }
          const double lb_lon = 2.0 * EARTH_R * asin(fmin(1.0, cos(fmin(amax, 90.0) * d2r) * s_lon));
          if (lb_lon > geo_dis * 1.000001) continue;
        }
        const int pos = atomicAdd(&x.total[0], 1);
        if (pos < x.TLC) x.tile_list[pos] = ((u64)(u32)slot << 40) | ((u64)(u32)bi << 20) | (u64)(u32)bj;
        else atomicOr(&d.status[job], (int)WBK_ST_PAIR_OVERFLOW);
      }
    }
    if (tid == 0) x.tile_off[(size_t)job * x.SC + si] = T * (T + 1) / 2;
  }
}

// tiled pair scan: geo < geo_dis and cont > cont_dis and |x1 - x2| <= 120 (streamer_index.py:130-157),
// without materialising the N x N matrices.  One WARP per 32 x 32 tile of the batch-wide active-tile list (lane = the
// point i of block bi, the 32 points of block bj are broadcast from shared memory); warps stride over the list on
// their own, no block barrier.  The haversine test is decided in fp32 on
// h = sin^2(dlat/2) + cos cos sin^2(dlon/2) against sin^2(geo_dis / 2R) with a margin derived from the error bounds
// of __sinf and of fp32 (below); only pairs inside the margin evaluate the reference's fp64 expression (and carry the
// near-threshold flag).
#define PS_WARPS (PS_THREADS / 32)
#define PS_EPS_S 1.25e-6  // absolute error bound of sqrt(h) in fp32
#define PS_EPS_H 1e-6     // relative error bound of h from the fp32 roundings
#define PS_BUF 256
#ifndef PS_MINCTA
#define PS_MINCTA 3  // resident CTAs per SM the register budget is sized for (2 -> 3: 1.03 -> 0.83 us per step)
#endif
__global__ void __launch_bounds__(PS_THREADS, PS_MINCTA) pair_scan_kernel(WbkDev d, WbkIdx x, PackedSet ps, CoordTabs ct,
                                                               const double* __restrict__ on,
                                                               const double* __restrict__ pfx, wbk_index_params prm,
                                                               int nslots) {
  __shared__ float4 sj4[PS_WARPS][PT];   // packed point (bits), lat, lon, cos(lat) of block bj in fp32
  __shared__ double sjpf[PS_WARPS][PT];  // along-contour prefix of block bj
  __shared__ u64 sbuf[PS_WARPS][PS_BUF];  // candidates of the current tile
  const int lane = wbk_lane(), warp = wbk_warp(), nlon = d.nlon;
  const int total = min(x.total[0], x.TLC);
  // margin of the fp32 test, from an absolute error bound on s = sqrt(h) = sin(distance / 2R):
  //   __sinf: 2^-21.41 absolute on [-pi, pi] (CUDA C programming guide), 3.65e-7 per sine;
  //   latitude sine argument: two latitudes rounded to fp32 (|lat| <= pi/2, 2^-24 each), their difference
  //     (|.| <= pi, 2^-23), halved: 1.2e-7;
  //   longitude sine argument: two longitudes rounded to fp32 (|lon| < 2 pi, 2^-22 each), their difference
  //     (2^-22), halved: 3.6e-7;
  //   so |s0 - s0_f| <= 4.85e-7, |s1 - s1_f| <= 7.25e-7 and |s - s_f| <= |s0 - s0_f| + |s1 - s1_f| < PS_EPS_S;
  //   relative: cos(lat) in fp32, the products and the sum of non-negative terms in fp32 and the rounding of the
  //     bounds to fp32 are each 2^-24 of h, a dozen of them < PS_EPS_H.
  // A fixed relative margin is too narrow at small geo_dis: the absolute sine error is then a large part of s.
  const double sthr = sin(prm.geo_dis / (2.0 * EARTH_R));
  const double s_lo = fmax(sthr - PS_EPS_S, 0.0), s_hi = sthr + PS_EPS_S;
  const float h_lo = (float)(s_lo * s_lo * (1.0 - PS_EPS_H)), h_hi = (float)(s_hi * s_hi * (1.0 + PS_EPS_H));
  const int nwarps_grid = gridDim.x * PS_WARPS;
  for (int w = blockIdx.x * PS_WARPS + warp; w < total; w += nwarps_grid) {
    const u64 tl = x.tile_list[w];
    const int slot = (int)(tl >> 40), bi = (int)((tl >> 20) & 0xfffffu), bj = (int)(tl & 0xfffffu);
    const int c = x.sel[slot];
    const int base = ps.pt_off[c], n = ps.pt_off[c + 1] - base;
    const int i = bi * PT + lane, j0 = bj * PT + lane;
    const float4* rec = reinterpret_cast<const float4*>(x.pairs + (size_t)slot * x.PC);  // streamer_prep_kernel
    const bool has_rec = n <= x.PC / 2;
    __syncwarp();  // the previous tile's readers are done
    if (j0 < n && has_rec) {
      sj4[warp][lane] = rec[j0];
      sjpf[warp][lane] = pfx[base + j0];
    }
    u32 pi = 0;
    float lai = 0.f, loi = 0.f, ci = 0.f;
    double pfi = 0.0;
    int ti = -1;
    if (i < n && has_rec) {
      const float4 r4 = rec[i];
      pi = __float_as_uint(r4.x);
      lai = r4.y;
      loi = r4.z;
      ci = r4.w;
      pfi = pfx[base + i];
      ti = x.flag[(size_t)slot * x.PC + i];
    }
    __syncwarp();
    // candidates are collected in a per-warp buffer and appended with ONE atomic per flush (an atomic with a return
    // value inside the loop would stall the warp for a round trip to L2 per candidate)
    const bool act = i < n && has_rec;  // without records the job carries WBK_ST_PAIR_OVERFLOW and is re-run
    const int xi = wbk_px(pi);
    const int nj = min(PT, n - bj * PT);
    int cnt = 0;
    auto flush = [&]() {
      int basep = 0;
      if (lane == 0) basep = atomicAdd(&x.cnt1[slot], cnt);
      basep = __shfl_sync(WBK_FULL, basep, 0);
      for (int k = lane; k < cnt; k += 32) {
        if (basep + k < x.PC) x.pairs2[(size_t)slot * x.PC + basep + k] = sbuf[warp][k];
        else atomicOr(&d.status[slot / x.SC], (int)WBK_ST_PAIR_OVERFLOW);
      }
      cnt = 0;
      __syncwarp();
    };
    const double cont_tol = 1e-9 * prm.cont_dis;
    for (int jj = 0; jj < nj; ++jj) {
      const int j = bj * PT + jj;
      bool cand = false;
      u64 key = 0;
      // The common case (pair too far along x, too close along the contour, or geographically too far) is decided
      // without a branch: every lane evaluates the cheap tests, only the few surviving lanes enter the block below.
      const float4 q4 = sj4[warp][jj];
      const u32 pj = __float_as_uint(q4.x);
      int dxi = xi - wbk_px(pj);
      if (dxi < 0) dxi = -dxi;
      double cont = __dsub_rn(sjpf[warp][jj], pfi);
      // hard-coded 120 index units (streamer_index.py:157), cont > cont_dis (:138).  Inside the tolerance band of
      // the threshold the reference's own summation decides: cont[i, j] = on[i+1] + ... + on[j], left to right
      // (streamer_index.py:133-135; a prefix difference differs from it by rounding)
      const bool cont_near = fabs(cont - prm.cont_dis) <= cont_tol;
      const float s0 = __sinf(0.5f * (lai - q4.y)), s1 = __sinf(0.5f * (loi - q4.z));
      const float h = s0 * s0 + ci * q4.w * s1 * s1;
      const bool pass = act && j > i && dxi <= 120 && (cont > prm.cont_dis || cont_near) && !(h > h_hi);
      if (pass) {
        if (cont_near) {
          double acc = 0.0;
          for (int k = i + 1; k <= j; ++k) acc = __dadd_rn(acc, on[base + k]);
          cont = acc;
        }
        const bool cont_ok = cont > prm.cont_dis;
        {
          {
            int near = cont_near;
            bool ok = cont_ok;
            if (h >= h_lo) {  // inside the margin: the reference's fp64 expression decides
              const int yi = wbk_py(pi), yj = wbk_py(pj);
              const double dist = hav_km(ct.lat_rad[yi], ct.lon_rad[xi % nlon], ct.cos_lat[yi], ct.lat_rad[yj],
                                         ct.lon_rad[wbk_px(pj) % nlon], ct.cos_lat[yj]);
              const bool geo_ok = dist < prm.geo_dis;
              const bool geo_near = fabs(dist - prm.geo_dis) <= 1e-9 * prm.geo_dis;
              near |= geo_near;
              if (!geo_ok && !geo_near) near = 0;  // clearly too far: the cont decision does not matter
              ok = ok && geo_ok;
              // every decision inside a tolerance band is listed, whether the pair was kept or rejected
              if (near) {
                const int pos = atomicAdd(x.near_cnt, 1);
                if (pos < x.NRC) {
                  int* rec4 = x.near_rec + 4 * pos;
                  rec4[0] = slot / x.SC;
                  rec4[1] = c;
                  rec4[2] = i;
                  rec4[3] = j | ((ok ? 1 : 0) << 28) | ((geo_near ? 1 : 0) << 29) | ((cont_near ? 1 : 0) << 30);
                }
              }
            } else if (near) {  // clearly close enough: only the cont decision is inside its band
              const int pos = atomicAdd(x.near_cnt, 1);
              if (pos < x.NRC) {
                int* rec4 = x.near_rec + 4 * pos;
                rec4[0] = slot / x.SC;
                rec4[1] = c;
                rec4[2] = i;
                rec4[3] = j | ((ok ? 1 : 0) << 28) | (1 << 30);
              }
            }
            if (ok) {
              // check_duplicates (:160-183): the rows equal to (i, j) after x % nlon are the candidates among
              // (tw i, tw j), (i, tw j), (tw i, j); they share the geographic positions, so only the index order,
              // the 120-column rule and the along-contour distance decide.  The second row of a group (row-major)
              // is dropped.
              const int tj = x.flag[(size_t)slot * x.PC + j];
              if (ti >= 0 || tj >= 0) {
                int smaller = 0;
                const int cc[3] = {ti, i, ti}, dd[3] = {tj, tj, j};
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                  const int ci2 = cc[q], dj = dd[q];
                  if (ci2 < 0 || dj < 0 || ci2 >= dj) continue;
                  int ddx = wbk_px(ps.pts[base + ci2]) - wbk_px(ps.pts[base + dj]);
                  if (ddx < 0) ddx = -ddx;
                  if (ddx > 120) continue;
                  if (!(__dsub_rn(pfx[base + dj], pfx[base + ci2]) > prm.cont_dis)) continue;
                  if (ci2 < i || (ci2 == i && dj < j)) ++smaller;
                }
                ok = smaller != 1;
              }
              if (ok) {
                cand = true;
                key = ((u64)(u32)i << 32) | ((u64)(u32)j << 1) | (u64)near;
              }
            }
          }
        }
      }
      const u32 m = __ballot_sync(WBK_FULL, cand);
      if (m) {  // warp-uniform
        if (cand) sbuf[warp][cnt + __popc(m & ((1u << lane) - 1u))] = key;
        cnt += __popc(m);
        __syncwarp();
        if (cnt > PS_BUF - 32) flush();
      }
    }
    if (cnt) flush();
  }
}

__device__ __forceinline__ int orient_i(int ax, int ay, int bx, int by, int cx, int cy) {
  return (bx - ax) * (cy - ay) - (by - ay) * (cx - ax);
}

// closed segments [p1,q1] and [p2,q2] share a point (shapely intersects on LineStrings)
__device__ __forceinline__ bool seg_intersect(int p1x, int p1y, int q1x, int q1y, int p2x, int p2y, int q2x, int q2y) {
  const int d1 = orient_i(p1x, p1y, q1x, q1y, p2x, p2y), d2 = orient_i(p1x, p1y, q1x, q1y, q2x, q2y);
  const int d3 = orient_i(p2x, p2y, q2x, q2y, p1x, p1y), d4 = orient_i(p2x, p2y, q2x, q2y, q1x, q1y);
  if (((d1 > 0 && d2 < 0) || (d1 < 0 && d2 > 0)) && ((d3 > 0 && d4 < 0) || (d3 < 0 && d4 > 0))) return true;
  if (d1 == 0 && min(p1x, q1x) <= p2x && p2x <= max(p1x, q1x) && min(p1y, q1y) <= p2y && p2y <= max(p1y, q1y)) return true;
  if (d2 == 0 && min(p1x, q1x) <= q2x && q2x <= max(p1x, q1x) && min(p1y, q1y) <= q2y && q2y <= max(p1y, q1y)) return true;
  if (d3 == 0 && min(p2x, q2x) <= p1x && p1x <= max(p2x, q2x) && min(p2y, q2y) <= p1y && p1y <= max(p2y, q2y)) return true;
  if (d4 == 0 && min(p2x, q2x) <= q1x && q1x <= max(p2x, q2x) && min(p2y, q2y) <= q1y && q1y <= max(p2y, q2y)) return true;
  return false;
}

// does contour segment [a,b] put a point of the polyline's interior into the OPEN chord (p,q)?
// (shapely LineString([p,q]).touches(contour) is false iff some segment does; SURVEY.md A.4)
__device__ __forceinline__ bool chord_violation(int px, int py, int qx, int qy, int ax, int ay, int bx, int by,
                                                int e0x, int e0y, int e1x, int e1y) {
  const int ux = qx - px, uy = qy - py;
  const int l2 = ux * ux + uy * uy;
  const int d1 = orient_i(px, py, qx, qy, ax, ay), d2 = orient_i(px, py, qx, qy, bx, by);
  const int ta = (ax - px) * ux + (ay - py) * uy, tb = (bx - px) * ux + (by - py) * uy;
  if (d1 == 0 && d2 == 0) {  // collinear: overlap of positive length
    const int lo = max(min(ta, tb), 0), hi = min(max(ta, tb), l2);
    if (lo < hi) return true;
  }
  if (d1 == 0 && ta > 0 && ta < l2 && !((ax == e0x && ay == e0y) || (ax == e1x && ay == e1y))) return true;
  if (d2 == 0 && tb > 0 && tb < l2 && !((bx == e0x && by == e0y) || (bx == e1x && by == e1y))) return true;
  if ((d1 > 0 && d2 < 0) || (d1 < 0 && d2 > 0)) {
    const int d3 = orient_i(ax, ay, bx, by, px, py), d4 = orient_i(ax, ay, bx, by, qx, qy);
    if ((d3 > 0 && d4 < 0) || (d3 < 0 && d4 > 0)) {
      // proper crossing; exempt if the crossing point is the location of a polyline end point
      const bool at_e0 = orient_i(px, py, qx, qy, e0x, e0y) == 0 && orient_i(ax, ay, bx, by, e0x, e0y) == 0;
      const bool at_e1 = orient_i(px, py, qx, qy, e1x, e1y) == 0 && orient_i(ax, ay, bx, by, e1x, e1y) == 0;
      if (!at_e0 && !at_e1) return true;
    }
  }
  return false;
}

// np.sum of a contiguous float64 slice, bit for bit: NumPy's pairwise summation (blocks of <= 128 elements with
// eight interleaved accumulators, recursive halving rounded down to multiples of 8).  The reference picks the
// longest streamer of a group with np.argmax over such sums (streamer_index.py:240-247); near ties between
// shifted base-point pairs are common on coarse grids, so the summation order matters.
__device__ inline double np_sum_leaf(const double* a, int n) {
  if (n < 8) {
    double res = 0.0;
    for (int i = 0; i < n; ++i) res = __dadd_rn(res, a[i]);
    return res;
  }
  double r[8];
  for (int j = 0; j < 8; ++j) r[j] = a[j];
  int i = 8;
  for (; i < n - (n % 8); i += 8)
    for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], a[i + j]);
  double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                         __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
  for (; i < n; ++i) res = __dadd_rn(res, a[i]);
  return res;
}

__device__ inline double np_pairwise_sum(const double* a, int n) {
  struct Frame { int off, n, stage; double left; };
  Frame st[24];
  int sp = 0;
  st[sp++] = Frame{0, n, 0, 0.0};
  double result = 0.0;
  bool have = false;
  while (sp > 0) {
    Frame& f = st[sp - 1];
    if (f.stage == 0) {
      if (f.n <= 128) {
        result = np_sum_leaf(a + f.off, f.n);
        have = true;
        --sp;
      } else {
        int n2 = f.n / 2;
        n2 -= n2 % 8;
        f.stage = 1;
        st[sp++] = Frame{f.off, n2, 0, 0.0};
        have = false;
      }
    } else if (f.stage == 1) {  // left half done
      int n2 = f.n / 2;
      n2 -= n2 % 8;
      f.left = result;
      f.stage = 2;
      st[sp++] = Frame{f.off + n2, f.n - n2, 0, 0.0};
      have = false;
    } else {  // right half done
      result = __dadd_rn(f.left, result);
      have = true;
      --sp;
    }
  }
  (void)have;
  return result;
}

// ordered compaction of src[0..P) with flag[] into dst; returns the new count to every thread
__device__ inline int compact_pairs(const u64* src, u64* dst, const int* flag, int* scanb, int P, int* sscan) {
  const int tid = wbk_tid(), nt = wbk_nthreads();
  for (int a = tid; a < P; a += nt) scanb[a] = flag[a];
  __syncthreads();
  const int total = wbk_block_excl_scan(scanb, P, sscan);
  for (int a = tid; a < P; a += nt)
    if (flag[a]) dst[scanb[a]] = src[a];
  __syncthreads();
  return total;
}

// ---------------------------------------------------------------------------------------- filter cascade
// streamer_index.py:160-264:
//   A  check_duplicates        resolved inside pair_scan_kernel through the twin index of every point
//   B  streamer_touch_kernel   (CTA per contour) check_intersections on the chords that can survive
//                                              check_overlapping, through a bin index of the contour's segments
//   C  streamer_finish_kernel  (CTA per job)   check_overlapping, sort, check_groups, events
// The reference's "while len(df) > 1" gating is kept: a stage only runs if more than one pair is left.

// B: check_intersections (:185-200) restricted to the chords that can still matter.  check_overlapping (:202-222)
// keeps only the maximal index ranges among the chords that touch, so a chord covered by a chord that is known to
// touch never needs the (expensive) geometric test.  Two rounds per contour, one CTA per (job, selected contour):
//   round 1: the maximal ranges M1 of ALL candidates are tested -> C1 = those that touch;
//   round 2: candidates covered by a member of C1 are dropped untested, the rest (ranges that were only covered by
//            failed chords) is tested.
// max(T) = max(C1 u T(round 2)): dropped chords are covered by a touching chord, hence neither maximal themselves nor
// needed to cover anything (cover is transitive).  The survivors (unordered) replace the candidate list; the finish
// kernel applies the order-free overlap filter to them.  Typical 0.25-degree contour: 26 k candidates, 120 + 390 tests.
// The geometric test: the contour's segments are binned into TB x TB lattice cells (CSR in shared memory), a chord
// is tested against the segments of the bins its line passes through.  Exact integer predicates.
#define TB_SHIFT 4                 // 16 x 16 cells per bin
#ifndef TOUCH_THREADS
#define TOUCH_THREADS 1024
#endif
#define TOUCH_MAXPTS 12288        // contour points staged in shared memory
#define TOUCH_MAXSEG 20480         // CSR capacity (segment incidences) in shared memory

__global__ void __launch_bounds__(TOUCH_THREADS) streamer_touch_kernel(WbkDev d, WbkIdx x, PackedSet ps, int nslots) {
  WBK_DYN_SMEM(unsigned char, dsm);
  const int nbx = (d.W >> TB_SHIFT) + 1, nby = (d.nlat >> TB_SHIFT) + 1;
  const int nbins = nbx * nby;
  int* boff = reinterpret_cast<int*>(dsm);                       // [nbins + 1]: bin starts, after the fill bin ends
  u32* spts = reinterpret_cast<u32*>(boff + nbins + 1);           // [TOUCH_MAXPTS]
  unsigned short* bseg = reinterpret_cast<unsigned short*>(spts + TOUCH_MAXPTS);  // [TOUCH_MAXSEG]
  __shared__ int sscan[40];
  __shared__ int s_total, s_cnt;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int lane = wbk_lane(), warp = wbk_warp(), nwarps = nt >> 5;
  // Slots are walked selection-major (all first selected contours of the jobs, then the second ones, ...): the heavy
  // slot of a job is its first one (the circumpolar contour), and a CTA-strided walk over job-major slots would hand
  // those to every SC-th CTA only while the others idle.
  for (int q = blockIdx.x; q < nslots; q += gridDim.x) {
    const int si = q / ps.njobs, job = q - si * ps.njobs;
    const int slot = job * x.SC + si;
    if (si >= x.nsel[job]) continue;
    const int P = x.cnt1[slot];
    if (P <= 1 || P > x.PC) continue;  // nothing to filter (streamer_index.py:261) / overflow already reported
    const int c = x.sel[slot];
    const int base = ps.pt_off[c], n = ps.pt_off[c + 1] - base;
    const u32* gpts = ps.pts + base;
    const u32* pts = n <= TOUCH_MAXPTS ? spts : gpts;  // the contour, in shared memory when it fits
    u64* A = x.pairs2 + (size_t)slot * x.PC;
    int* flag = x.flag + (size_t)slot * x.PC;    // 0 dropped / untested, 1 touches, 2 to be tested, 3 failed
    int* best = reinterpret_cast<int*>(x.hm1 + (size_t)slot * 2 * x.PC);  // 4 * PC ints (dedupe tables are dead)
    int* pm = best + n;
    int* wl = reinterpret_cast<int*>(x.pairs + (size_t)slot * x.PC);      // work list (the raw pair list is dead)
    u64* stage = x.hm2 + (size_t)slot * 2 * x.PC;
    if (2 * (size_t)n > 4 * (size_t)x.PC) {
      if (tid == 0) atomicOr(&d.status[job], (int)WBK_ST_PAIR_OVERFLOW);
      continue;
    }
    // ---- bin index of the n-1 segments (a segment goes into every bin its bounding box overlaps)
    __syncthreads();
    for (int b = tid; b < nbins; b += nt) boff[b] = 0;
    if (n <= TOUCH_MAXPTS)
      for (int i = tid; i < n; i += nt) spts[i] = gpts[i];
    __syncthreads();
    const bool use_bins = n <= 65535;
    if (use_bins) {
      for (int s0 = tid; s0 < n - 1; s0 += nt) {
        const u32 pa = pts[s0], pb = pts[s0 + 1];
        const int bx0 = min(wbk_px(pa), wbk_px(pb)) >> TB_SHIFT, bx1 = max(wbk_px(pa), wbk_px(pb)) >> TB_SHIFT;
        const int by0 = min(wbk_py(pa), wbk_py(pb)) >> TB_SHIFT, by1 = max(wbk_py(pa), wbk_py(pb)) >> TB_SHIFT;
        for (int by = by0; by <= by1; ++by)
          for (int bx = bx0; bx <= bx1; ++bx) atomicAdd(&boff[by * nbx + bx], 1);
      }
    }
    __syncthreads();
    const int ninc = wbk_block_excl_scan(boff, nbins, sscan);
    if (tid == 0) {
      boff[nbins] = ninc;
      s_total = ninc;
    }
    __syncthreads();
    const bool binned = use_bins && s_total <= TOUCH_MAXSEG;
    if (binned) {
      for (int s0 = tid; s0 < n - 1; s0 += nt) {
        const u32 pa = pts[s0], pb = pts[s0 + 1];
        const int bx0 = min(wbk_px(pa), wbk_px(pb)) >> TB_SHIFT, bx1 = max(wbk_px(pa), wbk_px(pb)) >> TB_SHIFT;
        const int by0 = min(wbk_py(pa), wbk_py(pb)) >> TB_SHIFT, by1 = max(wbk_py(pa), wbk_py(pb)) >> TB_SHIFT;
        for (int by = by0; by <= by1; ++by)
          for (int bx = bx0; bx <= bx1; ++bx) bseg[atomicAdd(&boff[by * nbx + bx], 1)] = (unsigned short)s0;
      }
    }
    __syncthreads();  // boff[b] is now the END of bin b (= start of bin b + 1)
    const u32 e0 = pts[0], e1 = pts[n - 1];
    const int e0x = wbk_px(e0), e0y = wbk_py(e0), e1x = wbk_px(e1), e1y = wbk_py(e1);

    for (int round = 0; round < 2; ++round) {
      // ---- best[i] = furthest ind2 of the reference set starting at ind1 == i, pm = running maximum
      for (int i = tid; i < n; i += nt) best[i] = -1;
      if (tid == 0) s_cnt = 0;
      __syncthreads();
      for (int a = tid; a < P; a += nt) {
        if (round == 0 || flag[a] == 1) {
          const u64 k = A[a];
          atomicMax(&best[(int)(k >> 32)], (int)(((u32)k) >> 1));
        }
      }
      __syncthreads();
      for (int i = tid; i < n; i += nt) pm[i] = best[i];
      __syncthreads();
      wbk_block_incl_max_scan(pm, n, sscan);
      // ---- work list: round 0 the maximal candidates, round 1 the untested candidates no touching chord covers
      for (int a = tid; a < P; a += nt) {
        if (round == 1 && flag[a] != 0) continue;
        const u64 k = A[a];
        const int i1 = (int)(k >> 32), i2 = (int)(((u32)k) >> 1);
        const bool covered = (i1 > 0 && pm[i1 - 1] >= i2) || (round == 0 ? best[i1] > i2 : best[i1] >= i2);
        if (!covered) wl[atomicAdd(&s_cnt, 1)] = a;
        flag[a] = covered ? 0 : 2;
      }
      __syncthreads();
      const int m = s_cnt;
      // ---- geometric test of the listed chords: one warp per chord, lanes over the segments of a bin
      for (int w = warp; w < m; w += nwarps) {
        const int a = wl[w];
        const u64 k = A[a];
        const u32 pi = pts[(u32)(k >> 32)], pj = pts[((u32)k) >> 1];
        const int px = wbk_px(pi), py = wbk_py(pi), qx = wbk_px(pj), qy = wbk_py(pj);
        const int x0 = min(px, qx), x1 = max(px, qx), y0 = min(py, qy), y1 = max(py, qy);
        bool bad = false;
        if (binned) {
          const int ux = qx - px, uy = qy - py;
          const int sdx = -(uy << TB_SHIFT), sdy = ux << TB_SHIFT;
          for (int by = y0 >> TB_SHIFT; by <= (y1 >> TB_SHIFT) && !bad; ++by)
            for (int bx = x0 >> TB_SHIFT; bx <= (x1 >> TB_SHIFT) && !bad; ++bx) {
              // skip bins whose (closed) cell rectangle lies strictly on one side of the chord's line: a segment can
              // only meet the chord inside a bin the chord passes through
              const int s00 = ux * ((by << TB_SHIFT) - py) - uy * ((bx << TB_SHIFT) - px);
              const int s10 = s00 + sdx, s01 = s00 + sdy, s11 = s10 + sdy;
              if (min(min(s00, s10), min(s01, s11)) > 0 || max(max(s00, s10), max(s01, s11)) < 0) continue;
              const int b = by * nbx + bx;
              const int q1 = boff[b];
              for (int q0 = b ? boff[b - 1] : 0; q0 < q1 && !bad; q0 += 32) {  // warp-uniform loop
                bool hit = false;
                const int q = q0 + lane;
                if (q < q1) {
                  const int s0 = bseg[q];
                  const u32 pa = pts[s0], pb = pts[s0 + 1];
                  const int ax = wbk_px(pa), ay = wbk_py(pa), bxx = wbk_px(pb), byy = wbk_py(pb);
                  if (!(max(ax, bxx) < x0 || min(ax, bxx) > x1 || max(ay, byy) < y0 || min(ay, byy) > y1))
                    hit = chord_violation(px, py, qx, qy, ax, ay, bxx, byy, e0x, e0y, e1x, e1y);
                }
                bad = __any_sync(WBK_FULL, hit);
              }
            }
        } else {
          for (int s00 = 0; s00 < n - 1 && !bad; s00 += 32) {
            bool hit = false;
            const int s0 = s00 + lane;
            if (s0 < n - 1) {
              const u32 pa = pts[s0], pb = pts[s0 + 1];
              const int ax = wbk_px(pa), ay = wbk_py(pa), bxx = wbk_px(pb), byy = wbk_py(pb);
              if (!(max(ax, bxx) < x0 || min(ax, bxx) > x1 || max(ay, byy) < y0 || min(ay, byy) > y1))
                hit = chord_violation(px, py, qx, qy, ax, ay, bxx, byy, e0x, e0y, e1x, e1y);
            }
            bad = __any_sync(WBK_FULL, hit);
          }
        }
        if (lane == 0) flag[a] = bad ? 3 : 1;
      }
      __syncthreads();
    }
    // ---- the touching chords (unordered) replace the candidate list
    if (tid == 0) s_cnt = 0;
    __syncthreads();
    for (int a = tid; a < P; a += nt)
      if (flag[a] == 1) stage[atomicAdd(&s_cnt, 1)] = A[a];
    __syncthreads();
    const int ns = s_cnt;
    for (int a = tid; a < ns; a += nt) A[a] = stage[a];
    if (tid == 0) x.cnt1[slot] = ns;
  }
}

// C: survivors -> row-major order, check_overlapping, check_groups, events (:202-272)
__global__ void __launch_bounds__(ST_THREADS) streamer_finish_kernel(WbkDev d, WbkIdx x, PackedSet ps,
                                                                     const double* __restrict__ on, int J) {
  const int job = blockIdx.x;
  if (job >= ps.njobs) return;
  const int tid = threadIdx.x, nt = blockDim.x;
  __shared__ int sscan[40];
  __shared__ int s_nev;
  WBK_DYN_SMEM(u64, ssort);  // [CS_SORT]
  if (tid == 0) s_nev = 0;
  __syncthreads();
  u64* B = x.pairs_b + (size_t)job * x.PC;
  int* scanb = x.scanb + (size_t)job * x.PC;
  int* label = x.label + (size_t)job * x.PC;
  u64* hk = x.hk + (size_t)job * 2 * x.PC;
  u32* hv1 = x.hv1 + (size_t)job * 2 * x.PC;

  const int nsel = x.nsel[job];
  for (int si = 0; si < nsel; ++si) {
    const int slot = job * x.SC + si;
    const int c = x.sel[slot];
    const int base = ps.pt_off[c];
    const u32* pts = ps.pts + base;
    int P = x.cnt1[slot];
    if (P > x.PC) P = 0;  // the pair arena overflowed (WBK_ST_PAIR_OVERFLOW is set): the batch is re-run with larger arenas
    u64* A = x.pairs2 + (size_t)slot * x.PC;
    int* flag = x.flag + (size_t)slot * x.PC;
    u64* cur = A;
    u64* oth = B;
    __syncthreads();
    // (2) check_intersections already ran (streamer_touch_kernel): the list holds the touching chords that are
    // not covered by another touching chord of the first round
    // (3) check_overlapping (:202-222): drop [ind1, ind2] fully covered by another pair.  Order-free form:
    // best[i] = largest ind2 among the pairs with ind1 == i, PM = running maximum of best; a pair is covered iff
    // a pair with a smaller ind1 reaches at least as far (PM[ind1-1] >= ind2) or one with the same ind1 reaches
    // further (best[ind1] > ind2; pairs are unique).
    if (P > 1) {
      const int n = ps.pt_off[c + 1] - base;
      int* best = reinterpret_cast<int*>(x.hm1 + (size_t)job * 2 * x.PC);  // >= 4 * PC ints >= n
      int* pm = best + n;
      for (int i = tid; i < n; i += nt) best[i] = -1;
      __syncthreads();
      for (int a = tid; a < P; a += nt) {
        const u64 k = cur[a];
        atomicMax(&best[(int)(k >> 32)], (int)(((u32)k) >> 1));
      }
      __syncthreads();
      for (int i = tid; i < n; i += nt) pm[i] = best[i];
      __syncthreads();
      wbk_block_incl_max_scan(pm, n, sscan);
      for (int a = tid; a < P; a += nt) {
        const u64 k = cur[a];
        const int i1 = (int)(k >> 32), i2 = (int)(((u32)k) >> 1);
        const bool covered = (i1 > 0 && pm[i1 - 1] >= i2) || best[i1] > i2;
        flag[a] = covered ? 0 : 1;
      }
      __syncthreads();
      P = compact_pairs(cur, oth, flag, scanb, P, sscan);
      u64* t = cur; cur = oth; oth = t;
    }
    // row-major order of np.nonzero for what is left: sort by (i, j)
    {
      const u32 p2 = wbk_pow2_ceil((u32)(P > 0 ? P : 1));
      if (p2 <= CS_SORT) {
        for (u32 a = tid; a < p2; a += nt) ssort[a] = (int)a < P ? cur[a] : ~0ull;
        __syncthreads();
        wbk_block_bitonic_sort(ssort, p2);
        for (int a = tid; a < P; a += nt) cur[a] = ssort[a];
        __syncthreads();
      } else {
        for (u32 a = P + tid; a < p2; a += nt) cur[a] = ~0ull;
        __syncthreads();
        wbk_block_bitonic_sort(cur, p2);
      }
    }
    // (4) check_groups (:224-251): chords that intersect describe one streamer; keep the longest
    int nout = P;
    if (P > 1) {
      // chord end points and labels live in shared memory (the sort buffer is free now) when they fit
      const bool in_smem = P <= CS_SORT * 2 / 3;
      u32* cp = reinterpret_cast<u32*>(ssort);         // [P] packed point p of chord a
      u32* cq = cp + P;                                 // [P] packed point q
      int* slab = reinterpret_cast<int*>(cq + P);       // [P] component labels
      int* lab = in_smem ? slab : label;
      __syncthreads();
      for (int a = tid; a < P; a += nt) {
        lab[a] = a;
        if (in_smem) {
          const u64 ka = cur[a];
          cp[a] = pts[(u32)(ka >> 32)];
          cq[a] = pts[((u32)ka) >> 1];
        }
      }
      __syncthreads();
      while (true) {
        int changed = 0;
        for (int a = tid; a < P; a += nt) {
          u32 pa, qa;
          if (in_smem) {
            pa = cp[a];
            qa = cq[a];
          } else {
            const u64 ka = cur[a];
            pa = pts[(u32)(ka >> 32)];
            qa = pts[((u32)ka) >> 1];
          }
          const int ax0 = min(wbk_px(pa), wbk_px(qa)), ax1 = max(wbk_px(pa), wbk_px(qa));
          const int ay0 = min(wbk_py(pa), wbk_py(qa)), ay1 = max(wbk_py(pa), wbk_py(qa));
          int m = lab[a];
          for (int b = 0; b < P; ++b) {
            const int lb = lab[b];
            if (lb >= m) continue;
            u32 pb, qb;
            if (in_smem) {
              pb = cp[b];
              qb = cq[b];
            } else {
              const u64 kb = cur[b];
              pb = pts[(u32)(kb >> 32)];
              qb = pts[((u32)kb) >> 1];
            }
            if (max(wbk_px(pb), wbk_px(qb)) < ax0 || min(wbk_px(pb), wbk_px(qb)) > ax1 ||
                max(wbk_py(pb), wbk_py(qb)) < ay0 || min(wbk_py(pb), wbk_py(qb)) > ay1)
              continue;
            if (seg_intersect(wbk_px(pa), wbk_py(pa), wbk_px(qa), wbk_py(qa), wbk_px(pb), wbk_py(pb), wbk_px(qb), wbk_py(qb)))
              m = lb;
          }
          if (m < lab[a]) {
            atomicMin(&lab[a], m);
            changed = 1;
          }
        }
        __syncthreads();
        for (int a = tid; a < P; a += nt) {  // pointer jumping
          const int l = lab[a], ll = lab[l];
          if (ll < l) {
            lab[a] = ll;
            changed = 1;
          }
        }
        if (!__syncthreads_or(changed)) break;
      }
      if (in_smem) {
        for (int a = tid; a < P; a += nt) label[a] = slab[a];
        __syncthreads();
      }
      // winner of every component: max of on[ind1 : ind2 + 1].sum(), first index on ties.  A component whose two
      // longest members lie within 1e-12 (relative) of each other is marked (bit 1 of the event's `near` column): such
      // a tie is broken by the last bits of sin / cos / asin, which are not the same in CUDA's and the host's libm,
      // so the reference may have kept the other member
      for (int a = tid; a < P; a += nt) {
        hk[a] = 0ull;
        hv1[a] = WBK_NONE;
        flag[a] = 0;  // members within the tie band, per component root
      }
      __syncthreads();
      for (int a = tid; a < P; a += nt) {
        const u64 k = cur[a];
        const int i1 = (int)(k >> 32), i2 = (int)(((u32)k) >> 1);
        const double len = np_pairwise_sum(on + base + i1, i2 - i1 + 1);  // on[ind1 : ind2 + 1].sum()
        scanb[a] = 0;
        reinterpret_cast<double*>(oth)[a] = len;  // `oth` is free until the winners are written
        atomicMax(&hk[label[a]], (u64)__double_as_longlong(len));
      }
      __syncthreads();
      for (int a = tid; a < P; a += nt) {
        const u64 k = cur[a];
        const int i1 = (int)(k >> 32), i2 = (int)(((u32)k) >> 1);
        const double len = reinterpret_cast<const double*>(oth)[a];
        (void)i1; (void)i2;
        const double top = __longlong_as_double((long long)hk[label[a]]);
        if ((u64)__double_as_longlong(len) == hk[label[a]]) atomicMin(&hv1[label[a]], (u32)a);
        if (top - len <= 1e-12 * top) atomicAdd(&flag[label[a]], 1);
      }
      __syncthreads();
      // components in order of their smallest member (combine_shared output order)
      for (int a = tid; a < P; a += nt) flag[a] = (label[a] == a ? 1 : 0) | (flag[a] >= 2 ? 2 : 0);
      __syncthreads();
      for (int a = tid; a < P; a += nt) scanb[a] = flag[a] & 1;
      __syncthreads();
      nout = wbk_block_excl_scan(scanb, P, sscan);
      for (int a = tid; a < P; a += nt)
        if (flag[a] & 1) oth[scanb[a]] = cur[hv1[a]] | ((flag[a] & 2) ? (1ull << 31) : 0ull);  // bit 31: tie mark
      __syncthreads();
      u64* t = cur; cur = oth; oth = t;
    }
    // events: polygon = contour points [ind1, ind2] (:269-272)
    const int ev_base = s_nev;
    __syncthreads();
    for (int a = tid; a < nout; a += nt) {
      const int e = ev_base + a;
      if (e >= x.EC) continue;
      const u64 k = cur[a];
      int* ev = ev_int_ptr(x, J, WBK_EV_STREAMER, job, e);
      ev[0] = c; ev[1] = (int)(k >> 32); ev[2] = (int)((((u32)k) & 0x7fffffffu) >> 1);
      for (int q = 3; q < WBK_EV_INTS - 1; ++q) ev[q] = 0;
      ev[9] = (int)(k & 1ull) | (int)((k >> 31) & 1ull) << 1;  // 1: near-threshold pair, 2: near-tie group winner
    }
    if (tid == 0) s_nev = ev_base + nout;
    __syncthreads();
  }
  if (tid == 0) {
    int nev = s_nev;
    if (nev > x.EC) {
      atomicOr(&d.status[job], (int)WBK_ST_EVENT_OVERFLOW);
      nev = x.EC;
    }
    x.ev_count[WBK_EV_STREAMER * J + job] = nev;
  }
}

__global__ void status_clear_kernel(int* status, int n, int keep_mask) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) status[i] &= keep_mask;
}

// ------------------------------------------------------------------------------------------ host API
extern "C" int wbk_index_run(wbk_ctx* ctx, int njobs, int nlevels, const int* d_job_off, const int* d_pt_off,
                             const int* d_meta, const uint32_t* d_pts, int ncontours, int npoints,
                             const double* d_coords, double* d_work, const wbk_index_params* prm, void* stream) {
  if (!ctx || !prm || njobs < 0 || nlevels < 1 || !d_job_off || !d_pt_off || !d_coords) {
    wbk_set_error("wbk_index_run: invalid argument");
    return WBK_ERR_INVALID;
  }
  if (njobs > ctx->caps.max_jobs) {
    wbk_set_error("wbk_index_run: %d jobs exceed max_jobs=%d", njobs, ctx->caps.max_jobs);
    return WBK_ERR_CAPACITY;
  }
  cudaStream_t st = (cudaStream_t)stream;
  ctx->njobs = njobs;
  ctx->nlevels = nlevels;
  if (njobs == 0) return WBK_OK;
  WbkDev& d = ctx->d;
  WbkIdx& x = ctx->x;
  const int J = ctx->caps.max_jobs;
  PackedSet ps{d_job_off, d_pt_off, d_meta, (const u32*)d_pts, njobs, nlevels, ncontours, npoints};
  CoordTabs ct = make_coords(d_coords, d.nlat);
  // status bits of an earlier index run on this context are cleared; the bits of the contour / packing stages
  // (segment, contour, pack overflow, lattice vertex) belong to the batch and stay
  WBK_LAUNCH(KID_MISC, status_clear_kernel, dim3((njobs + 255) / 256), dim3(256), 0, st, d.status, njobs,
             ~(int)(WBK_ST_PAIR_OVERFLOW | WBK_ST_EVENT_OVERFLOW | WBK_ST_SEL_OVERFLOW | WBK_ST_WIDTH_OVERFLOW |
                    WBK_ST_FETCH_OVERFLOW | WBK_ST_SPLIT_CHAINS));
  WBK_LAUNCH_CHECK();
  WBK_LAUNCH(KID_SELECT, select_kernel, dim3((njobs + 7) / 8), dim3(256), 0, st, d, x, ps, *prm, J);
  WBK_LAUNCH_CHECK();
  if (prm->do_overturnings) {
    const size_t smem = (size_t)6 * d.W * sizeof(int);
    if (smem > 200 * 1024) {
      wbk_set_error("wbk_index_run: extended width %d too large for the overturning column tables", d.W);
      return WBK_ERR_CAPACITY;
    }
    WBK_CUDA_CHECK(cudaFuncSetAttribute(overturning_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    WBK_LAUNCH(KID_OVERTURNING, overturning_kernel, dim3(njobs), dim3(OT_THREADS), smem, st, d, x, ps, ct, *prm, J);
    WBK_LAUNCH_CHECK();
  }
  if (prm->do_streamers) {
    if (!d_work) {
      wbk_set_error("wbk_index_run: d_work required for streamers");
      return WBK_ERR_INVALID;
    }
    double* on = d_work;
    double* pfx = d_work + npoints;
    const int nslots = njobs * x.SC;
    WBK_CUDA_CHECK(cudaMemsetAsync(x.total, 0, sizeof(int), st));
    WBK_CUDA_CHECK(cudaMemsetAsync(x.near_cnt, 0, sizeof(int), st));
    WBK_LAUNCH(KID_STREAMER_PREP, streamer_prep_kernel, dim3(njobs), dim3(ST_THREADS), 0, st, d, x, ps, ct, on, pfx, prm->dlon,
               prm->geo_dis, prm->cont_dis);
    WBK_LAUNCH_CHECK();
    WBK_CUDA_CHECK(cudaMemsetAsync(x.cnt1, 0, sizeof(int) * nslots, st));
    WBK_LAUNCH(KID_PAIR_SCAN, pair_scan_kernel, dim3(148 * 8), dim3(PS_THREADS), 0, st, d, x, ps, ct, (const double*)on, (const double*)pfx, *prm, nslots);
    WBK_LAUNCH_CHECK();
    {
      const int nbins = ((d.W >> TB_SHIFT) + 1) * ((d.nlat >> TB_SHIFT) + 1);
      const size_t tsmem = (size_t)(nbins + 1 + TOUCH_MAXPTS) * sizeof(int) + (size_t)TOUCH_MAXSEG * sizeof(unsigned short);
      if (tsmem > 200 * 1024) {
        wbk_set_error("wbk_index_run: grid too large for the touch-kernel bin index");
        return WBK_ERR_CAPACITY;
      }
      WBK_CUDA_CHECK(cudaFuncSetAttribute(streamer_touch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsmem));
      const int tgrid = nslots < 148 * 2 ? nslots : 148 * 2;
      WBK_LAUNCH(KID_TOUCH, streamer_touch_kernel, dim3(tgrid), dim3(TOUCH_THREADS), tsmem, st, d, x, ps, nslots);
      WBK_LAUNCH_CHECK();
    }
    WBK_CUDA_CHECK(cudaFuncSetAttribute(streamer_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CS_SMEM));
    WBK_LAUNCH(KID_FINISH, streamer_finish_kernel, dim3(njobs), dim3(ST_THREADS), CS_SMEM, st, d, x, ps, (const double*)on, J);
    WBK_LAUNCH_CHECK();
  }
  return WBK_OK;
}

extern "C" int wbk_near_list(wbk_ctx* ctx, int* d_recs, int cap, int* d_count, void* stream) {
  if (!ctx || !d_count || cap < 0 || (cap > 0 && !d_recs)) {
    wbk_set_error("wbk_near_list: invalid argument");
    return WBK_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int n = cap < ctx->x.NRC ? cap : ctx->x.NRC;
  WBK_CUDA_CHECK(cudaMemcpyAsync(d_count, ctx->x.near_cnt, sizeof(int), cudaMemcpyDeviceToDevice, st));
  if (n > 0) WBK_CUDA_CHECK(cudaMemcpyAsync(d_recs, ctx->x.near_rec, sizeof(int) * 4 * n, cudaMemcpyDeviceToDevice, st));
  return WBK_OK;
}

extern "C" int wbk_events_counts(wbk_ctx* ctx, int* h_counts, int* h_status, void* stream) {
  if (!ctx || !h_counts || !h_status) {
    wbk_set_error("wbk_events_counts: invalid argument");
    return WBK_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int n = ctx->njobs, J = ctx->caps.max_jobs;
  if (n == 0) return WBK_OK;
  for (int k = 0; k < 3; ++k)
    WBK_CUDA_CHECK(cudaMemcpyAsync(h_counts + (size_t)k * n, ctx->x.ev_count + (size_t)k * J, sizeof(int) * n, cudaMemcpyDeviceToHost, st));
  WBK_CUDA_CHECK(cudaMemcpyAsync(h_status, ctx->d.status, sizeof(int) * n, cudaMemcpyDeviceToHost, st));
  WBK_CUDA_CHECK(cudaStreamSynchronize(st));
  if (h_status[0] & WBK_ST_SPLIT_CHAINS) {
    wbk_set_error("wbk_events_raster: an event crosses the last meridian too often for the device clipper (status %d)", h_status[0]);
    return WBK_ERR_INVALID;
  }
  for (int j = 0; j < n; ++j) {
    if (h_status[j] & (WBK_ST_PAIR_OVERFLOW | WBK_ST_EVENT_OVERFLOW | WBK_ST_SEL_OVERFLOW)) {
      wbk_set_error("wbk_index_run: job %d overflowed an arena (status %d); raise pair_cap / event_cap / sel_cap", j, h_status[j]);
      return WBK_ERR_CAPACITY;
    }
  }
  return WBK_OK;
}

__global__ void events_gather_kernel(WbkIdx x, int J, int njobs, int kind, const int* __restrict__ off, int* __restrict__ o_int,
                                     double* __restrict__ o_f64, int* __restrict__ o_job) {
  const int job = blockIdx.x;
  if (job >= njobs) return;
  const int n = x.ev_count[kind * J + job], o = off[job];
  const int* si = x.ev_int + (((size_t)kind * J + job) * x.EC) * WBK_EV_INTS;
  const double* sf = x.ev_f64 + (((size_t)kind * J + job) * x.EC) * WBK_EV_F64;
  for (int i = threadIdx.x; i < n * WBK_EV_INTS; i += blockDim.x) o_int[(size_t)o * WBK_EV_INTS + i] = si[i];
  for (int i = threadIdx.x; i < n * WBK_EV_F64; i += blockDim.x) o_f64[(size_t)o * WBK_EV_F64 + i] = sf[i];
  for (int i = threadIdx.x; i < n; i += blockDim.x) o_job[o + i] = job;
}

extern "C" int wbk_events_fetch(wbk_ctx* ctx, int kind, int n, int* h_ints, double* h_f64, int* h_job, void* stream) {
  if (!ctx || kind < 0 || kind > 2 || n < 0 || (n > 0 && (!h_ints || !h_f64 || !h_job))) {
    wbk_set_error("wbk_events_fetch: invalid argument");
    return WBK_ERR_INVALID;
  }
  if (n == 0 || ctx->njobs == 0) return WBK_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int nj = ctx->njobs, J = ctx->caps.max_jobs;
  // job-major gather into the (now free) contour scratch, then one copy per table
  int* hc = new int[nj + 1];
  cudaError_t e = cudaMemcpyAsync(hc, ctx->x.ev_count + (size_t)kind * J, sizeof(int) * nj, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) {
    delete[] hc;
    WBK_CUDA_CHECK(e);
  }
  int tot = 0;
  for (int j = 0; j < nj; ++j) {
    int c = hc[j];
    hc[j] = tot;
    tot += c;
  }
  hc[nj] = tot;
  if (tot != n) {
    delete[] hc;
    wbk_set_error("wbk_events_fetch: n=%d but the context holds %d events of kind %d", n, tot, kind);
    return WBK_ERR_INVALID;
  }
  // staging buffers inside the linking scratch (sized [J][S] u32 / u64: ample for J*EC records)
  WbkDev& d = ctx->d;
  const size_t need_i = (size_t)n * WBK_EV_INTS * 4, need_f = (size_t)n * WBK_EV_F64 * 8;
  const size_t have_i = (size_t)J * d.S * 4, have_f = (size_t)J * d.S * 8;
  if (need_i > have_i || need_f > have_f || (size_t)(nj + 1) * 4 > have_i || (size_t)n * 4 > have_i) {
    delete[] hc;
    wbk_set_error("wbk_events_fetch: staging arena too small");
    return WBK_ERR_CAPACITY;
  }
  int* s_off = (int*)d.nxt;
  int* s_int = (int*)d.rid;
  int* s_job = (int*)d.prv;
  double* s_f64 = (double*)d.w64;
  e = cudaMemcpyAsync(s_off, hc, sizeof(int) * (nj + 1), cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  delete[] hc;
  WBK_CUDA_CHECK(e);
  WBK_LAUNCH(KID_EVENTS_GATHER, events_gather_kernel, dim3(nj), dim3(128), 0, st, ctx->x, J, nj, kind, (const int*)s_off, s_int, s_f64, s_job);
  WBK_LAUNCH_CHECK();
  WBK_CUDA_CHECK(cudaMemcpyAsync(h_ints, s_int, need_i, cudaMemcpyDeviceToHost, st));
  WBK_CUDA_CHECK(cudaMemcpyAsync(h_f64, s_f64, need_f, cudaMemcpyDeviceToHost, st));
  WBK_CUDA_CHECK(cudaMemcpyAsync(h_job, s_job, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  WBK_CUDA_CHECK(cudaStreamSynchronize(st));
  return WBK_OK;
}
