// Sync-free batch plumbing: device-side packing of the contour set, one summary record per batch, and a
// single gather of all event tables (+ the ring vertices of the events), so that the host enqueues a whole
// batch without waiting and reads everything back after ONE synchronisation.
#include "wbk_ctx.cuh"

// x.total layout: [0] pair-scan tiles, [1] events, [2] contours, [3] points, [8..15] summary record
__global__ void __launch_bounds__(1024) pack_scan_kernel(WbkDev d, WbkIdx x, int njobs, int* __restrict__ job_off,
                                                         int* __restrict__ pt_job_off, int cap_c, int cap_p) {
  __shared__ int sscan[40];
  for (int j = threadIdx.x; j < njobs; j += blockDim.x) {
    job_off[j] = d.out_nc[j];
    pt_job_off[j] = d.out_np[j];
  }
  __syncthreads();
  const int C = wbk_block_excl_scan(job_off, njobs, sscan);
  const int P = wbk_block_excl_scan(pt_job_off, njobs, sscan);
  const bool over = C > cap_c || P > cap_p;  // block-uniform (the scans return the totals to every thread)
  if (over) {
    // the caller's buffers are too small: nothing is packed (WBK_ST_PACK_OVERFLOW, the batch is re-run with larger
    // buffers); the job offsets are zeroed so that the index kernels of this batch see an EMPTY contour set instead of
    // offsets into buffers that were never written
    for (int j = threadIdx.x; j <= njobs; j += blockDim.x) {
      job_off[j] = 0;
      pt_job_off[j] = 0;
    }
  }
  if (threadIdx.x == 0) {
    if (!over) {
      job_off[njobs] = C;
      pt_job_off[njobs] = P;
    }
    x.total[2] = C;
    x.total[3] = P;
    if (over) atomicOr(&d.status[0], (int)WBK_ST_PACK_OVERFLOW);
  }
}

__global__ void contours_pack_auto_kernel(WbkDev d, WbkIdx x, int njobs, const int* __restrict__ job_off,
                                          const int* __restrict__ pt_job_off, int* __restrict__ pt_off,
                                          int* __restrict__ meta, u32* __restrict__ pts, int cap_c, int cap_p) {
  const int job = blockIdx.x;
  if (job >= njobs) return;
  if (x.total[2] > cap_c || x.total[3] > cap_p) {
    if (job == 0 && threadIdx.x == 0) pt_off[0] = 0;
    return;
  }
  const int nc = d.out_nc[job], np = d.out_np[job];
  const int c0 = job_off[job], p0 = pt_job_off[job];
  const int* tab = d.out_tab + (size_t)job * d.CC * 4;
  const int* sumy = d.out_sumy + (size_t)job * d.CC;
  const u32* src = d.out_pts + (size_t)job * d.R;
  for (int c = threadIdx.x; c < nc; c += blockDim.x) {
    pt_off[c0 + c] = p0 + tab[4 * c + 0];
    meta[4 * (c0 + c) + 0] = tab[4 * c + 2];
    meta[4 * (c0 + c) + 1] = tab[4 * c + 3];
    meta[4 * (c0 + c) + 2] = sumy[c];
    meta[4 * (c0 + c) + 3] = job;
  }
  for (int i = threadIdx.x; i < np; i += blockDim.x) pts[p0 + i] = src[i];
  if (job == njobs - 1 && threadIdx.x == 0) pt_off[c0 + nc] = p0 + np;
}

extern "C" int wbk_contours_pack_auto(wbk_ctx* ctx, int* d_job_off, int* d_pt_off, int* d_meta, uint32_t* d_pts,
                                      int cap_contours, int cap_points, void* stream) {
  if (!ctx || !d_job_off || !d_pt_off || !d_meta || !d_pts || cap_contours < 1 || cap_points < 1) {
    wbk_set_error("wbk_contours_pack_auto: invalid argument");
    return WBK_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int J = ctx->njobs;
  if (J == 0) return WBK_OK;
  int* d_pt_job_off = ctx->d.scan;  // scratch, free after wbk_contours
  WBK_LAUNCH(KID_CONTOUR_PACK, pack_scan_kernel, dim3(1), dim3(1024), 0, st, ctx->d, ctx->x, J, d_job_off, d_pt_job_off,
             cap_contours, cap_points);
  WBK_LAUNCH_CHECK();
  WBK_LAUNCH(KID_CONTOUR_PACK, contours_pack_auto_kernel, dim3(J), dim3(256), 0, st, ctx->d, ctx->x, J,
             (const int*)d_job_off, (const int*)d_pt_job_off, d_pt_off, d_meta, (u32*)d_pts, cap_contours, cap_points);
  WBK_LAUNCH_CHECK();
  return WBK_OK;
}

// ---------------------------------------------------------------------------------------- events: one gather
// out_int [cap][WBK_EV_INTS], out_f64 [cap][WBK_EV_F64], out_job [cap]: events kind-major, then job, then
// reference order; ring_off [cap+1] / ring_pts [cap_ring]: vertices of every streamer / cutoff ring.
__global__ void events_gather_all_kernel(WbkDev d, WbkIdx x, int J, int njobs, int* __restrict__ o_int,
                                         double* __restrict__ o_f64, int* __restrict__ o_job, int cap) {
  const int i = blockIdx.x;  // kind * njobs + job
  if (i >= 3 * njobs) return;
  const int kind = i / njobs, job = i - kind * njobs;
  const int n = x.ev_count[kind * J + job], o = x.ev_off[i];
  if (o + n > cap) {
    if (threadIdx.x == 0) atomicOr(&d.status[0], (int)WBK_ST_FETCH_OVERFLOW);
    return;
  }
  const int* si = x.ev_int + (((size_t)kind * J + job) * x.EC) * WBK_EV_INTS;
  const double* sf = x.ev_f64 + (((size_t)kind * J + job) * x.EC) * WBK_EV_F64;
  for (int k = threadIdx.x; k < n * WBK_EV_INTS; k += blockDim.x) o_int[(size_t)o * WBK_EV_INTS + k] = si[k];
  for (int k = threadIdx.x; k < n * WBK_EV_F64; k += blockDim.x) o_f64[(size_t)o * WBK_EV_F64 + k] = sf[k];
  for (int k = threadIdx.x; k < n; k += blockDim.x) o_job[o + k] = job;
}

__global__ void __launch_bounds__(1024) ring_scan_kernel(WbkDev d, WbkIdx x, int njobs, const int* __restrict__ o_int,
                                                         int* __restrict__ ring_off, int cap, int cap_ring) {
  __shared__ int sscan[40];
  const int total = x.ev_off[3 * njobs];
  if (total > cap) {
    // more events than the caller's buffers hold: the gather left records unwritten, nothing below may be trusted.
    // The batch is re-run with larger buffers (WBK_ST_FETCH_OVERFLOW).
    if (threadIdx.x == 0) {
      ring_off[0] = 0;
      atomicOr(&d.status[0], (int)WBK_ST_FETCH_OVERFLOW);
    }
    return;
  }
  const int n = total;
  const int n_box = x.ev_off[2 * njobs] - x.ev_off[njobs];  // overturnings carry a box, no ring
  const int b0 = x.ev_off[njobs];
  for (int e = threadIdx.x; e < n; e += blockDim.x) {
    const bool box = e >= b0 && e < b0 + n_box;
    ring_off[e] = box ? 0 : (o_int[(size_t)e * WBK_EV_INTS + 2] - o_int[(size_t)e * WBK_EV_INTS + 1] + 1);
  }
  __syncthreads();
  const int tot = wbk_block_excl_scan(ring_off, n, sscan);
  if (threadIdx.x == 0) {
    ring_off[n] = tot;
    if (tot > cap_ring) atomicOr(&d.status[0], (int)WBK_ST_FETCH_OVERFLOW);
  }
}

__global__ void ring_copy_kernel(WbkIdx x, int njobs, const int* __restrict__ o_int, const int* __restrict__ ring_off,
                                 const int* __restrict__ pt_off, const u32* __restrict__ pts, u32* __restrict__ ring_pts,
                                 int cap, int cap_ring) {
  const int total = x.ev_off[3 * njobs];
  if (total > cap) return;  // see ring_scan_kernel
  const int n = total;
  for (int e = blockIdx.x; e < n; e += gridDim.x) {
    const int a = ring_off[e], len = ring_off[e + 1] - a;
    if (len <= 0 || a + len > cap_ring) continue;
    const u32* src = pts + pt_off[o_int[(size_t)e * WBK_EV_INTS]] + o_int[(size_t)e * WBK_EV_INTS + 1];
    for (int k = threadIdx.x; k < len; k += blockDim.x) ring_pts[a + k] = src[k];
  }
}

// summary record: contours, points, events[3], OR of the status bits, max_nx, split events; then the work counters
// marching-squares segments, streamer candidate pairs, near-threshold decisions, active pair-scan tiles
__global__ void __launch_bounds__(1024) summary_kernel(WbkDev d, WbkIdx x, int J, int njobs, int* __restrict__ out) {
  __shared__ int acc[8];
  __shared__ unsigned long long acc64[2];
  if (threadIdx.x < 8) acc[threadIdx.x] = 0;
  if (threadIdx.x < 2) acc64[threadIdx.x] = 0;
  __syncthreads();
  int c = 0, p = 0, e0 = 0, e1 = 0, e2 = 0, st = 0;
  unsigned long long sg = 0, pr = 0;
  for (int j = threadIdx.x; j < njobs; j += blockDim.x) {
    c += d.out_nc[j];
    p += d.out_np[j];
    e0 += x.ev_count[0 * J + j];
    e1 += x.ev_count[1 * J + j];
    e2 += x.ev_count[2 * J + j];
    st |= d.status[j];
    sg += (unsigned long long)d.seg_count[j];
    for (int s = 0; s < x.SC; ++s)
      if (s < x.nsel[j]) pr += (unsigned long long)x.cnt1[j * x.SC + s];
  }
  atomicAdd(&acc[0], c); atomicAdd(&acc[1], p); atomicAdd(&acc[2], e0); atomicAdd(&acc[3], e1); atomicAdd(&acc[4], e2);
  atomicOr(&acc[5], st);
  atomicAdd(&acc64[0], sg);
  atomicAdd(&acc64[1], pr);
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 0; k < 6; ++k) out[k] = acc[k];
    out[6] = *d.max_nx;
    out[7] = x.split_count[1];
    out[8] = (int)(acc64[0] > 0x7fffffffULL ? 0x7fffffffULL : acc64[0]);
    out[9] = (int)(acc64[1] > 0x7fffffffULL ? 0x7fffffffULL : acc64[1]);
    out[10] = *x.near_cnt;
    out[11] = x.total[0];
    out[12] = out[13] = out[14] = out[15] = 0;
  }
}

extern "C" int wbk_batch_fetch(wbk_ctx* ctx, const int* d_pt_off, const uint32_t* d_pts, int* d_out_int,
                               double* d_out_f64, int* d_out_job, int* d_ring_off, uint32_t* d_ring_pts,
                               int cap_events, int cap_ring, int* d_summary, void* stream) {
  if (!ctx || !d_out_int || !d_out_f64 || !d_out_job || !d_summary || cap_events < 1) {
    wbk_set_error("wbk_batch_fetch: invalid argument");
    return WBK_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int nj = ctx->njobs, J = ctx->caps.max_jobs;
  if (nj == 0) {
    WBK_CUDA_CHECK(cudaMemsetAsync(d_summary, 0, 16 * sizeof(int), st));
    return WBK_OK;
  }
  WBK_LAUNCH(KID_EVENTS_GATHER, events_gather_all_kernel, dim3(3 * nj), dim3(128), 0, st, ctx->d, ctx->x, J, nj, d_out_int,
             d_out_f64, d_out_job, cap_events);
  WBK_LAUNCH_CHECK();
  if (d_ring_off && d_ring_pts && d_pt_off && d_pts) {
    WBK_LAUNCH(KID_EVENTS_GATHER, ring_scan_kernel, dim3(1), dim3(1024), 0, st, ctx->d, ctx->x, nj, (const int*)d_out_int,
               d_ring_off, cap_events, cap_ring);
    WBK_LAUNCH_CHECK();
    WBK_LAUNCH(KID_EVENTS_GATHER, ring_copy_kernel, dim3(148 * 4), dim3(128), 0, st, ctx->x, nj, (const int*)d_out_int,
               (const int*)d_ring_off, d_pt_off, (const u32*)d_pts, (u32*)d_ring_pts, cap_events, cap_ring);
    WBK_LAUNCH_CHECK();
  }
  WBK_LAUNCH(KID_MISC, summary_kernel, dim3(1), dim3(1024), 0, st, ctx->d, ctx->x, J, nj, d_summary);
  WBK_LAUNCH_CHECK();
  return WBK_OK;
}

// ------------------------------------------------------------------------------------------------------------
// Bit-packing of the int8 flag grids for the device -> host link (processing/events.py:105-106 makes them int8; on
// the wire one bit per cell is enough: 3.1 -> 0.39 MB per 721 x 1440 time step).  Cell c goes to bit (c & 7) of byte
// c >> 3 (numpy.unpackbits(..., bitorder="little") restores the grid).  Every thread packs 32 cells (two 16-byte
// loads) into one 32-bit store.
__global__ void __launch_bounds__(256) pack_bits_kernel(const int8_t* __restrict__ in, u32* __restrict__ out, long long ncells) {
  const long long nwords = (ncells + 31) >> 5;
  for (long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x; w < nwords; w += (long long)gridDim.x * blockDim.x) {
    const long long c0 = w << 5;
    u32 bits = 0;
    if (c0 + 32 <= ncells) {
      const uint4 a = *reinterpret_cast<const uint4*>(in + c0), b = *reinterpret_cast<const uint4*>(in + c0 + 16);
      const u32 v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const u32 x = v[k];
        const u32 nz = ((x & 0xffu) ? 1u : 0u) | ((x & 0xff00u) ? 2u : 0u) | ((x & 0xff0000u) ? 4u : 0u) | ((x & 0xff000000u) ? 8u : 0u);
        bits |= nz << (4 * k);
      }
    } else {
      for (int k = 0; k < 32 && c0 + k < ncells; ++k) bits |= (in[c0 + k] != 0 ? 1u : 0u) << k;
    }
    out[w] = bits;
  }
}

extern "C" int wbk_pack_flags(const int8_t* d_flags, uint8_t* d_packed, long long ncells, void* stream) {
  if (ncells < 0 || (ncells > 0 && (!d_flags || !d_packed)) || ((uintptr_t)d_flags & 15) || ((uintptr_t)d_packed & 3)) {
    wbk_set_error("wbk_pack_flags: invalid argument (flags 16-byte, packed 4-byte aligned; packed holds 4 * ceil(ncells / 32) bytes)");
    return WBK_ERR_INVALID;
  }
  if (ncells == 0) return WBK_OK;
  const long long nwords = (ncells + 31) >> 5;
  const int grid = (int)((nwords + 255) / 256 < 148 * 16 ? (nwords + 255) / 256 : 148 * 16);
  WBK_LAUNCH(KID_MISC, pack_bits_kernel, dim3(grid), dim3(256), 0, (cudaStream_t)stream, d_flags, (u32*)d_packed, ncells);
  WBK_LAUNCH_CHECK();
  return WBK_OK;
}

// ------------------------------------------------------------------------------------------------------------
// Occurrence counts behind a flag-frequency climatology: counts[g][k][c] += #{t : group[t] == g, flags[k][t][c] != 0}.
// A thread owns consecutive cells of one kind and walks the time axis, keeping its counts in registers while the group
// stays the same.  group[t] is the same for every thread at a given t, so the flushes (RED.ADD) do not diverge and
// happen once per run of equal groups.  Steps whose group is outside [0, ngroups) are neither loaded nor counted.  The
// flags are read exactly once; the loads of FC_STEPS steps are issued before any of them is counted.
#define FC_STEPS 4

__device__ __forceinline__ int fc_group(const int* __restrict__ group, int t, int ntime, int ngroups) {
  const int g = t < ntime ? group[t] : -1;
  return (g >= 0 && g < ngroups) ? g : -1;
}

// 16 cells per thread, one 16-byte load per step (ncells % 16 == 0, flags 16-byte aligned).  The counts are kept as
// 16-bit lanes, two per register (lo: bytes 0 and 2 of a word, hi: bytes 1 and 3), and flushed at least every 65535
// counted steps so that no lane overflows.
__device__ __forceinline__ void fc_flush16(u32* __restrict__ dst, const u32 (&lo)[4], const u32 (&hi)[4]) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const u32 c[4] = {lo[q] & 0xffffu, hi[q] & 0xffffu, lo[q] >> 16, hi[q] >> 16};
#pragma unroll
    for (int b = 0; b < 4; ++b)
      if (c[b]) atomicAdd(dst + 4 * q + b, c[b]);
  }
}

__global__ void __launch_bounds__(256, 4) flag_counts16_kernel(const int8_t* __restrict__ flags, int nkinds, int ntime,
                                                            long long ncells, const int* __restrict__ group, int ngroups,
                                                            u32* __restrict__ counts) {
  const long long nrun = ncells >> 4;
  const long long items = (long long)nkinds * nrun;
  for (long long it = (long long)blockIdx.x * blockDim.x + threadIdx.x; it < items;
       it += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(it / nrun);
    const long long c0 = (it - (long long)k * nrun) << 4;
    const int8_t* base = flags + (size_t)k * (size_t)ntime * (size_t)ncells + (size_t)c0;
    u32 lo[4] = {0u, 0u, 0u, 0u}, hi[4] = {0u, 0u, 0u, 0u};
    int cur = -1, run = 0;
    for (int t0 = 0; t0 < ntime; t0 += FC_STEPS) {
      int g[FC_STEPS];
      uint4 v[FC_STEPS];
#pragma unroll
      for (int u = 0; u < FC_STEPS; ++u) {
        g[u] = fc_group(group, t0 + u, ntime, ngroups);
        v[u] = g[u] >= 0 ? *reinterpret_cast<const uint4*>(base + (size_t)(t0 + u) * (size_t)ncells)
                         : make_uint4(0u, 0u, 0u, 0u);
      }
#pragma unroll
      for (int u = 0; u < FC_STEPS; ++u) {
        if (g[u] != cur || run == 0xffff) {
          if (cur >= 0) fc_flush16(counts + ((size_t)cur * (size_t)nkinds + (size_t)k) * (size_t)ncells + (size_t)c0, lo, hi);
#pragma unroll
          for (int q = 0; q < 4; ++q) lo[q] = hi[q] = 0u;
          cur = g[u];
          run = 0;
        }
        if (g[u] < 0) continue;
        const u32 w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          // bit 7 of every byte := byte != 0 (no carry crosses a byte: 0x7f + 0x7f < 0x100)
          const u32 nz = ((((w[q] & 0x7f7f7f7fu) + 0x7f7f7f7fu) | w[q]) >> 7) & 0x01010101u;
          lo[q] += nz & 0x00ff00ffu;
          hi[q] += (nz >> 8) & 0x00ff00ffu;
        }
        ++run;
      }
    }
    if (cur >= 0) fc_flush16(counts + ((size_t)cur * (size_t)nkinds + (size_t)k) * (size_t)ncells + (size_t)c0, lo, hi);
  }
}

// any ncells or alignment: one cell (one byte per lane and step) per thread
__global__ void __launch_bounds__(256) flag_counts1_kernel(const int8_t* __restrict__ flags, int nkinds, int ntime,
                                                           long long ncells, const int* __restrict__ group, int ngroups,
                                                           u32* __restrict__ counts) {
  const long long items = (long long)nkinds * ncells;
  for (long long it = (long long)blockIdx.x * blockDim.x + threadIdx.x; it < items;
       it += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(it / ncells);
    const long long c = it - (long long)k * ncells;
    const int8_t* base = flags + (size_t)k * (size_t)ntime * (size_t)ncells + (size_t)c;
    u32 cnt = 0;
    int cur = -1;
    for (int t0 = 0; t0 < ntime; t0 += FC_STEPS) {
      int g[FC_STEPS];
      int8_t v[FC_STEPS];
#pragma unroll
      for (int u = 0; u < FC_STEPS; ++u) {
        g[u] = fc_group(group, t0 + u, ntime, ngroups);
        v[u] = g[u] >= 0 ? base[(size_t)(t0 + u) * (size_t)ncells] : (int8_t)0;
      }
#pragma unroll
      for (int u = 0; u < FC_STEPS; ++u) {
        if (g[u] != cur) {
          if (cur >= 0 && cnt) atomicAdd(counts + ((size_t)cur * (size_t)nkinds + (size_t)k) * (size_t)ncells + (size_t)c, cnt);
          cnt = 0;
          cur = g[u];
        }
        cnt += v[u] != 0 ? 1u : 0u;
      }
    }
    if (cur >= 0 && cnt) atomicAdd(counts + ((size_t)cur * (size_t)nkinds + (size_t)k) * (size_t)ncells + (size_t)c, cnt);
  }
}

extern "C" int wbk_flag_counts(const int8_t* d_flags, int nkinds, int ntime, long long ncells, const int* d_group,
                               int ngroups, uint32_t* d_counts, void* stream) {
  if (nkinds < 1 || ntime < 0 || ncells < 0 || ngroups < 1) {
    wbk_set_error("wbk_flag_counts: invalid argument (nkinds %d, ntime %d, ncells %lld, ngroups %d)", nkinds, ntime,
                  ncells, ngroups);
    return WBK_ERR_INVALID;
  }
  if (ntime == 0 || ncells == 0) return WBK_OK;
  if (!d_flags || !d_group || !d_counts) {
    wbk_set_error("wbk_flag_counts: invalid argument (null pointer)");
    return WBK_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const bool vec = ncells % 16 == 0 && ((uintptr_t)d_flags & 15) == 0;
  const long long items = (long long)nkinds * (vec ? ncells / 16 : ncells);
  const long long blocks = (items + 255) / 256;
  const int grid = (int)(blocks < 148 * 64 ? blocks : 148 * 64);
  if (vec) {
    WBK_LAUNCH(KID_FLAG_COUNTS, flag_counts16_kernel, dim3(grid), dim3(256), 0, st, d_flags, nkinds, ntime, ncells,
               d_group, ngroups, (u32*)d_counts);
  } else {
    WBK_LAUNCH(KID_FLAG_COUNTS, flag_counts1_kernel, dim3(grid), dim3(256), 0, st, d_flags, nkinds, ntime, ncells,
               d_group, ngroups, (u32*)d_counts);
  }
  WBK_LAUNCH_CHECK();
  return WBK_OK;
}

// ------------------------------------------------------------------------------------------------------------
// Pieces of the events that straddle the last meridian (utils/index_utils.py:148-173), as the device clipper of
// wbk_events_raster left them: compacted into ring r = vertices [ring_off[r], ring_off[r+1]) of d_xy (folded index
// coordinates of the real grid), ring_ev[r] = the event (row of the wbk_batch_fetch tables) the piece belongs to.
__global__ void __launch_bounds__(1024) split_scan_kernel(WbkIdx x, int* __restrict__ ring_ev, int* __restrict__ ring_off,
                                                          int cap_rings, int cap_vertices, int* __restrict__ count) {
  __shared__ int sscan[40];
  const int n = min(min(x.split_count[1], x.SPR), cap_rings);
  for (int r = threadIdx.x; r < n; r += blockDim.x) {
    ring_off[r] = x.split_ring[4 * (size_t)r + 1];
    ring_ev[r] = x.split_ring[4 * (size_t)r + 3] >> 2;
  }
  __syncthreads();
  const int tot = wbk_block_excl_scan(ring_off, n, sscan);
  if (threadIdx.x == 0) {
    ring_off[n] = tot;
    count[0] = x.split_count[1];  // pieces found (> cap_rings: the caller's buffers were too small)
    count[1] = tot;               // their vertices (> cap_vertices: too small)
    count[2] = x.split_count[2];  // the clipper's own arenas overflowed
  }
}

__global__ void split_copy_kernel(WbkIdx x, const int* __restrict__ ring_off, int* __restrict__ xy, int cap_rings,
                                  int cap_vertices) {
  const int n = min(min(x.split_count[1], x.SPR), cap_rings);
  for (int r = blockIdx.x; r < n; r += gridDim.x) {
    const int a = ring_off[r], len = ring_off[r + 1] - a;
    if (a + len > cap_vertices) continue;
    const int* src = x.split_xy + 2 * (size_t)x.split_ring[4 * (size_t)r];
    for (int k = threadIdx.x; k < 2 * len; k += blockDim.x) xy[2 * (size_t)a + k] = src[k];
  }
}

extern "C" int wbk_split_fetch(wbk_ctx* ctx, int* d_ring_ev, int* d_ring_off, int* d_xy, int cap_rings, int cap_vertices,
                               int* d_count, void* stream) {
  if (!ctx || !d_ring_ev || !d_ring_off || !d_xy || !d_count || cap_rings < 1 || cap_vertices < 1) {
    wbk_set_error("wbk_split_fetch: invalid argument");
    return WBK_ERR_INVALID;
  }
  cudaStream_t st = (cudaStream_t)stream;
  WBK_LAUNCH(KID_EVENTS_GATHER, split_scan_kernel, dim3(1), dim3(1024), 0, st, ctx->x, d_ring_ev, d_ring_off, cap_rings,
             cap_vertices, d_count);
  WBK_LAUNCH_CHECK();
  WBK_LAUNCH(KID_EVENTS_GATHER, split_copy_kernel, dim3(148), dim3(128), 0, st, ctx->x, (const int*)d_ring_off, d_xy,
             cap_rings, cap_vertices);
  WBK_LAUNCH_CHECK();
  return WBK_OK;
}
