// Spatial pre-processing kernels: generic convolution, momentum flux, orientation flip / int16 decode,
// synthetic PV generator.  (The fused multi-pass smoothing stencil lives in wbk_smooth.cu.)
// Reference: wavebreaking/processing/spatial.py:27-128, utils/data_utils.py:196-213.
#include <type_traits>

#include "wbk_common.cuh"

__device__ __forceinline__ int wrap_idx(int i, int n) {
  i %= n;
  return i < 0 ? i + n : i;
}

// ------------------------------------------------------------------------------------------
// generic single-pass scipy.ndimage.convolve (any 2-D weights, five boundary modes)
// ------------------------------------------------------------------------------------------
#define CV_MAX_TAPS 225
struct ConvTaps {
  int n;
  int dy[CV_MAX_TAPS];
  int dx[CV_MAX_TAPS];
  double w[CV_MAX_TAPS];
};

__device__ __forceinline__ int extend_index(int i, int n, int mode, bool* outside) {
  *outside = false;
  if (i >= 0 && i < n) return i;
  switch (mode) {
    case 0:  // wrap
      return wrap_idx(i, n);
    case 1: {  // reflect: d c b a | a b c d | d c b a
      int period = 2 * n;
      int m = wrap_idx(i, period);
      return m < n ? m : period - 1 - m;
    }
    case 2: {  // mirror: d c b | a b c d | c b a
      if (n == 1) return 0;
      int period = 2 * n - 2;
      int m = wrap_idx(i, period);
      return m < n ? m : period - m;
    }
    case 3:  // nearest
      return i < 0 ? 0 : n - 1;
    default:  // constant
      *outside = true;
      return 0;
  }
}

template <typename TIn, typename TMid, typename TOut>
__global__ void convolve2d_cast_kernel(const TIn* __restrict__ in, TOut* __restrict__ out, int nlat, int nlon,
                                       ConvTaps taps, int mode, int divide, double divisor) {
  const size_t plane = (size_t)nlat * nlon;
  const TIn* src = in + plane * blockIdx.z;
  TOut* dst = out + plane * blockIdx.z;
  int gx = blockIdx.x * blockDim.x + threadIdx.x;
  int gy = blockIdx.y;
  if (gx >= nlon) return;
  double acc = 0.0;
  for (int t = 0; t < taps.n; ++t) {
    bool oy, ox;
    int yy = extend_index(gy + taps.dy[t], nlat, mode, &oy);
    int xx = extend_index(gx + taps.dx[t], nlon, mode, &ox);
    double v = (oy || ox) ? 0.0 : (double)src[(size_t)yy * nlon + xx];
    acc = __dadd_rn(acc, __dmul_rn(v, taps.w[t]));
  }
  TMid r = (TMid)acc;
  double rr = (double)r;
  if (divide) rr = __ddiv_rn(rr, divisor);
  dst[(size_t)gy * nlon + gx] = (TOut)rr;
}

extern "C" int wbk_convolve2d(const void* d_in, int in_dtype, void* d_out, int out_dtype, int ntime, int nlat,
                              int nlon, const double* h_weights, int kh, int kw, int mode, int divide, double divisor,
                              void* stream) {
  if (!d_in || !d_out || !h_weights || kh < 1 || kw < 1 || mode < 0 || mode > 4 || nlat < 1 || nlon < 1) {
    wbk_set_error("wbk_convolve2d: invalid argument");
    return WBK_ERR_INVALID;
  }
  if (ntime == 0) return WBK_OK;
  ConvTaps taps;
  taps.n = 0;
  // convolve(input, w) == correlate(input, flipped w) with origin shifted by -1 on even sizes
  const int cy = kh / 2 - ((kh % 2 == 0) ? 1 : 0);
  const int cx = kw / 2 - ((kw % 2 == 0) ? 1 : 0);
  for (int a = 0; a < kh; ++a)
    for (int b = 0; b < kw; ++b) {
      double w = h_weights[(kh - 1 - a) * kw + (kw - 1 - b)];
      if (w != 0.0) {
        if (taps.n >= CV_MAX_TAPS) {
          wbk_set_error("wbk_convolve2d: more than %d non-zero weights", CV_MAX_TAPS);
          return WBK_ERR_INVALID;
        }
        taps.dy[taps.n] = a - cy;
        taps.dx[taps.n] = b - cx;
        taps.w[taps.n] = w;
        ++taps.n;
      }
    }
  cudaStream_t st = (cudaStream_t)stream;
  if (nlat > 65535) {
    wbk_set_error("wbk_convolve2d: more than 65535 latitudes");
    return WBK_ERR_INVALID;
  }
  dim3 block(128);
  const size_t isz = in_dtype == WBK_F32 ? 4 : 8, osz = out_dtype == WBK_F32 ? 4 : 8;
  const size_t plane = (size_t)nlat * nlon;
  // gridDim.z is limited to 65535: long records go in chunks of time steps
  for (int t0 = 0; t0 < ntime; t0 += 65535) {
    const int nt = ntime - t0 < 65535 ? ntime - t0 : 65535;
    dim3 grid((nlon + 127) / 128, nlat, nt);
    const char* pin = (const char*)d_in + plane * t0 * isz;
    char* pout = (char*)d_out + plane * t0 * osz;
    if (in_dtype == WBK_F32 && out_dtype == WBK_F32) {
      WBK_LAUNCH(KID_CONVOLVE, (convolve2d_cast_kernel<float, float, float>), grid, block, 0, st, (const float*)pin, (float*)pout, nlat, nlon, taps, mode, divide, divisor);
    } else if (in_dtype == WBK_F32 && out_dtype == WBK_F64) {
      WBK_LAUNCH(KID_CONVOLVE, (convolve2d_cast_kernel<float, float, double>), grid, block, 0, st, (const float*)pin, (double*)pout, nlat, nlon, taps, mode, divide, divisor);
    } else if (in_dtype == WBK_F64 && out_dtype == WBK_F64) {
      WBK_LAUNCH(KID_CONVOLVE, (convolve2d_cast_kernel<double, double, double>), grid, block, 0, st, (const double*)pin, (double*)pout, nlat, nlon, taps, mode, divide, divisor);
    } else {
      wbk_set_error("wbk_convolve2d: unsupported dtype combination");
      return WBK_ERR_INVALID;
    }
    WBK_LAUNCH_CHECK();
  }
  return WBK_OK;
}

// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void nan_border_kernel(T* f, int nlat, int nlon, int border) {
  int gx = blockIdx.x * blockDim.x + threadIdx.x;
  if (gx >= nlon) return;
  int k = blockIdx.y;  // 0 .. 2*border-1
  int gy = k < border ? k : nlat - 2 * border + k;
  if (gy < 0 || gy >= nlat) return;
  f[(size_t)blockIdx.z * nlat * nlon + (size_t)gy * nlon + gx] = (T)__longlong_as_double(0x7ff8000000000000LL);
}

extern "C" int wbk_nan_border(void* d_field, int dtype, int ntime, int nlat, int nlon, int border, void* stream) {
  if (!d_field || border < 0 || nlat < 1 || nlon < 1) {
    wbk_set_error("wbk_nan_border: invalid argument");
    return WBK_ERR_INVALID;
  }
  if (ntime == 0 || border == 0) return WBK_OK;
  const size_t plane = (size_t)nlat * nlon;
  for (int t0 = 0; t0 < ntime; t0 += 65535) {  // gridDim.z <= 65535: long records go in chunks of time steps
    const int nt = ntime - t0 < 65535 ? ntime - t0 : 65535;
    dim3 grid((nlon + 255) / 256, 2 * border, nt);
    if (dtype == WBK_F32) WBK_LAUNCH(KID_NAN_BORDER, nan_border_kernel<float>, grid, dim3(256), 0, (cudaStream_t)stream, (float*)d_field + plane * t0, nlat, nlon, border);
    else WBK_LAUNCH(KID_NAN_BORDER, nan_border_kernel<double>, grid, dim3(256), 0, (cudaStream_t)stream, (double*)d_field + plane * t0, nlat, nlon, border);
    WBK_LAUNCH_CHECK();
  }
  return WBK_OK;
}

// ------------------------------------------------------------------------------------------
// K2: momentum flux.  One CTA per (time, lat) row: NaN-skipping zonal means of u and v, then
// (u - ubar) * (v - vbar) in the data dtype (xarray arithmetic keeps float32).
// The means are xarray's `.mean(lon)` = numpy.nanmean along the contiguous longitude axis: NaNs replaced by 0,
// numpy's PAIRWISE summation in the data dtype (blocks of <= 128 values with 8 interleaved accumulators, halves
// split at multiples of 8; numpy/_core/src/umath/loops_utils.h.src), count of the non-NaN values, and the
// quotient evaluated in float64 and rounded to the data dtype.  Reproducing that order makes the result
// bit-identical to the reference on a (time, lat, lon) array.  `sequential` selects the plain left-to-right order
// numpy uses when longitude is NOT the contiguous axis of the user's array (e.g. dims (time, lon, lat)).
// ------------------------------------------------------------------------------------------
#define MF_MAXLEAF 1024

// leaves [off, off + len) of numpy's recursion for n values, in order; returns their number
__device__ inline int mf_leaves(int n, int* off, int* len) {
  int stack_o[40], stack_n[40], sp = 0, nl = 0;
  stack_o[0] = 0;
  stack_n[0] = n;
  sp = 1;
  while (sp > 0) {
    --sp;
    const int o = stack_o[sp], m = stack_n[sp];
    if (m <= 128) {
      if (nl < MF_MAXLEAF) {
        off[nl] = o;
        len[nl] = m;
      }
      ++nl;
    } else {
      int n2 = m / 2;
      n2 -= n2 % 8;
      // right half is pushed first so that the left one is expanded first (leaves come out in order)
      stack_o[sp] = o + n2;
      stack_n[sp] = m - n2;
      ++sp;
      stack_o[sp] = o;
      stack_n[sp] = n2;
      ++sp;
    }
  }
  return nl;
}

// CF packing of an int16 field (wbk_smooth_opts): value = float64(s) * scale + offset (two roundings), s == fill -> NaN
struct MfPack {
  double scale, offset;
  int fill;  // outside the int16 range: no fill value
};

// value i of a stored field: as stored for float data, decoded for packed int16 (T = double)
template <typename TL, typename T>
__device__ __forceinline__ T mf_load(const TL* __restrict__ a, size_t i, const MfPack& pk) {
  if constexpr (std::is_same<TL, short>::value) {
    const short s = a[i];
    return (int)s == pk.fill ? (T)__longlong_as_double(0x7ff8000000000000LL)
                             : (T)__dadd_rn(__dmul_rn((double)s, pk.scale), pk.offset);
  } else {
    (void)pk;
    return a[i];
  }
}

// numpy's block sum of one leaf (n <= 128) over values with NaN -> 0
template <typename TL, typename T>
__device__ inline T mf_leaf_sum(const TL* __restrict__ a, int n, const MfPack& pk) {
  auto val = [&](int i) {
    const T v = mf_load<TL, T>(a, i, pk);
    return v != v ? (T)0 : v;
  };
  if (n < 8) {
    T res = (T)-0.0;
    for (int i = 0; i < n; ++i) res = res + val(i);
    return res;
  }
  T r[8];
  for (int j = 0; j < 8; ++j) r[j] = val(j);
  int i = 8;
  for (; i < n - (n % 8); i += 8)
    for (int j = 0; j < 8; ++j) r[j] = r[j] + val(i + j);
  T res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
  for (; i < n; ++i) res = res + val(i);
  return res;
}

// combine the leaf sums in numpy's recursion order: sum(node) = sum(left) + sum(right)
template <typename T>
__device__ inline T mf_combine(const T* leaf, int n) {
  // the recursion over (offset, length) is replayed with an explicit stack of partial results
  struct Frame { int n; int state; T left; };
  Frame st[40];
  int sp = 0, next_leaf = 0;
  T ret = (T)0;
  st[0].n = n; st[0].state = 0; st[0].left = (T)0;
  sp = 1;
  while (sp > 0) {
    Frame& f = st[sp - 1];
    if (f.n <= 128) {
      ret = leaf[next_leaf++];
      --sp;
      continue;
    }
    int n2 = f.n / 2;
    n2 -= n2 % 8;
    if (f.state == 0) {
      f.state = 1;
      st[sp].n = n2; st[sp].state = 0; st[sp].left = (T)0;
      ++sp;
    } else if (f.state == 1) {
      f.left = ret;
      f.state = 2;
      st[sp].n = f.n - n2; st[sp].state = 0; st[sp].left = (T)0;
      ++sp;
    } else {
      ret = f.left + ret;
      --sp;
    }
  }
  return ret;
}

// TL: the stored type (T, or short for packed int16 fields, which are decoded as they are loaded and give T = double)
template <typename TL, typename T>
__global__ void mflux_kernel(const TL* __restrict__ u, const TL* __restrict__ v, T* __restrict__ out, int nlon,
                             long long nrows, int sequential, MfPack pu, MfPack pv) {
  __shared__ int s_off[MF_MAXLEAF], s_len[MF_MAXLEAF];
  __shared__ T s_leaf[2][MF_MAXLEAF];
  __shared__ int s_nl, s_cnt[2];
  __shared__ double means[2];
  if (threadIdx.x == 0) s_nl = sequential ? 0 : mf_leaves(nlon, s_off, s_len);
  __syncthreads();
  const int nl = s_nl;
  for (long long r = blockIdx.x; r < nrows; r += gridDim.x) {
    const size_t row = (size_t)r * nlon;
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    int cu = 0, cv = 0;
    for (int x = threadIdx.x; x < nlon; x += blockDim.x) {
      const T a = mf_load<TL, T>(u, row + x, pu), b = mf_load<TL, T>(v, row + x, pv);
      cu += a == a;
      cv += b == b;
    }
    atomicAdd(&s_cnt[0], cu);
    atomicAdd(&s_cnt[1], cv);
    if (!sequential) {
      for (int k = threadIdx.x; k < 2 * nl; k += blockDim.x) {
        const int w = k >= nl, l = w ? k - nl : k;
        s_leaf[w][l] = mf_leaf_sum<TL, T>((w ? v : u) + row + s_off[l], s_len[l], w ? pv : pu);
      }
    }
    __syncthreads();
    if (threadIdx.x < 2) {
      const TL* src = (threadIdx.x ? v : u) + row;
      const MfPack& pk = threadIdx.x ? pv : pu;
      T tot;
      if (sequential) {
        tot = (T)0;  // strided reduce: out = a[0], then out += a[i] one row of the other axis at a time
        for (int x = 0; x < nlon; ++x) {
          const T val = mf_load<TL, T>(src, x, pk);
          tot = x == 0 ? (val != val ? (T)0 : val) : tot + (val != val ? (T)0 : val);
        }
      } else {
        tot = mf_combine<T>(s_leaf[threadIdx.x], nlon);
      }
      // numpy's _divide_by_count: true_divide(float, intp) runs in float64 and is cast back to the data dtype
      means[threadIdx.x] = (double)(T)((double)tot / (double)s_cnt[threadIdx.x]);
    }
    __syncthreads();
    const T mu = (T)means[0], mv = (T)means[1];
    for (int x = threadIdx.x; x < nlon; x += blockDim.x) {
      T up = mf_load<TL, T>(u, row + x, pu) - mu;
      T vp = mf_load<TL, T>(v, row + x, pv) - mv;
      out[row + x] = up * vp;
    }
    __syncthreads();
  }
}

static MfPack mf_pack(const wbk_smooth_opts& o) {
  return MfPack{o.scale, o.offset, o.has_fill ? o.fill : 0x7fffffff};
}

extern "C" int wbk_mflux(const void* d_u, const void* d_v, void* d_out, int dtype, int ntime, int nlat, int nlon,
                         int sequential, const wbk_smooth_opts* packing, void* stream) {
  if (!d_u || !d_v || !d_out || nlat < 1 || nlon < 1 || (!sequential && nlon > 64 * MF_MAXLEAF)) {
    wbk_set_error("wbk_mflux: invalid argument");
    return WBK_ERR_INVALID;
  }
  if (dtype != WBK_F32 && dtype != WBK_F64 && dtype != WBK_I16) {
    wbk_set_error("wbk_mflux: unsupported dtype %d", dtype);
    return WBK_ERR_INVALID;
  }
  if ((dtype == WBK_I16) != (packing != nullptr)) {
    wbk_set_error("wbk_mflux: packed int16 u / v need their two packings (u, v); float u / v take none");
    return WBK_ERR_INVALID;
  }
  if (packing && (packing[0].flip_lat || packing[0].flip_lon || packing[1].flip_lat || packing[1].flip_lon)) {
    wbk_set_error("wbk_mflux: the flux is computed and written in stored order (packing with flip set)");
    return WBK_ERR_INVALID;
  }
  if (ntime == 0) return WBK_OK;
  const long long nrows = (long long)nlat * ntime;
  dim3 grid((unsigned)(nrows < (1 << 20) ? nrows : (1 << 20)));
  cudaStream_t st = (cudaStream_t)stream;
  const MfPack none{1.0, 0.0, 0x7fffffff};
  if (dtype == WBK_F32) WBK_LAUNCH(KID_MFLUX, (mflux_kernel<float, float>), grid, dim3(256), 0, st, (const float*)d_u, (const float*)d_v, (float*)d_out, nlon, nrows, sequential, none, none);
  else if (dtype == WBK_F64) WBK_LAUNCH(KID_MFLUX, (mflux_kernel<double, double>), grid, dim3(256), 0, st, (const double*)d_u, (const double*)d_v, (double*)d_out, nlon, nrows, sequential, none, none);
  else WBK_LAUNCH(KID_MFLUX, (mflux_kernel<short, double>), grid, dim3(256), 0, st, (const short*)d_u, (const short*)d_v, (double*)d_out, nlon, nrows, sequential, mf_pack(packing[0]), mf_pack(packing[1]));
  WBK_LAUNCH_CHECK();
  return WBK_OK;
}

// ------------------------------------------------------------------------------------------
// orientation fix + (for packed int16 input) the CF decode float64(v) * scale_factor + add_offset; time is folded
// into blockIdx.x so that series of any length fit the grid limits
template <typename TIn, typename TOut>
__global__ void orient_kernel(const TIn* __restrict__ in, TOut* __restrict__ out, int nlat, int nlon, long long rows,
                              int flip_lat, int flip_lon, bool decode, double scale, double offset, int fill) {
  for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
    const long long t = r / nlat;
    const int gy = (int)(r - t * nlat);
    const int sy = flip_lat ? nlat - 1 - gy : gy;
    const TIn* src = in + ((size_t)t * nlat + sy) * nlon;
    TOut* dst = out + (size_t)r * nlon;
    for (int gx = threadIdx.x; gx < nlon; gx += blockDim.x) {
      const TIn v = src[flip_lon ? nlon - 1 - gx : gx];
      if (decode) {
        dst[gx] = (int)v == fill ? (TOut)__longlong_as_double(0x7ff8000000000000LL)
                                 : (TOut)__dadd_rn(__dmul_rn((double)v, scale), offset);
      } else {
        dst[gx] = (TOut)v;
      }
    }
  }
}

extern "C" int wbk_orient(const void* d_in, int in_dtype, void* d_out, int ntime, int nlat, int nlon,
                          const wbk_smooth_opts* opts, void* stream) {
  if (!d_in || !d_out || d_in == d_out || nlat < 1 || nlon < 1 || ntime < 0) {
    wbk_set_error("wbk_orient: invalid argument (in-place is not supported)");
    return WBK_ERR_INVALID;
  }
  if (ntime == 0) return WBK_OK;
  const int fl = opts ? opts->flip_lat : 0, fo = opts ? opts->flip_lon : 0;
  const double sc = opts ? opts->scale : 1.0, of = opts ? opts->offset : 0.0;
  const int fill = (opts && opts->has_fill) ? opts->fill : 0x7fffffff;
  const long long rows = (long long)ntime * nlat;
  const int grid = (int)(rows < 148 * 16 ? rows : 148 * 16);
  cudaStream_t st = (cudaStream_t)stream;
  if (in_dtype == WBK_F32) WBK_LAUNCH(KID_FLIP, (orient_kernel<float, float>), dim3(grid), dim3(256), 0, st, (const float*)d_in, (float*)d_out, nlat, nlon, rows, fl, fo, false, sc, of, fill);
  else if (in_dtype == WBK_F64) WBK_LAUNCH(KID_FLIP, (orient_kernel<double, double>), dim3(grid), dim3(256), 0, st, (const double*)d_in, (double*)d_out, nlat, nlon, rows, fl, fo, false, sc, of, fill);
  else if (in_dtype == WBK_I16) WBK_LAUNCH(KID_FLIP, (orient_kernel<short, double>), dim3(grid), dim3(256), 0, st, (const short*)d_in, (double*)d_out, nlat, nlon, rows, fl, fo, true, sc, of, fill);
  else {
    wbk_set_error("wbk_orient: unsupported dtype");
    return WBK_ERR_INVALID;
  }
  WBK_LAUNCH_CHECK();
  return WBK_OK;
}

extern "C" int wbk_flip(const void* d_in, void* d_out, int dtype, int ntime, int nlat, int nlon, int flip_lat,
                        int flip_lon, void* stream) {
  if (dtype != WBK_F32 && dtype != WBK_F64) {
    wbk_set_error("wbk_flip: unsupported dtype");
    return WBK_ERR_INVALID;
  }
  wbk_smooth_opts o = {};
  o.flip_lat = flip_lat;
  o.flip_lon = flip_lon;
  o.scale = 1.0;
  return wbk_orient(d_in, dtype, d_out, ntime, nlat, nlon, &o, stream);
}

// ------------------------------------------------------------------------------------------
// synthetic PV (mirror of wavebreaking_b200/synthetic.py)
// ------------------------------------------------------------------------------------------
#define SYN_MAX_BLOB 32
struct SynthParams {
  double A, k, tilt, c, env0, env1, env_speed, blob_amp, sh_shift, A2, k2, c2, tilt2;
  int n_blob;
  double lat0[2][SYN_MAX_BLOB], lon0[2][SYN_MAX_BLOB], rad[2][SYN_MAX_BLOB];
};

__device__ __forceinline__ double synth_background(double alat, double lam_deg, double hours, const SynthParams& p) {
  const double d2r = 0.017453292519943295;
  double lam = lam_deg * d2r;
  double env = p.env0 + p.env1 * cos(lam - p.env_speed * hours * d2r);
  double phase = p.k * (lam - p.c * hours * d2r) + p.tilt * (alat - 45.0) / 10.0 + 0.7 * sin(2.0 * lam);
  double phase2 = p.k2 * (lam - p.c2 * hours * d2r) + p.tilt2 * (alat - 45.0) / 10.0;
  double phi = alat - p.A * env * sin(phase) - p.A2 * sin(phase2);
  double s = sin(phi * d2r) / sin(45.0 * d2r);
  double a = fabs(s);
  double r = 2.0 * a * a * a;
  return s < 0 ? -r : r;
}

template <typename T>
__global__ void synth_pv_kernel(T* out, int nlat, int nlon, double hour0, double hour_step, SynthParams p) {
  int gx = blockIdx.x * blockDim.x + threadIdx.x;
  if (gx >= nlon) return;
  int gy = blockIdx.y;
  int t = blockIdx.z;
  const double d2r = 0.017453292519943295;
  double hours = hour0 + hour_step * t;
  double lat = -90.0 + 180.0 * gy / (double)(nlat - 1);
  double lon = gx * (360.0 / nlon);
  bool south = lat < 0;
  double alat = fabs(lat);
  int hemi = south ? 1 : 0;
  double pv = synth_background(alat, south ? lon + p.sh_shift : lon, hours, p);
  for (int b = 0; b < p.n_blob; ++b) {
    double lonc = fmod(p.lon0[hemi][b] + p.c * hours, 360.0);
    double bg = synth_background(p.lat0[hemi][b], lonc + (hemi ? p.sh_shift : 0.0), hours, p);
    double sign = bg > 2.0 ? -1.0 : 1.0;
    double dl = fmod(lon - lonc + 180.0, 360.0);
    if (dl < 0) dl += 360.0;
    dl -= 180.0;
    double dy = alat - p.lat0[hemi][b];
    double dxs = dl * cos(p.lat0[hemi][b] * d2r);
    double d2 = dy * dy + dxs * dxs;
    double rad = p.rad[hemi][b];
    pv += sign * p.blob_amp * exp(-d2 / (2.0 * rad * rad));
  }
  out[((size_t)t * nlat + gy) * nlon + gx] = (T)(south ? -pv : pv);
}

extern "C" int wbk_synth_pv(void* d_out, int dtype, int ntime, int nlat, int nlon, double hour0, double hour_step,
                            const double* h_blobs, int n_blob, void* stream) {
  if (!d_out || nlat < 2 || nlon < 1 || n_blob < 0 || n_blob > SYN_MAX_BLOB || (n_blob > 0 && !h_blobs) || ntime > 65535 ||
      nlat > 65535) {
    wbk_set_error("wbk_synth_pv: invalid argument (at most 65535 time steps per call)");
    return WBK_ERR_INVALID;
  }
  if (ntime == 0) return WBK_OK;
  SynthParams p;
  // frozen recipe: keep in sync with wavebreaking_b200/synthetic.py PARAMS
  p.A = 12.0; p.k = 7.0; p.tilt = 2.6; p.c = 0.5; p.env0 = 0.6; p.env1 = 0.4; p.env_speed = 1.5;
  p.blob_amp = 3.0; p.sh_shift = 37.0; p.A2 = 4.5; p.k2 = 19.0; p.c2 = 1.1; p.tilt2 = 2.0; p.n_blob = n_blob;
  for (int h = 0; h < 2; ++h)
    for (int b = 0; b < n_blob; ++b) {
      p.lat0[h][b] = h_blobs[(h * n_blob + b) * 3 + 0];
      p.lon0[h][b] = h_blobs[(h * n_blob + b) * 3 + 1];
      p.rad[h][b] = h_blobs[(h * n_blob + b) * 3 + 2];
    }
  dim3 grid((nlon + 127) / 128, nlat, ntime);
  if (dtype == WBK_F32) WBK_LAUNCH(KID_SYNTH, synth_pv_kernel<float>, grid, dim3(128), 0, (cudaStream_t)stream, (float*)d_out, nlat, nlon, hour0, hour_step, p);
  else WBK_LAUNCH(KID_SYNTH, synth_pv_kernel<double>, grid, dim3(128), 0, (cudaStream_t)stream, (double*)d_out, nlat, nlon, hour0, hour_step, p);
  WBK_LAUNCH_CHECK();
  return WBK_OK;
}
