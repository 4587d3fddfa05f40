// Eulerian grid operators (one launch per reference operator).
// Each operator reproduces the cells the reference MPI wrapper writes:
// interior + six boundary slabs + zeroed physical ring (SbGeom::written/in_ring).
#include "sb200_common.h"

#include <cstdarg>

static thread_local char g_err[512] = "";
void sb_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
extern "C" const char* sb200_last_error(void) { return g_err; }
extern "C" int sb200_version(void) { return 100; }

// ------------------------------------------------------------ pointwise ----
template <typename T>
struct FillOp {
  T* f;
  T v;
  SB_D void operator()(long long i) const { f[i] = v; }
};
template <typename T>
struct SumOp {
  T* s;
  const T* a;
  const T* b;
  SB_D void operator()(long long i) const { s[i] = a[i] + b[i]; }
};
template <typename T>
struct CopyOp {
  T* d;
  const T* s;
  SB_D void operator()(long long i) const { d[i] = s[i]; }
};
template <typename T>
struct SaxpbyOp {
  T* s;
  const T* a;
  const T* b;
  T pa, pb;
  SB_D void operator()(long long i) const { s[i] = pa * a[i] + pb * b[i]; }
};
template <typename T>
struct CrossOp {
  T* r;
  const T* a;
  const T* b;
  long long n;
  SB_D void operator()(long long i) const {
    const T a0 = a[i], a1 = a[i + n], a2 = a[i + 2 * n];
    const T b0 = b[i], b1 = b[i + n], b2 = b[i + 2 * n];
    r[i] = a1 * b2 - a2 * b1;
    r[i + n] = a2 * b0 - a0 * b2;
    r[i + 2 * n] = a0 * b1 - a1 * b0;
  }
};
template <typename T>
struct AddFixedOp {
  T* f;
  long long n;
  int ncomp;
  T v0, v1, v2;
  SB_D void operator()(long long i) const {
    f[i] += v0;
    if (ncomp > 1) f[i + n] += v1;
    if (ncomp > 2) f[i + 2 * n] += v2;
  }
};

extern "C" int sb200_set_fixed_val(int dtype, void* field, int64_t count, double value, void* stream) {
  SB_REQUIRE(field || count == 0, "set_fixed_val: null field");
  if (value == 0.0) {
    size_t w = dtype == SB200_F32 ? 4 : 8;
    int e = sb_memset_async(field, 0, (size_t)count * w, stream);
    if (e) {
      sb_set_error("memset: %s", sb_error_string(e));
      return -2;
    }
    return 0;
  }
  SB_DISPATCH_DTYPE(dtype, return sb_launch_flat(count, FillOp<T>{(T*)field, (T)value}, stream, "fill"));
}
extern "C" int sb200_elementwise_sum(int dtype, void* sum, const void* a, const void* b, int64_t count,
                                     void* stream) {
  SB_DISPATCH_DTYPE(dtype, return sb_launch_flat(count, SumOp<T>{(T*)sum, (const T*)a, (const T*)b},
                                                 stream, "sum"));
}
extern "C" int sb200_elementwise_copy(int dtype, void* dst, const void* src, int64_t count, void* stream) {
  SB_DISPATCH_DTYPE(dtype,
                    return sb_launch_flat(count, CopyOp<T>{(T*)dst, (const T*)src}, stream, "copy"));
}
extern "C" int sb200_elementwise_saxpby(int dtype, void* sum, const void* a, double pa, const void* b,
                                        double pb, int64_t count, void* stream) {
  SB_DISPATCH_DTYPE(dtype, return sb_launch_flat(
                               count, SaxpbyOp<T>{(T*)sum, (const T*)a, (const T*)b, (T)pa, (T)pb},
                               stream, "saxpby"));
}
extern "C" int sb200_elementwise_cross_product(int dtype, void* result, const void* f1, const void* f2,
                                               int64_t count, void* stream) {
  SB_DISPATCH_DTYPE(dtype, return sb_launch_flat(
                               count, CrossOp<T>{(T*)result, (const T*)f1, (const T*)f2, count}, stream,
                               "cross"));
}
extern "C" int sb200_add_fixed_val(int dtype, void* field, int ncomp, int64_t count, const double* vals,
                                   void* stream) {
  SB_REQUIRE(ncomp >= 1 && ncomp <= 3 && vals, "add_fixed_val: bad ncomp/vals");
  double v[3] = {vals[0], ncomp > 1 ? vals[1] : 0.0, ncomp > 2 ? vals[2] : 0.0};
  SB_DISPATCH_DTYPE(dtype, return sb_launch_flat(
                               count, AddFixedOp<T>{(T*)field, count, ncomp, (T)v[0], (T)v[1], (T)v[2]},
                               stream, "add_fixed"));
}

// -------------------------------------------------------------- stencils ---
// curl components of a (3,z,y,x) field at linear index i (unit prefactor applied by caller)
template <typename T>
SB_D void curl3_at(const SbGeom& g, const T* f, long long i, T p, T& cx, T& cy, T& cz) {
  const long long n = g.vol, sy = g.mx, sz = g.plane;
  const T* fx = f;
  const T* fy = f + n;
  const T* fz = f + 2 * n;
  cx = p * (fz[i + sy] - fz[i - sy] - fy[i + sz] + fy[i - sz]);
  cy = p * (fx[i + sz] - fx[i - sz] - fz[i + 1] + fz[i - 1]);
  cz = p * (fy[i + 1] - fy[i - 1] - fx[i + sy] + fx[i - sy]);
}

template <typename T>
struct UpdateVorticityOp {
  T* w;
  const T* f;
  T p;
  SB_D void operator()(const SbGeom& g, int z, int y, int x) const {
    if (!g.deep(z, y, x) && !g.written(z, y, x, 1)) return;
    const long long i = g.idx(z, y, x);
    if (g.dim == 3) {
      T cx, cy, cz;
      curl3_at(g, f, i, p, cx, cy, cz);
      w[i] += cx;
      w[i + g.vol] += cy;
      w[i + 2 * g.vol] += cz;
    } else {
      // omega += p * (dFy/dx - dFx/dy), F is (2,y,x)
      const T* fx = f;
      const T* fy = f + g.vol;
      w[i] += p * (fy[i + 1] - fy[i - 1] - fx[i + g.mx] + fx[i - g.mx]);
    }
  }
};

// ---- forcing update for a forcing field that is zero almost everywhere (immersed-boundary forcing
// lives within two cells of the Lagrangian points).  The padded array is cut into flat chunks of 1024
// consecutive cells.  Pass 1 reads F once (vectorised, the only dense traffic: 3 W per cell) and flags
// the chunks that hold a non-zero value; pass 2 applies UpdateVorticityOp's arithmetic to the chunks
// whose stencil neighbourhood (x +- 1, y +- 1, z +- 1) touches a flagged chunk and skips the others
// (omega + prefactor * curl(0) == omega); sb200_clear_flagged_tiles zeroes the flagged chunks only, which
// is the `F = 0` that ends the step (flow_simulators_mpi_3d.py:422-424).  Exact for any F.
#define SB_CHUNK 1024
// work buffer (ints): flags[n] | active[n] | list of flagged chunks [n] | list of active chunks [n] | 2 counters
struct SbChunkBuf {
  int *flags, *active, *nz_list, *act_list, *count;
};
static inline SbChunkBuf sb_chunk_buf(void* p, long long n) {
  int* b = (int*)p;
  return SbChunkBuf{b, b + n, b + 2 * n, b + 3 * n, b + 4 * n};
}
template <typename T>
__global__ void __launch_bounds__(256)
    sb_flag_nonzero_chunks_kernel(const T* __restrict__ f, int ncomp, long long vol, long long nchunks, SbChunkBuf b) {
  const bool vec = (vol & 3) == 0;
  for (long long c = blockIdx.x; c < nchunks; c += gridDim.x) {
    const long long i = c * SB_CHUNK + 4 * (long long)threadIdx.x;
    bool nz = false;
    if (vec && i + 3 < vol) {
      for (int k = 0; k < ncomp; ++k) {
        const T* q = f + k * vol + i;
        if constexpr (sizeof(T) == 4) {
          const float4 v = *reinterpret_cast<const float4*>(q);
          nz = nz || v.x != 0.f || v.y != 0.f || v.z != 0.f || v.w != 0.f;
        } else {
          nz = nz || q[0] != T(0) || q[1] != T(0) || q[2] != T(0) || q[3] != T(0);
        }
      }
    } else {
      for (int k = 0; k < ncomp; ++k)
        for (int e = 0; e < 4; ++e)
          if (i + e < vol) nz = nz || f[k * vol + i + e] != T(0);
    }
    // the first thread to flag a chunk appends it to the list
    if (nz && atomicAdd(&b.flags[c], 1) == 0) b.nz_list[atomicAdd(&b.count[0], 1)] = (int)c;
  }
}
// every chunk whose stencil (x +- 1, y +- 1, z +- 1) reads a flagged chunk becomes active
__global__ void __launch_bounds__(256) sb_dilate_chunks_kernel(SbGeom g, long long nchunks, SbChunkBuf b) {
  const int n = b.count[0];
  const long long offs[3] = {1, (long long)g.mx, g.plane};
  const int noff = g.dim == 3 ? 3 : 2;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
    const long long c = b.nz_list[k], lo = c * SB_CHUNK, hi = lo + SB_CHUNK - 1;
    if (atomicAdd(&b.active[c], 1) == 0) b.act_list[atomicAdd(&b.count[1], 1)] = (int)c;
    for (int o = 0; o < noff; ++o)
      for (int sgn = -1; sgn <= 1; sgn += 2) {
        const long long a = lo + sgn * offs[o], e = hi + sgn * offs[o];
        if (e < 0) continue;
        for (long long q = (a < 0 ? 0 : a / SB_CHUNK); q <= e / SB_CHUNK && q < nchunks; ++q)
          if (atomicAdd(&b.active[q], 1) == 0) b.act_list[atomicAdd(&b.count[1], 1)] = (int)q;
      }
  }
}
template <typename T>
__global__ void __launch_bounds__(256)
    sb_update_vorticity_flagged_kernel(SbGeom g, T* __restrict__ w, const T* __restrict__ f, T p, SbChunkBuf b) {
  const UpdateVorticityOp<T> op{w, f, p};
  const int n = b.count[1];
  for (int k = blockIdx.x; k < n; k += gridDim.x) {
    const long long c = b.act_list[k];
    for (int e = 0; e < 4; ++e) {
      const long long i = c * SB_CHUNK + e * 256 + threadIdx.x;
      if (i >= g.vol) continue;
      int z, y, x;
      if (g.vol < (1LL << 31)) {  // 32-bit divisions (a 512^3 slab has 1.4e8 cells)
        const unsigned ui = (unsigned)i, uz = ui / (unsigned)g.plane, r = ui - uz * (unsigned)g.plane;
        const unsigned uy = r / (unsigned)g.mx;
        z = (int)uz, y = (int)uy, x = (int)(r - uy * (unsigned)g.mx);
      } else {
        z = (int)(i / g.plane);
        const long long r = i - (long long)z * g.plane;
        y = (int)(r / g.mx), x = (int)(r - (long long)y * g.mx);
      }
      op(g, z, y, x);
    }
  }
}
template <typename T>
__global__ void __launch_bounds__(256)
    sb_clear_flagged_kernel(T* __restrict__ f, int ncomp, long long vol, SbChunkBuf b) {
  const int n = b.count[0];
  for (int k = blockIdx.x; k < n; k += gridDim.x) {
    const long long c = b.nz_list[k];
    for (int e = 0; e < 4; ++e) {
      const long long i = c * SB_CHUNK + e * 256 + threadIdx.x;
      if (i < vol)
        for (int q = 0; q < ncomp; ++q) f[q * vol + i] = T(0);
    }
  }
}
static inline long long sb_chunk_count(const SbGeom& g) { return (g.vol + SB_CHUNK - 1) / SB_CHUNK; }
static inline unsigned sb_chunk_grid(long long nchunks) {
  const long long cap = 148LL * 16;
  return (unsigned)(nchunks < cap ? nchunks : cap);
}
static inline size_t sb_chunk_buf_bytes(long long nchunks) { return sizeof(int) * (size_t)(4 * nchunks + 4); }

extern "C" int64_t sb200_tile_flag_count(const sb200_grid_t* gr) {
  SbGeom g;
  if (sb_make_geom(gr, &g) != 0) return 0;
  return (int64_t)sb_chunk_buf_bytes(sb_chunk_count(g));
}
extern "C" int sb200_update_vorticity_from_sparse_forcing(const sb200_grid_t* gr, void* vorticity,
                                                          const void* velocity_forcing, double prefactor,
                                                          void* tile_flags, void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  SB_REQUIRE(vorticity && velocity_forcing && tile_flags, "update_vorticity_from_sparse_forcing: null pointer");
  SB_REQUIRE(g.vol / SB_CHUNK < (1LL << 30), "update_vorticity_from_sparse_forcing: field too large");
  const long long nchunks = sb_chunk_count(g);
  const SbChunkBuf b = sb_chunk_buf(tile_flags, nchunks);
  const unsigned grid = sb_chunk_grid(nchunks);
  SB_DISPATCH_DTYPE(gr->dtype, {
    SB_LAUNCH(sb_flag_nonzero_chunks_kernel<T>, dim3(grid), dim3(256), 0, stream, (const T*)velocity_forcing,
              g.dim, g.vol, nchunks, b);
  });
  SB_CHECK_LAUNCH("flag_nonzero_chunks");
  SB_LAUNCH(sb_dilate_chunks_kernel, dim3(148), dim3(256), 0, stream, g, nchunks, b);
  SB_CHECK_LAUNCH("dilate_chunks");
  SB_DISPATCH_DTYPE(gr->dtype, {
    SB_LAUNCH(sb_update_vorticity_flagged_kernel<T>, dim3(grid), dim3(256), 0, stream, g, (T*)vorticity,
              (const T*)velocity_forcing, (T)prefactor, b);
  });
  SB_CHECK_LAUNCH("update_vorticity_flagged");
  return 0;
}
extern "C" int sb200_clear_flagged_tiles(const sb200_grid_t* gr, void* field, int ncomp, void* tile_flags,
                                         void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  SB_REQUIRE(field && tile_flags && ncomp >= 1 && ncomp <= 3, "clear_flagged_tiles: bad arguments");
  const long long nchunks = sb_chunk_count(g);
  const SbChunkBuf b = sb_chunk_buf(tile_flags, nchunks);
  SB_DISPATCH_DTYPE(gr->dtype, {
    SB_LAUNCH(sb_clear_flagged_kernel<T>, dim3(sb_chunk_grid(nchunks)), dim3(256), 0, stream, (T*)field, ncomp,
              g.vol, b);
  });
  SB_CHECK_LAUNCH("clear_flagged_tiles");
  const int e = sb_memset_async(tile_flags, 0, sb_chunk_buf_bytes(nchunks), stream);
  if (e) {
    sb_set_error("memset: %s", sb_error_string(e));
    return -2;
  }
  return 0;
}

template <typename T>
struct CurlOp {
  T* c;
  const T* f;
  T p;
  SB_D void operator()(const SbGeom& g, int z, int y, int x) const {
    const long long i = g.idx(z, y, x);
    const bool ring = g.in_ring(z, y, x);
    const bool wr = g.written(z, y, x, 1, /*x_full=*/g.dim == 3);
    if (!ring && !wr) return;
    if (g.dim == 3) {
      T cx = 0, cy = 0, cz = 0;
      if (!ring) curl3_at(g, f, i, p, cx, cy, cz);
      c[i] = cx;
      c[i + g.vol] = cy;
      c[i + 2 * g.vol] = cz;
    } else {
      // outplane curl: psi (y,x) -> (u_x, u_y) = p * (dpsi/dy, -dpsi/dx)
      T ux = 0, uy = 0;
      if (!ring) {
        ux = p * (f[i + g.mx] - f[i - g.mx]);
        uy = -p * (f[i + 1] - f[i - 1]);
      }
      c[i] = ux;
      c[i + g.vol] = uy;
    }
  }
};

template <typename T>
struct DiffusionFluxOp {
  T* flux;
  const T* f;
  T p;
  SB_D void operator()(const SbGeom& g, int z, int y, int x) const {
    const long long i = g.idx(z, y, x);
    if (!g.deep(z, y, x)) {
      if (g.in_ring(z, y, x)) {
        flux[i] = 0;
        return;
      }
      if (!g.written(z, y, x, 1)) return;
    }
    T s = f[i + 1] + f[i - 1] + f[i + g.mx] + f[i - g.mx];
    if (g.dim == 3) {
      s += f[i + g.plane] + f[i - g.plane];
      flux[i] = p * (s - T(6) * f[i]);
    } else {
      flux[i] = p * (s - T(4) * f[i]);
    }
  }
};

template <typename T>
struct DivergenceOp {
  T* d;
  const T* f;
  T p;  // 0.5 * inv_dx
  SB_D void operator()(const SbGeom& g, int z, int y, int x) const {
    const long long i = g.idx(z, y, x);
    if (g.in_ring(z, y, x)) {
      d[i] = 0;
      return;
    }
    if (!g.written(z, y, x, 1)) return;
    const T* fx = f;
    const T* fy = f + g.vol;
    T s = fx[i + 1] - fx[i - 1] + fy[i + g.mx] - fy[i - g.mx];
    if (g.dim == 3) {
      const T* fz = f + 2 * g.vol;
      s += fz[i + g.plane] - fz[i - g.plane];
    }
    d[i] = p * s;
  }
};

// ENO3 upwinded flux difference along one axis (stride st) for cell i
template <typename T>
SB_D T eno3_axis(const T* q, const T* v, long long i, long long st) {
  const T half = T(0.5), sixth = T(1.0 / 6.0);
  const T qm2 = q[i - 2 * st], qm1 = q[i - st], q0 = q[i], qp1 = q[i + st], qp2 = q[i + 2 * st];
  const T vp = half * (v[i] + v[i + st]);
  const T vm = half * (v[i] + v[i - st]);
  const T fl_p = sixth * (-qm1 + T(5) * q0 + T(2) * qp1);
  const T fr_p = sixth * (T(2) * q0 + T(5) * qp1 - qp2);
  const T fl_m = sixth * (-qm2 + T(5) * qm1 + T(2) * q0);
  const T fr_m = sixth * (T(2) * qm1 + T(5) * q0 - qp1);
  const T zero = T(0);
  const T flux_p = (vp > zero ? vp : zero) * fl_p + (vp < zero ? vp : zero) * fr_p;
  const T flux_m = (vm > zero ? vm : zero) * fl_m + (vm < zero ? vm : zero) * fr_m;
  return flux_p - flux_m;
}

template <typename T>
struct AdvectionFluxOp {
  T* flux;
  const T* q;
  const T* vel;
  T inv_dx;
  SB_D void operator()(const SbGeom& g, int z, int y, int x) const {
    if (!g.written(z, y, x, 2)) return;
    const long long i = g.idx(z, y, x);
    T s = eno3_axis(q, vel, i, 1) + eno3_axis(q, vel + g.vol, i, (long long)g.mx);
    if (g.dim == 3) s += eno3_axis(q, vel + 2 * g.vol, i, g.plane);
    flux[i] = inv_dx * s;
  }
};

template <typename T>
struct FilterAxisOp {
  T* flux;
  const T* f;
  long long st;
  SB_D void operator()(const SbGeom& g, int z, int y, int x) const {
    const long long i = g.idx(z, y, x);
    // the wrapper clears the ring right after the seven calls
    if (g.in_ring(z, y, x)) {
      flux[i] = 0;
      return;
    }
    if (!g.written(z, y, x, 1)) return;
    flux[i] = T(0.25) * (-f[i + st] - f[i - st] + T(2) * f[i]);
  }
};

// One filter stage with the wrapper's bookkeeping folded in: the reference runs
// {seven-region filter, ring clear, field_buffer[...] = filter_flux} per stage, i.e. after a stage both
// arrays hold  ring ? 0 : written ? F(in) : (what the flux array held before),  and "before" equals the
// stage's own input for every stage but the first (where it is the stale flux array).  Writing that
// value out of place (ping-pong between the two arrays) saves the copy; the last stage also applies
// field -= flux (reference laplacian_filter_mpi_3d.py:267-385).
template <typename T>
struct FilterStageOp {
  T* out;
  const T* in;
  long long st;
  T* field;    // non-null on the last stage of a chain
  int first;   // first stage of a chain: `in` is the field, `out` the (stale) flux array
  SB_D void operator()(const SbGeom& g, int z, int y, int x) const {
    const long long i = g.idx(z, y, x);
    T v;
    if (g.deep(z, y, x) || (!g.in_ring(z, y, x) && g.written(z, y, x, 1)))  // (deep: the cheap common case)
      v = T(0.25) * (-in[i + st] - in[i - st] + T(2) * in[i]);
    else if (g.in_ring(z, y, x))
      v = 0;
    else
      v = first ? out[i] : in[i];
    out[i] = v;
    if (field) field[i] -= v;
  }
};

template <typename T>
struct ClearRingOp {
  T* f;
  int ncomp = 1, width = 1;
  SB_D void operator()(const SbGeom& g, int z, int y, int x) const {
    if (!g.in_ring(z, y, x, width)) return;
    const long long i = g.idx(z, y, x);
    for (int c = 0; c < ncomp; ++c) f[i + c * g.vol] = 0;
  }
};

extern "C" int sb200_update_vorticity_from_velocity_forcing(const sb200_grid_t* gr, void* vorticity,
                                                            const void* forcing, double prefactor,
                                                            void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  SB_REQUIRE(g.gs >= 1, "ghost_size < kernel_support");
  SB_DISPATCH_DTYPE(gr->dtype,
                    return sb_launch_cells(g, UpdateVorticityOp<T>{(T*)vorticity, (const T*)forcing,
                                                                   (T)prefactor},
                                           stream, "update_vorticity"));
}
extern "C" int sb200_curl(const sb200_grid_t* gr, void* curl, const void* field, double prefactor,
                          void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  SB_REQUIRE(g.gs >= 1, "ghost_size < kernel_support");
  SB_DISPATCH_DTYPE(gr->dtype, return sb_launch_cells(
                                   g, CurlOp<T>{(T*)curl, (const T*)field, (T)prefactor}, stream, "curl"));
}
extern "C" int sb200_diffusion_flux(const sb200_grid_t* gr, void* flux, const void* field, double prefactor,
                                    void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  SB_REQUIRE(g.gs >= 1, "ghost_size < kernel_support");
  SB_DISPATCH_DTYPE(gr->dtype,
                    return sb_launch_cells(g, DiffusionFluxOp<T>{(T*)flux, (const T*)field, (T)prefactor},
                                           stream, "diffusion_flux"));
}
extern "C" int sb200_diffusion_timestep(const sb200_grid_t* gr, void* field, int ncomp, void* flux,
                                        double nu_dt_by_dx2, void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  const size_t w = gr->dtype == SB200_F32 ? 4 : 8;
  for (int c = 0; c < ncomp; ++c) {
    char* fc = (char*)field + (size_t)c * g.vol * w;
    int e = sb200_diffusion_flux(gr, flux, fc, nu_dt_by_dx2, stream);
    if (e) return e;
    e = sb200_elementwise_sum(gr->dtype, fc, fc, flux, g.vol, stream);
    if (e) return e;
  }
  return 0;
}
extern "C" int sb200_advection_flux_eno3(const sb200_grid_t* gr, void* flux, const void* field,
                                         const void* velocity, double inv_dx, void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  SB_REQUIRE(g.gs >= 2, "ghost_size < kernel_support");
  SB_DISPATCH_DTYPE(gr->dtype, return sb_launch_cells(g,
                                                      AdvectionFluxOp<T>{(T*)flux, (const T*)field,
                                                                         (const T*)velocity, (T)inv_dx},
                                                      stream, "advection_flux"));
}
extern "C" int sb200_advection_timestep_eno3(const sb200_grid_t* gr, void* field, int ncomp, void* flux,
                                             const void* velocity, double dt_by_dx, void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  const size_t w = gr->dtype == SB200_F32 ? 4 : 8;
  for (int c = 0; c < ncomp; ++c) {
    char* fc = (char*)field + (size_t)c * g.vol * w;
    int e = sb200_set_fixed_val(gr->dtype, flux, g.vol, 0.0, stream);
    if (e) return e;
    e = sb200_advection_flux_eno3(gr, flux, fc, velocity, -dt_by_dx, stream);
    if (e) return e;
    e = sb200_elementwise_sum(gr->dtype, fc, fc, flux, g.vol, stream);
    if (e) return e;
  }
  return 0;
}
extern "C" int sb200_divergence(const sb200_grid_t* gr, void* divergence, const void* field, double inv_dx,
                                void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  SB_REQUIRE(g.gs >= 1, "ghost_size < kernel_support");
  SB_DISPATCH_DTYPE(gr->dtype, return sb_launch_cells(g,
                                                      DivergenceOp<T>{(T*)divergence, (const T*)field,
                                                                      (T)(0.5 * inv_dx)},
                                                      stream, "divergence"));
}

template <typename T>
static int laplacian_filter_scalar(const sb200_grid_t* gr, const SbGeom& g, T* field, int order, int type,
                                   T* flux, T* buf, void* stream) {
  int e;
  // array strides of the x, y, z filters
  const long long strides[3] = {1, (long long)g.mx, g.plane};
  const int naxes = g.dim;
  if ((e = sb_launch_cells(g, ClearRingOp<T>{flux}, stream, "filter_clear"))) return e;
  if (order == 0) {  // no stage runs: field -= (ring-cleared) flux, once (multiplicative) or per axis
    for (int a = 0; a < (type == 0 ? 1 : naxes); ++a)
      if ((e = sb200_elementwise_saxpby(gr->dtype, field, field, 1.0, flux, -1.0, g.vol, stream))) return e;
    return 0;
  }
  // a chain of stages ping-pongs flux -> buf -> flux ...; stage 0 reads the field itself
  auto chain = [&](int nstages, auto axis_of) -> int {
    const T* in = field;
    T* out = flux;
    for (int s = 0; s < nstages; ++s) {
      // the subtraction rides on the last stage unless that stage still reads the field's neighbours
      const bool fuse_sub = s == nstages - 1 && s > 0;
      if (int err = sb_launch_cells(g, FilterStageOp<T>{out, in, strides[axis_of(s)], fuse_sub ? field : nullptr,
                                                         s == 0},
                                    stream, "filter_stage"))
        return err;
      in = out;
      out = out == flux ? buf : flux;
    }
    if (nstages == 1)
      if (int err = sb200_elementwise_saxpby(gr->dtype, field, field, 1.0, flux, -1.0, g.vol, stream)) return err;
    // the reference leaves the last stage's flux in filter_flux_buffer (the stale values of the next
    // call's first stage): an even number of stages ended in `buf`
    if (in != flux) return sb200_elementwise_copy(gr->dtype, flux, buf, g.vol, stream);
    return 0;
  };
  if (type == 0) return chain(order * naxes, [&](int s) { return s % naxes; });
  for (int a = 0; a < naxes; ++a)
    if ((e = chain(order, [&](int) { return a; }))) return e;
  return 0;
}

extern "C" int sb200_laplacian_filter_stage(const sb200_grid_t* gr, void* out, const void* in, int axis,
                                            void* field, int first, void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  SB_REQUIRE(g.gs >= 1, "ghost_size < kernel_support");
  SB_REQUIRE(axis >= 0 && axis < g.dim && out && in && out != in, "filter_stage: bad arguments");
  const long long strides[3] = {1, (long long)g.mx, g.plane};
  SB_DISPATCH_DTYPE(gr->dtype, return sb_launch_cells(g,
                                                      FilterStageOp<T>{(T*)out, (const T*)in, strides[axis],
                                                                       (T*)field, first},
                                                      stream, "filter_stage"));
}
extern "C" int sb200_laplacian_filter_axis(const sb200_grid_t* gr, void* flux, const void* buf, int axis,
                                           void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  SB_REQUIRE(g.gs >= 1, "ghost_size < kernel_support");
  SB_REQUIRE(axis >= 0 && axis < g.dim, "bad filter axis");
  const long long strides[3] = {1, (long long)g.mx, g.plane};
  SB_DISPATCH_DTYPE(gr->dtype, return sb_launch_cells(
                                   g, FilterAxisOp<T>{(T*)flux, (const T*)buf, strides[axis]}, stream,
                                   "filter_axis"));
}
extern "C" int sb200_clear_physical_ring(const sb200_grid_t* gr, void* field, int ncomp, int width,
                                         void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  SB_DISPATCH_DTYPE(gr->dtype, return sb_launch_cells(g, ClearRingOp<T>{(T*)field, ncomp, width}, stream,
                                                      "clear_ring"));
}

// ---- order-1 multiplicative filter in ONE pass (the setting of the rod examples,
// examples/3d_examples/FlowPastRodCase/flow_past_rod_case.py:114-115) on a rank whose six faces are all
// physical.  There every cell is either "deep" (written by each stage's interior call and outside
// the zeroed ring) or in the ring, so the chain of FilterStageOp collapses to
//     a = deep ? Fx(f) : 0,  b = deep ? Fy(a) : 0,  c = deep ? Fz(b) : 0,  f -= c
// with F the 1D kernel 0.25 (-in(+1) - in(-1) + 2 in) (laplacian_filter_mpi_3d.py:62-99,267-319): 2 W per
// cell and component instead of 8 W + a copy.  OUT OF PLACE (a block reads a halo of cells that belong to
// its neighbours): the simulator alternates between its two vorticity allocations.  The last component
// also leaves the reference's buffer contents behind (filter_flux_buffer = field_buffer = c).
// The filter is a z MARCH: a block owns an 8 x 32 (y, x) tile and walks along z.  The x and y stages are
// in-plane, so per plane it stages the tile + 1 halo cell (10 x 34) in shared memory, forms a = Fx(f) on
// 10 x 32 and b = Fy(a) for the thread's own cell; the z stage only needs b at the SAME (y, x) one plane up
// and down, which the thread carries in registers together with f of the previous plane.  Every plane is
// read once (+ the in-plane halo, served by L2), with no index arithmetic inside the march; the next plane
// is prefetched into registers.  The expressions and their order are those of the stage chain, so the
// results are bit-identical to it.
template <typename T>
__global__ void __launch_bounds__(256)
    sb_filter_o1_mult_march_kernel(SbGeom g, T* __restrict__ out, const T* __restrict__ field, int ncomp,
                                   T* __restrict__ flux, T* __restrict__ buf, int zchunk) {
  constexpr int TX = 32, TY = 8, FX = TX + 2, FY = TY + 2;
  __shared__ T sf[FY * FX];
  __shared__ T sa[FY * TX];
  const int tid = threadIdx.x, lx = tid & 31, ly = tid >> 5;
  const int x0 = blockIdx.x * TX, y0 = blockIdx.y * TY;
  const int nzc = (g.mz + zchunk - 1) / zchunk;
  const int c = blockIdx.z / nzc, zb = (blockIdx.z - c * nzc) * zchunk;
  const int ze = zb + zchunk < g.mz ? zb + zchunk : g.mz;
  const T* f = field + (long long)c * g.vol;
  T* o = out + (long long)c * g.vol;
  const bool last = c == ncomp - 1;
  // the (up to two) cells of the staged plane this thread loads: element e of the FY x FX frame
  long long off[2];
  bool have[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int e = tid + k * 256, fy = e / FX, fx = e - fy * FX;
    const int x = x0 + fx - 1, y = y0 + fy - 1;
    have[k] = e < FY * FX && x >= 0 && x < g.mx && y >= 0 && y < g.my;
    off[k] = have[k] ? (long long)y * g.mx + x : 0;
  }
  // the (up to two) cells of a = Fx(f) this thread forms: rows y0 - 1 .. y0 + 8, columns x0 .. x0 + 31
  bool adeep[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int e = tid + k * 256, ay = e / TX, ax = e - ay * TX;
    const int x = x0 + ax, y = y0 + ay - 1;
    adeep[k] = e < FY * TX && x < g.mx && y >= 0 && y < g.my && (unsigned)(x - g.gs - 1) < (unsigned)(g.mx - 2 * g.gs - 2) &&
               (unsigned)(y - g.gs - 1) < (unsigned)(g.my - 2 * g.gs - 2);
  }
  const int x = x0 + lx, y = y0 + ly;
  const bool mine = x < g.mx && y < g.my;
  const bool deep_yx = mine && (unsigned)(x - g.gs - 1) < (unsigned)(g.mx - 2 * g.gs - 2) &&
                       (unsigned)(y - g.gs - 1) < (unsigned)(g.my - 2 * g.gs - 2);
  const long long cell = (long long)y * g.mx + x;
  auto deep_z = [&](int z) { return (unsigned)(z - g.gs - 1) < (unsigned)(g.mz - 2 * g.gs - 2); };
  auto fetch = [&](int z, T (&r)[2]) {
    const bool zin = z >= 0 && z < g.mz;
#pragma unroll
    for (int k = 0; k < 2; ++k) r[k] = (zin && have[k]) ? f[(long long)z * g.plane + off[k]] : T(0);
  };
  T nf[2];
  fetch(zb - 1, nf);
  T b_lo = T(0), b_mid = T(0), f_mid = T(0);  // b at z - 2 and z - 1, f at z - 1 (own cell)
  for (int z = zb - 1; z <= ze; ++z) {
    sf[tid] = nf[0];
    if (tid + 256 < FY * FX) sf[tid + 256] = nf[1];
    __syncthreads();
    if (z < ze) fetch(z + 1, nf);  // the next plane is in flight while this one is processed
    const bool dz = z >= 0 && z < g.mz && deep_z(z);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int e = tid + k * 256;
      if (e < FY * TX) {
        const int ay = e / TX, ax = e - ay * TX;
        const T* q = sf + ay * FX + ax + 1;
        sa[e] = (dz && adeep[k]) ? T(0.25) * (-q[1] - q[-1] + T(2) * q[0]) : T(0);
      }
    }
    const T f_hi = sf[(ly + 1) * FX + lx + 1];  // (before the barrier: the next plane overwrites sf behind it)
    __syncthreads();
    const T* q = sa + (ly + 1) * TX + lx;
    const T b_hi = (dz && deep_yx) ? T(0.25) * (-q[TX] - q[-TX] + T(2) * q[0]) : T(0);
    // plane z - 1 is complete: b on both sides of it is known
    const int zo = z - 1;
    if (zo >= zb && zo < ze && mine) {
      const T cz = (deep_z(zo) && deep_yx) ? T(0.25) * (-b_hi - b_lo + T(2) * b_mid) : T(0);
      const long long gi = (long long)zo * g.plane + cell;
      o[gi] = f_mid - cz;
      if (last) {  // (the reference copies the flux into field_buffer after every stage)
        flux[gi] = cz;
        buf[gi] = cz;
      }
    }
    b_lo = b_mid;
    b_mid = b_hi;
    f_mid = f_hi;
  }
}

template <typename T>
static int launch_filter_o1_mult(const SbGeom& g, void* out, const void* field, int ncomp, void* flux, void* buf,
                                 void* stream) {
  // z chunks: enough blocks for ~8 waves of the 148 x 8 resident blocks, at least 16 planes per chunk
  const long long tiles = (long long)((g.mx + 31) / 32) * ((g.my + 7) / 8) * ncomp;
  int nzc = (int)((148LL * 8 * 8 + tiles - 1) / tiles);
  if (nzc < 1) nzc = 1;
  int zchunk = (g.mz + nzc - 1) / nzc;
  if (zchunk < 16) zchunk = g.mz < 16 ? g.mz : 16;
  nzc = (g.mz + zchunk - 1) / zchunk;
  const dim3 grid((unsigned)((g.mx + 31) / 32), (unsigned)((g.my + 7) / 8), (unsigned)(nzc * ncomp));
  SB_LAUNCH_COOP(sb_filter_o1_mult_march_kernel<T>, grid, dim3(256), 0, stream, g, (T*)out, (const T*)field, ncomp,
                 (T*)flux, (T*)buf, zchunk);
  SB_CHECK_LAUNCH("filter_o1_mult_march");
  return 0;
}

extern "C" int sb200_laplacian_filter_order1_out_of_place(const sb200_grid_t* gr, void* out, const void* field,
                                                          int ncomp, void* flux, void* buf, void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  SB_REQUIRE(g.dim == 3 && g.gs >= 1 && ncomp >= 1 && ncomp <= 3, "filter_order1: 3D fields, ghost_size >= 1");
  for (int k = 0; k < 6; ++k) SB_REQUIRE(g.phys[k], "filter_order1: every face of the block must be physical");
  SB_REQUIRE(out && field && flux && buf && out != field, "filter_order1: bad pointers (out of place)");
  SB_DISPATCH_DTYPE(gr->dtype, return launch_filter_o1_mult<T>(g, out, field, ncomp, flux, buf, stream));
}

extern "C" int sb200_laplacian_filter(const sb200_grid_t* gr, void* field, int ncomp, int filter_order,
                                      int filter_type, void* flux, void* buf, void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  SB_REQUIRE(g.gs >= 1, "ghost_size < kernel_support");
  SB_REQUIRE(filter_order >= 0 && (filter_type == 0 || filter_type == 1), "invalid filter setting");
  for (int c = 0; c < ncomp; ++c) {
    int e = 0;
    SB_DISPATCH_DTYPE(gr->dtype, e = laplacian_filter_scalar<T>(gr, g, (T*)field + (size_t)c * g.vol,
                                                                 filter_order, filter_type, (T*)flux,
                                                                 (T*)buf, stream));
    if (e) return e;
  }
  return 0;
}

// ---- operators of the reference API that no simulator path uses (SURVEY 8(f)4): Brinkmann
// penalisation, characteristic function of a level set, vorticity update from a penalised velocity
// (stencil_ops_3d/brinkmann_penalise_mpi_3d.py:7, char_func_from_level_set_mpi_3d.py:8,
// update_vorticity_from_velocity_forcing_mpi_3d.py:181-330).  The arithmetic lives in the un-vendored
// `sopht` package; the published forms are restated (PARITY UNPINNED).
template <typename T>
struct BrinkmannOp {
  T* out;
  const T* chi;
  const T* target;
  const T* f;
  T lambda;
  long long n;
  int ncomp;
  SB_D void operator()(long long i) const {
    const T c = lambda * chi[i];
    for (int k = 0; k < ncomp; ++k)
      out[i + k * n] = (f[i + k * n] + c * target[i + k * n]) / (T(1) + c);
  }
};
template <typename T>
struct SineHeavisideOp {
  T* chi;
  const T* ls;
  T bw;
  SB_D void operator()(long long i) const {
    const T v = ls[i];
    T r;
    if (v > bw)
      r = T(1);
    else if (v < -bw)
      r = T(0);
    else
      r = T(0.5) * (T(1) + v / bw + sin(T(M_PI) * v / bw) / T(M_PI));
    chi[i] = r;
  }
};
template <typename T>
struct UpdateVorticityPenalisedOp {
  T* w;
  const T* up;
  const T* u;
  T p;
  SB_D T d(int c, long long i, const SbGeom& g) const { return up[i + c * g.vol] - u[i + c * g.vol]; }
  SB_D void operator()(const SbGeom& g, int z, int y, int x) const {
    if (!g.deep(z, y, x) && !g.written(z, y, x, 1)) return;
    const long long i = g.idx(z, y, x), sy = g.mx, sz = g.plane;
    w[i] += p * (d(2, i + sy, g) - d(2, i - sy, g) - d(1, i + sz, g) + d(1, i - sz, g));
    w[i + g.vol] += p * (d(0, i + sz, g) - d(0, i - sz, g) - d(2, i + 1, g) + d(2, i - 1, g));
    w[i + 2 * g.vol] += p * (d(1, i + 1, g) - d(1, i - 1, g) - d(0, i + sy, g) + d(0, i - sy, g));
  }
};
extern "C" int sb200_brinkmann_penalise(int dtype, void* penalised, double penalty_factor, const void* char_func,
                                        const void* penalty_field, const void* field, int ncomp, int64_t count,
                                        void* stream) {
  SB_REQUIRE(penalised && char_func && penalty_field && field && ncomp >= 1 && ncomp <= 3,
             "brinkmann_penalise: bad arguments");
  SB_DISPATCH_DTYPE(dtype, return sb_launch_flat(count,
                                                 BrinkmannOp<T>{(T*)penalised, (const T*)char_func,
                                                                (const T*)penalty_field, (const T*)field,
                                                                (T)penalty_factor, count, ncomp},
                                                 stream, "brinkmann_penalise"));
}
extern "C" int sb200_char_func_from_level_set(int dtype, void* char_func, const void* level_set, double blend_width,
                                              int64_t count, void* stream) {
  SB_REQUIRE(char_func && level_set && blend_width > 0, "char_func_from_level_set: bad arguments");
  SB_DISPATCH_DTYPE(dtype, return sb_launch_flat(count,
                                                 SineHeavisideOp<T>{(T*)char_func, (const T*)level_set,
                                                                    (T)blend_width},
                                                 stream, "char_func_from_level_set"));
}
extern "C" int sb200_update_vorticity_from_penalised_velocity(const sb200_grid_t* gr, void* vorticity,
                                                              const void* penalised_velocity, const void* velocity,
                                                              double prefactor, void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  SB_REQUIRE(g.dim == 3 && g.gs >= 1, "update_vorticity_from_penalised_velocity: 3D, ghost_size >= 1");
  SB_DISPATCH_DTYPE(gr->dtype,
                    return sb_launch_cells(g,
                                           UpdateVorticityPenalisedOp<T>{(T*)vorticity, (const T*)penalised_velocity,
                                                                         (const T*)velocity, (T)prefactor},
                                           stream, "update_vorticity_penalised"));
}

// ------------------------------------------------------------- penalise ----
// Sequential reference semantics (X front/back, then Y, then Z; copy the plane
// gs+w-1 outwards, then multiply by the sine factor) collapse to
//   f[z,y,x] = ((f[cz,cy,cx] * sx) * sy) * sz
// with c* = index clamped into [gs+w-1, m-gs-w] along physical axes.
// Phase 0 writes every zone cell that is not itself a source cell; phase 1 then
// scales the source cells lying on the clamp planes.
template <typename T>
struct PenaliseOp {
  T* f;
  const T* fac;  // [2*dim][gs+w], order z_front,z_back,y_front,y_back,x_front,x_back (2D: y.., x..)
  int w;         // gs + width
  int phase;
  int ncomp;
  // returns true when index i lies in a physical penalty slab of this axis
  SB_D bool axis(int i, int m, int pf, int pb, int tab, int& ci, T& s, bool& moved) const {
    ci = i;
    s = T(1);
    if (pf && i < w) {
      ci = w - 1;
      s = fac[tab * w + i];
      moved = moved || (i != w - 1);
      return true;
    }
    if (pb && i >= m - w) {
      ci = m - w;
      s = fac[(tab + 1) * w + (i - (m - w))];
      moved = moved || (i != m - w);
      return true;
    }
    return false;
  }
  SB_D void operator()(const SbGeom& g, int z, int y, int x) const {
    int cz = z, cy, cx;
    T sz = T(1), sy, sx;
    bool moved = false;
    const int t0 = g.dim == 3 ? 2 : 0;
    const bool inx = axis(x, g.mx, g.phys[4], g.phys[5], t0 + 2, cx, sx, moved);
    const bool iny = axis(y, g.my, g.phys[2], g.phys[3], t0, cy, sy, moved);
    bool inz = false;
    if (g.dim == 3) inz = axis(z, g.mz, g.phys[0], g.phys[1], 0, cz, sz, moved);
    if (!(inx || iny || inz)) return;
    if ((phase == 0) != moved) return;
    const long long src = g.idx(cz, cy, cx), dst = g.idx(z, y, x);
    for (int c = 0; c < ncomp; ++c) {  // all components in one launch
      T v = f[c * g.vol + src];
      // multiply by the factors of the slabs this cell belongs to, in X,Y,Z order
      if (inx) v = v * sx;
      if (iny) v = v * sy;
      if (inz) v = v * sz;
      f[c * g.vol + dst] = v;
    }
  }
};

extern "C" int sb200_penalise_field_boundary(const sb200_grid_t* gr, void* field, int ncomp, int width,
                                             const void* factors, void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  SB_REQUIRE(width >= 0, "invalid zone width");
  if (width == 0) return 0;
  const int w = g.gs + width;
  SB_REQUIRE(g.mx >= 2 * w && g.my >= 2 * w && (g.dim == 2 || g.mz >= 2 * w), "penalty zones overlap");
  // the penalty zone as disjoint boxes: x slabs (all z,y), y slabs (x in the middle),
  // z slabs (y,x in the middle)
  SbBoxes b;
  b.n = 0;
  auto add = [&](int z0, int z1, int y0, int y1, int x0, int x1) {
    const int lo[3] = {z0, y0, x0}, hi[3] = {z1, y1, x1};
    for (int d = 0; d < 3; ++d) {
      b.lo[b.n][d] = lo[d];
      b.hi[b.n][d] = hi[d];
    }
    ++b.n;
  };
  const int xl = g.phys[4] ? w : 0, xh = g.phys[5] ? g.mx - w : g.mx;
  const int yl = g.phys[2] ? w : 0, yh = g.phys[3] ? g.my - w : g.my;
  if (g.phys[4]) add(0, g.mz, 0, g.my, 0, w);
  if (g.phys[5]) add(0, g.mz, 0, g.my, g.mx - w, g.mx);
  if (g.phys[2]) add(0, g.mz, 0, w, xl, xh);
  if (g.phys[3]) add(0, g.mz, g.my - w, g.my, xl, xh);
  if (g.dim == 3 && g.phys[0]) add(0, w, yl, yh, xl, xh);
  if (g.dim == 3 && g.phys[1]) add(g.mz - w, g.mz, yl, yh, xl, xh);
  for (int phase = 0; phase < 2; ++phase) {
    int e = 0;
    SB_DISPATCH_DTYPE(gr->dtype,
                      e = sb_launch_boxes(g, b, PenaliseOp<T>{(T*)field, (const T*)factors, w, phase, ncomp},
                                          stream, "penalise"));
    if (e) return e;
  }
  return 0;
}
