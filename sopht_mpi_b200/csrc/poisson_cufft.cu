// Unbounded (Hockney-Eastwood) Poisson solve, generic backend: fused
// pad / Green's-multiply / crop kernels around cuFFT R2C/C2R on the doubled domain, and a z-slab
// mode for distributed solves of any grid size (below).
// Reference: numeric/eulerian_grid_ops/poisson_solver_3d/UnboundedPoissonSolverMPI3D.py:22-187,
// fft_mpi_3d.py:34-48 and the 2D twins.  Used for arbitrary grid sizes; the
// power-of-two hot path lives in poisson_fft.cu (backend 1).
#include "sb200_common.h"
#include "poisson.h"

#ifndef SB200_EMU
#include <cufft.h>

#include "fft_device.h"

#define SB_CUFFT(call, what)                                  \
  do {                                                        \
    cufftResult r__ = (call);                                 \
    if (r__ != CUFFT_SUCCESS) {                               \
      sb_set_error("cufft %s failed: %d", what, (int)r__);    \
      return -3;                                              \
    }                                                         \
  } while (0)
#define SB_CUDA(call, what)                                                     \
  do {                                                                          \
    cudaError_t e__ = (call);                                                   \
    if (e__ != cudaSuccess) {                                                   \
      sb_set_error("%s: %s", what, cudaGetErrorString(e__));                    \
      return -2;                                                                \
    }                                                                           \
  } while (0)

struct SbCufftState {
  cufftHandle fwd = 0, inv = 0;
  void* real_buf = nullptr;   // (2nz,2ny,2nx) reals
  void* spec_buf = nullptr;   // (2nz,2ny,nx+1) complex
  void* ghat = nullptr;       // (2nz,2ny,nx+1) reals: Re(rfftn(G)) * dx^dim / prod(2n)
  size_t bytes = 0;
};

// rhs interior -> top-left corner of the (pre-zeroed) doubled buffer
template <typename T>
struct PadCopyOp {
  T* dst;
  const T* src;
  int nz, ny, nx, gs, dim;
  long long s_my, s_mx;  // padded source sizes
  SB_D void operator()(long long i) const {
    const int x = (int)(i % nx);
    const long long r = i / nx;
    const int y = (int)(r % ny), z = (int)(r / ny);
    const long long si = dim == 3 ? ((long long)(z + gs) * s_my + (y + gs)) * s_mx + (x + gs)
                                  : (long long)(y + gs) * s_mx + (x + gs);
    dst[((long long)z * 2 * ny + y) * 2 * nx + x] = src[si];
  }
};
template <typename T>
struct CropCopyOp {
  T* dst;
  const T* src;
  int nz, ny, nx, gs, dim;
  long long s_my, s_mx;
  SB_D void operator()(long long i) const {
    const int x = (int)(i % nx);
    const long long r = i / nx;
    const int y = (int)(r % ny), z = (int)(r / ny);
    const long long di = dim == 3 ? ((long long)(z + gs) * s_my + (y + gs)) * s_mx + (x + gs)
                                  : (long long)(y + gs) * s_mx + (x + gs);
    dst[di] = src[((long long)z * 2 * ny + y) * 2 * nx + x];
  }
};
template <typename T>
struct SpecMulOp {
  T* spec;  // interleaved complex
  const T* g;
  SB_D void operator()(long long i) const {
    const T s = g[i];
    spec[2 * i] *= s;
    spec[2 * i + 1] *= s;
  }
};
template <typename T>
struct GhatFromSpecOp {
  T* g;
  const T* spec;
  T scale;
  SB_D void operator()(long long i) const { g[i] = spec[2 * i] * scale; }
};

// rfftn of the Green's function on the doubled grid: G -> real_buf -> spec_buf through `fwd`, the 2D / 3D R2C
// plan of the doubled grid.  The single-rank solve keeps buffers and plan; the z-slab set-up frees them.
static int cufft_greens_spectrum(sb200_poisson* p, cufftHandle fwd, void* real_buf, void* spec_buf, void* stream) {
  SB_CUFFT(cufftSetStream(fwd, (cudaStream_t)stream), "set stream");
  int e = sb_poisson_fill_greens(p, real_buf, stream);
  if (e) return e;
  if (p->dtype == SB200_F32)
    SB_CUFFT(cufftExecR2C(fwd, (cufftReal*)real_buf, (cufftComplex*)spec_buf), "R2C(G)");
  else
    SB_CUFFT(cufftExecD2Z(fwd, (cufftDoubleReal*)real_buf, (cufftDoubleComplex*)spec_buf), "D2Z(G)");
  return 0;
}

static double cufft_greens_scale(const sb200_poisson* p) {
  const double n2z = p->dim == 3 ? 2.0 * p->nz : 1.0;
  double dxp = 1.0;
  for (int d = 0; d < p->dim; ++d) dxp *= p->dx;
  return dxp / (n2z * 2.0 * p->ny * 2.0 * p->nx);
}

static int cufft_slab_create(sb200_poisson* p, void* stream);

int sb_poisson_cufft_create(sb200_poisson* p, void* stream) {
  if (p->nranks > 1) return cufft_slab_create(p, stream);
  auto* st = new SbCufftState();
  p->backend_state = st;
  const long long n2z = p->dim == 3 ? 2LL * p->nz : 1, n2y = 2LL * p->ny, n2x = 2LL * p->nx;
  const long long nreal = n2z * n2y * n2x, nspec = n2z * n2y * (p->nx + 1);
  const size_t w = p->dtype == SB200_F32 ? 4 : 8;
  SB_CUDA(cudaMalloc(&st->real_buf, nreal * w), "poisson real buffer");
  SB_CUDA(cudaMalloc(&st->spec_buf, nspec * 2 * w), "poisson spectral buffer");
  SB_CUDA(cudaMalloc(&st->ghat, nspec * w), "poisson greens buffer");
  st->bytes = nreal * w + nspec * 3 * w;
  const cufftType ft = p->dtype == SB200_F32 ? CUFFT_R2C : CUFFT_D2Z;
  const cufftType it = p->dtype == SB200_F32 ? CUFFT_C2R : CUFFT_Z2D;
  if (p->dim == 3) {
    SB_CUFFT(cufftPlan3d(&st->fwd, (int)n2z, (int)n2y, (int)n2x, ft), "plan3d fwd");
    SB_CUFFT(cufftPlan3d(&st->inv, (int)n2z, (int)n2y, (int)n2x, it), "plan3d inv");
  } else {
    SB_CUFFT(cufftPlan2d(&st->fwd, (int)n2y, (int)n2x, ft), "plan2d fwd");
    SB_CUFFT(cufftPlan2d(&st->inv, (int)n2y, (int)n2x, it), "plan2d inv");
  }
  // Green's function on the doubled grid -> spectrum -> real scaled table
  int e = cufft_greens_spectrum(p, st->fwd, st->real_buf, st->spec_buf, stream);
  if (e) return e;
  const double scale = cufft_greens_scale(p);
  SB_DISPATCH_DTYPE(p->dtype, e = sb_launch_flat(nspec,
                                                 GhatFromSpecOp<T>{(T*)st->ghat, (const T*)st->spec_buf,
                                                                   (T)scale},
                                                 stream, "ghat"));
  if (e) return e;
  SB_CUDA(cudaStreamSynchronize((cudaStream_t)stream), "poisson create sync");
  return 0;
}

static void cufft_slab_destroy(sb200_poisson* p);

int sb_poisson_cufft_destroy(sb200_poisson* p) {
  if (p->nranks > 1) {
    cufft_slab_destroy(p);
    return 0;
  }
  auto* st = (SbCufftState*)p->backend_state;
  if (!st) return 0;
  if (st->fwd) cufftDestroy(st->fwd);
  if (st->inv) cufftDestroy(st->inv);
  cudaFree(st->real_buf);
  cudaFree(st->spec_buf);
  cudaFree(st->ghat);
  delete st;
  p->backend_state = nullptr;
  return 0;
}

static int64_t cufft_slab_bytes(const sb200_poisson* p);

int64_t sb_poisson_cufft_bytes(const sb200_poisson* p) {
  if (p->nranks > 1) return cufft_slab_bytes(p);
  auto* st = (SbCufftState*)p->backend_state;
  return st ? (int64_t)st->bytes : 0;
}

int sb_poisson_cufft_solve(sb200_poisson* p, void* solution, const void* rhs, int ncomp, void* stream) {
  auto* st = (SbCufftState*)p->backend_state;
  const long long nzz = p->dim == 3 ? p->nz : 1;
  const long long n2z = p->dim == 3 ? 2LL * p->nz : 1, n2y = 2LL * p->ny, n2x = 2LL * p->nx;
  const long long nreal = n2z * n2y * n2x, nspec = n2z * n2y * (p->nx + 1);
  const long long nint = nzz * p->ny * p->nx;
  const size_t w = p->dtype == SB200_F32 ? 4 : 8;
  const long long smy = p->ny + 2 * p->gs, smx = p->nx + 2 * p->gs;
  const long long svol = (p->dim == 3 ? (p->nz + 2LL * p->gs) : 1) * smy * smx;
  SB_CUFFT(cufftSetStream(st->fwd, (cudaStream_t)stream), "set stream");
  SB_CUFFT(cufftSetStream(st->inv, (cudaStream_t)stream), "set stream");
  for (int c = 0; c < ncomp; ++c) {
    const char* rc = (const char*)rhs + (size_t)c * svol * w;
    char* sc = (char*)solution + (size_t)c * svol * w;
    int e = sb_memset_async(st->real_buf, 0, nreal * w, stream);
    SB_REQUIRE(e == 0, "poisson memset failed");
    SB_DISPATCH_DTYPE(p->dtype, e = sb_launch_flat(nint,
                                                   PadCopyOp<T>{(T*)st->real_buf, (const T*)rc, p->nz,
                                                                p->ny, p->nx, p->gs, p->dim, smy, smx},
                                                   stream, "pad_copy"));
    if (e) return e;
    if (p->dtype == SB200_F32)
      SB_CUFFT(cufftExecR2C(st->fwd, (cufftReal*)st->real_buf, (cufftComplex*)st->spec_buf), "R2C");
    else
      SB_CUFFT(cufftExecD2Z(st->fwd, (cufftDoubleReal*)st->real_buf, (cufftDoubleComplex*)st->spec_buf),
               "D2Z");
    SB_DISPATCH_DTYPE(p->dtype,
                      e = sb_launch_flat(nspec, SpecMulOp<T>{(T*)st->spec_buf, (const T*)st->ghat}, stream,
                                         "spec_mul"));
    if (e) return e;
    if (p->dtype == SB200_F32)
      SB_CUFFT(cufftExecC2R(st->inv, (cufftComplex*)st->spec_buf, (cufftReal*)st->real_buf), "C2R");
    else
      SB_CUFFT(cufftExecZ2D(st->inv, (cufftDoubleComplex*)st->spec_buf, (cufftDoubleReal*)st->real_buf),
               "Z2D");
    SB_DISPATCH_DTYPE(p->dtype, e = sb_launch_flat(nint,
                                                   CropCopyOp<T>{(T*)sc, (const T*)st->real_buf, p->nz,
                                                                 p->ny, p->nx, p->gs, p->dim, smy, smx},
                                                   stream, "crop_copy"));
    if (e) return e;
  }
  return 0;
}

// ------------------------------------------------------------------ z-slab mode (nranks > 1, 3D)
// The three stages of poisson_fft.cu's z-slab pipeline on cuFFT, for grids of any size, with the same
// exchange format (SbRowBlocks).  Rank r of P holds planes [r nz/P, (r+1) nz/P) and, between the two
// all-to-alls, kx bins [r kxl, (r+1) kxl) of all planes.  Per component:
//   forward : pad the local rows to 2nx (Xr: its upper halves are never written, so they stay zero),
//             batched R2C, pack the nx+1 bins into the send blocks          S[kxb][c][zl][y][kx_in]
//   spectral: the (2nz, 2ny) zero-padded convolution of each kx line, without the padding: with
//             kz = 2 mz + sz and ky = 2 my + sy, the doubled transform of a (nz, ny) block x is
//               X[kz][ky] = FFT_{nz,ny}( x[z][y] e^{-i pi (sz z / nz + sy y / ny)} )[mz][my]
//             and the kept quarter of the inverse is
//               x'[z][y] = sum_{sz,sy} e^{+i pi (sz z / nz + sy y / ny)} IFFT_{nz,ny}(X_{sz,sy})[z][y]
//             so four twiddled copies of the block go through one batched (nz, ny) C2C transform,
//             are scaled by the real Green's spectrum and come back; nothing is zero-padded and the
//             work buffer is exactly the rank's kx slab of the doubled plane      W[s][kx_in][z][y]
//   backward: unpack the returned blocks, batched C2R of length 2nx, keep the first nx values.
// The Green's table holds the rank's kx columns folded by the even symmetry in ky and kz,
// g[kx_in][min(kz, 2nz - kz)][min(ky, 2ny - ky)], zero for kx > nx (padding bins, or a rank whose block
// holds no bin at all), with dx^3 / (8 nx ny nz) folded in.
struct SbCufftSlabState {
  cufftHandle xf = 0, xi = 0, yz = 0;  // x R2C and C2R (nz/P * ny rows of 2nx), (nz, ny) C2C batch 4 kxl
  void* fft_area = nullptr;            // one work area for the three plans (they run one after another)
  void* xr = nullptr;    // [nz/P][ny][2nx] reals, the forward x input
  void* work = nullptr;  // W; the x passes use it for their complex rows Xc and the C2R output Xo
  size_t xo_off = 0;     // byte offset of Xo in work
  void* g = nullptr;     // [kxl][nz+1][ny+1] reals
  void* twz = nullptr;   // e^{-i pi z / nz}, z < nz
  void* twy = nullptr;   // e^{-i pi y / ny}, y < ny
  size_t bytes = 0;
};

template <typename T>
struct SlabPadOp {  // field interior rows of the local planes -> first nx reals of the rows of Xr
  T* dst;
  const T* src;
  int ny, nx, gs;
  long long s_my, s_mx;
  SB_D void operator()(long long i) const {
    const int x = (int)(i % nx);
    const long long r = i / nx;
    const int y = (int)(r % ny), z = (int)(r / ny);
    dst[r * 2 * nx + x] = src[((long long)(z + gs) * s_my + (y + gs)) * s_mx + (x + gs)];
  }
};
template <typename T>
struct SlabCropOp {  // first nx reals of the rows of Xo -> field interior rows
  T* dst;
  const T* src;
  int ny, nx, gs;
  long long s_my, s_mx;
  SB_D void operator()(long long i) const {
    const int x = (int)(i % nx);
    const long long r = i / nx;
    const int y = (int)(r % ny), z = (int)(r / ny);
    dst[((long long)(z + gs) * s_my + (y + gs)) * s_mx + (x + gs)] = src[r * 2 * nx + x];
  }
};
// Xc rows (nx + 1 bins) <-> rows of component c in the blocked exchange buffer
template <typename T, bool PACK>
struct SlabBlocksOp {
  C2<T>* xc;
  C2<T>* blocks;
  SbRowBlocks rb;
  long long line0;  // first row of component c in the exchange buffer
  int nb;           // nx + 1
  SB_D void operator()(long long i) const {
    const int k = (int)(i % nb);
    const long long line = i / nb;
    C2<T>* b = blocks + rb.row(line0 + line, 0) + rb.rel(k);
    if (PACK) *b = xc[i]; else xc[i] = *b;
  }
};
// R[zb][c][zl][y][kx_in] of component c -> the four twiddled copies W[s][kx_in][z][y], s = 2 sz + sy
template <typename T>
struct SlabSpreadOp {
  C2<T>* w;
  const C2<T>* r;
  const C2<T>*twz, *twy;
  SbRowBlocks rb;
  long long line0;
  int nz, ny, nzl;
  long long q;  // kxl nz ny
  SB_D void operator()(long long i) const {
    const int y = (int)(i % ny);
    const long long t = i / ny;
    const int z = (int)(t % nz), kx = (int)(t / nz);
    const int zb = z / nzl, zl = z - zb * nzl;
    const C2<T> v = r[rb.row(line0 + (long long)zl * ny + y, 0) + rb.rel(zb * rb.kxl + kx)];
    const C2<T> a = twz[z], b = twy[y];
    w[i] = v;
    w[q + i] = cmul(v, b);
    w[2 * q + i] = cmul(v, a);
    w[3 * q + i] = cmul(v, cmul(a, b));
  }
};
template <typename T>
struct SlabGreensMulOp {
  C2<T>* w;
  const T* g;
  int nz, ny, kxl;
  long long q;
  SB_D void operator()(long long i) const {
    const int s = (int)(i / q);
    const long long j = i - s * q;
    const int my = (int)(j % ny);
    const long long t = j / ny;
    const int mz = (int)(t % nz), kx = (int)(t / nz);
    const int ky = 2 * my + (s & 1), kz = 2 * mz + (s >> 1);
    const int fy = ky <= ny ? ky : 2 * ny - ky, fz = kz <= nz ? kz : 2 * nz - kz;
    const T f = g[((long long)kx * (nz + 1) + fz) * (ny + 1) + fy];
    w[i] = C2<T>{w[i].x * f, w[i].y * f};
  }
};
template <typename T>
struct SlabGatherOp {  // sum of the four back-twiddled copies -> R
  C2<T>* r;
  const C2<T>* w;
  const C2<T>*twz, *twy;
  SbRowBlocks rb;
  long long line0;
  int nz, ny, nzl;
  long long q;
  SB_D void operator()(long long i) const {
    const int y = (int)(i % ny);
    const long long t = i / ny;
    const int z = (int)(t % nz), kx = (int)(t / nz);
    const int zb = z / nzl, zl = z - zb * nzl;
    const C2<T> a = cconj(twz[z]), b = cconj(twy[y]);
    const C2<T> lo = cadd(w[i], cmul(w[q + i], b));
    const C2<T> hi = cadd(w[2 * q + i], cmul(w[3 * q + i], b));
    r[rb.row(line0 + (long long)zl * ny + y, 0) + rb.rel(zb * rb.kxl + kx)] = cadd(lo, cmul(hi, a));
  }
};
// Re(rfftn(G)) * scale, columns kx0 .. kx0 + kxl - 1, folded -> g[kx_in][kz][ky]
template <typename T>
struct SlabGreensExtractOp {
  T* g;
  const C2<T>* spec;  // (2nz, 2ny, nx + 1)
  int nz, ny, nx, kx0;
  T scale;
  SB_D void operator()(long long i) const {
    const int ky = (int)(i % (ny + 1));
    const long long t = i / (ny + 1);
    const int kz = (int)(t % (nz + 1)), kx = kx0 + (int)(t / (nz + 1));
    g[i] = kx <= nx ? spec[((long long)kz * 2 * ny + ky) * (nx + 1) + kx].x * scale : T(0);
  }
};

struct SbCufftSlabDims {
  int nzl, kxl, kx0;
  long long rows;  // x-pass rows per component: nzl ny
  long long q;     // one twiddled copy of the rank's kx slab: kxl nz ny
  SbRowBlocks rb;  // the exchange buffers of ncomp components
};
static SbCufftSlabDims cufft_slab_dims(const sb200_poisson* p, int ncomp) {
  SbCufftSlabDims d;
  d.nzl = p->nz / p->nranks;
  d.kxl = sb_slab_kxl(p->nx, p->nranks);
  d.kx0 = p->rank * d.kxl;
  d.rows = (long long)d.nzl * p->ny;
  d.q = (long long)d.kxl * p->nz * p->ny;
  d.rb = sb_row_blocks(d.kxl, ncomp * d.rows * d.kxl);
  return d;
}

template <typename T>
static int cufft_slab_setup_t(sb200_poisson* p, SbCufftSlabState* st, void* stream) {
  const SbCufftSlabDims d = cufft_slab_dims(p, 1);
  const int nz = p->nz, ny = p->ny, nx = p->nx;
  const size_t w = sizeof(T);
  const bool f32 = sizeof(T) == 4;
  // plans: x rows (R2C / C2R of length 2nx), the four copies of every kx line ((nz, ny) C2C); they share one
  // work area, allocated here and counted in the workspace
  size_t area = 0;
  {
    SB_CUFFT(cufftCreate(&st->xf), "slab plan x fwd");
    SB_CUFFT(cufftCreate(&st->xi), "slab plan x inv");
    SB_CUFFT(cufftCreate(&st->yz), "slab plan yz");
    for (cufftHandle h : {st->xf, st->xi, st->yz}) SB_CUFFT(cufftSetAutoAllocation(h, 0), "slab plan work area");
    int n[1] = {2 * nx}, re[1] = {2 * nx}, ce[1] = {nx + 1}, n2[2] = {nz, ny};
    size_t ws[3] = {0, 0, 0};
    SB_CUFFT(cufftMakePlanMany(st->xf, 1, n, re, 1, 2 * nx, ce, 1, nx + 1, f32 ? CUFFT_R2C : CUFFT_D2Z, (int)d.rows,
                               &ws[0]),
             "slab plan x fwd");
    SB_CUFFT(cufftMakePlanMany(st->xi, 1, n, ce, 1, nx + 1, re, 1, 2 * nx, f32 ? CUFFT_C2R : CUFFT_Z2D, (int)d.rows,
                               &ws[1]),
             "slab plan x inv");
    SB_CUFFT(cufftMakePlanMany(st->yz, 2, n2, nullptr, 1, nz * ny, nullptr, 1, nz * ny, f32 ? CUFFT_C2C : CUFFT_Z2Z,
                               4 * d.kxl, &ws[2]),
             "slab plan yz");
    for (size_t v : ws) area = v > area ? v : area;
    if (area) SB_CUDA(cudaMalloc(&st->fft_area, area), "slab cufft work area");
    for (cufftHandle h : {st->xf, st->xi, st->yz}) SB_CUFFT(cufftSetWorkArea(h, st->fft_area), "slab plan work area");
  }
  const size_t xr_bytes = (size_t)d.rows * 2 * nx * w;
  const size_t xc_bytes = ((size_t)d.rows * (nx + 1) * 2 * w + 255) & ~(size_t)255;
  const size_t w_bytes = (size_t)4 * d.q * 2 * w;
  const size_t work_bytes = w_bytes > xc_bytes + xr_bytes ? w_bytes : xc_bytes + xr_bytes;
  const size_t g_bytes = (size_t)d.kxl * (nz + 1) * (ny + 1) * w;
  SB_CUDA(cudaMalloc(&st->xr, xr_bytes), "slab x buffer");
  SB_CUDA(cudaMalloc(&st->work, work_bytes), "slab work buffer");
  SB_CUDA(cudaMalloc(&st->g, g_bytes), "slab greens table");
  st->twz = make_twiddles<T>(nz, nz, 2.0 * nz, stream);
  st->twy = make_twiddles<T>(ny, ny, 2.0 * ny, stream);
  SB_REQUIRE(st->twz && st->twy, "cufft backend: slab twiddle allocation");
  st->xo_off = xc_bytes;
  st->bytes = area + xr_bytes + work_bytes + g_bytes + (size_t)(nz + ny) * 2 * w;
  SB_CUDA(cudaMemsetAsync(st->xr, 0, xr_bytes, (cudaStream_t)stream), "slab x buffer zero");
  // Green's spectrum on the doubled grid through the single-rank code, the rank's columns kept
  struct Scratch {
    cufftHandle fwd = 0;
    void *real = nullptr, *spec = nullptr;
    ~Scratch() {
      if (fwd) cufftDestroy(fwd);
      cudaFree(real);
      cudaFree(spec);
    }
  } sc;
  const long long nreal = 8LL * nz * ny * nx, nspec = 4LL * nz * ny * (nx + 1);
  SB_CUDA(cudaMalloc(&sc.real, nreal * w), "slab greens scratch");
  SB_CUDA(cudaMalloc(&sc.spec, nspec * 2 * w), "slab greens spectrum");
  SB_CUFFT(cufftPlan3d(&sc.fwd, 2 * nz, 2 * ny, 2 * nx, f32 ? CUFFT_R2C : CUFFT_D2Z), "slab greens plan");
  int e = cufft_greens_spectrum(p, sc.fwd, sc.real, sc.spec, stream);
  if (e) return e;
  e = sb_launch_flat((long long)d.kxl * (nz + 1) * (ny + 1),
                     SlabGreensExtractOp<T>{(T*)st->g, (const C2<T>*)sc.spec, nz, ny, nx, d.kx0,
                                            (T)cufft_greens_scale(p)},
                     stream, "slab_greens_extract");
  if (e) return e;
  SB_CUDA(cudaStreamSynchronize((cudaStream_t)stream), "slab create sync");
  return 0;
}

static int cufft_slab_create(sb200_poisson* p, void* stream) {
  SB_REQUIRE(p->dim == 3, "cufft backend: the z-slab mode is implemented for 3D grids");
  SB_REQUIRE(p->nz % p->nranks == 0 && p->rank >= 0 && p->rank < p->nranks,
             "cufft backend: nz must split into one slab per rank");
  auto* st = new SbCufftSlabState();
  p->backend_state = st;
  SB_DISPATCH_DTYPE(p->dtype, return cufft_slab_setup_t<T>(p, st, stream));
}

static void cufft_slab_destroy(sb200_poisson* p) {
  auto* st = (SbCufftSlabState*)p->backend_state;
  if (!st) return;
  if (st->xf) cufftDestroy(st->xf);
  if (st->xi) cufftDestroy(st->xi);
  if (st->yz) cufftDestroy(st->yz);
  cudaFree(st->xr);
  cudaFree(st->work);
  cudaFree(st->g);
  cudaFree(st->twz);
  cudaFree(st->twy);
  cudaFree(st->fft_area);
  delete st;
  p->backend_state = nullptr;
}

static int64_t cufft_slab_bytes(const sb200_poisson* p) {
  auto* st = (SbCufftSlabState*)p->backend_state;
  return st ? (int64_t)st->bytes : 0;
}

template <typename T>
static int cufft_slab_forward_t(sb200_poisson* p, const void* rhs, int ncomp, void* send, void* stream) {
  auto* st = (SbCufftSlabState*)p->backend_state;
  const SbCufftSlabDims d = cufft_slab_dims(p, ncomp);
  const long long smy = p->ny + 2 * p->gs, smx = p->nx + 2 * p->gs, svol = (d.nzl + 2LL * p->gs) * smy * smx;
  C2<T>* xc = (C2<T>*)st->work;
  SB_CUFFT(cufftSetStream(st->xf, (cudaStream_t)stream), "set stream");
  for (int c = 0; c < ncomp; ++c) {
    int e = sb_launch_flat(d.rows * p->nx,
                           SlabPadOp<T>{(T*)st->xr, (const T*)rhs + c * svol, p->ny, p->nx, p->gs, smy, smx}, stream,
                           "slab_pad");
    if (e) return e;
    if (sizeof(T) == 4)
      SB_CUFFT(cufftExecR2C(st->xf, (cufftReal*)st->xr, (cufftComplex*)xc), "slab R2C");
    else
      SB_CUFFT(cufftExecD2Z(st->xf, (cufftDoubleReal*)st->xr, (cufftDoubleComplex*)xc), "slab D2Z");
    e = sb_launch_flat(d.rows * (p->nx + 1), SlabBlocksOp<T, true>{xc, (C2<T>*)send, d.rb, c * d.rows, p->nx + 1},
                       stream, "slab_pack");
    if (e) return e;
  }
  return 0;
}

template <typename T>
static int cufft_slab_spectral_t(sb200_poisson* p, void* recv, int ncomp, void* stream) {
  auto* st = (SbCufftSlabState*)p->backend_state;
  const SbCufftSlabDims d = cufft_slab_dims(p, ncomp);
  C2<T>* w = (C2<T>*)st->work;
  const C2<T>*twz = (const C2<T>*)st->twz, *twy = (const C2<T>*)st->twy;
  SB_CUFFT(cufftSetStream(st->yz, (cudaStream_t)stream), "set stream");
  for (int c = 0; c < ncomp; ++c) {
    int e = sb_launch_flat(
        d.q, SlabSpreadOp<T>{w, (const C2<T>*)recv, twz, twy, d.rb, c * d.rows, p->nz, p->ny, d.nzl, d.q}, stream,
        "slab_spread");
    if (e) return e;
    if (sizeof(T) == 4)
      SB_CUFFT(cufftExecC2C(st->yz, (cufftComplex*)w, (cufftComplex*)w, CUFFT_FORWARD), "slab C2C fwd");
    else
      SB_CUFFT(cufftExecZ2Z(st->yz, (cufftDoubleComplex*)w, (cufftDoubleComplex*)w, CUFFT_FORWARD), "slab Z2Z fwd");
    e = sb_launch_flat(4 * d.q, SlabGreensMulOp<T>{w, (const T*)st->g, p->nz, p->ny, d.kxl, d.q}, stream,
                       "slab_greens_mul");
    if (e) return e;
    if (sizeof(T) == 4)
      SB_CUFFT(cufftExecC2C(st->yz, (cufftComplex*)w, (cufftComplex*)w, CUFFT_INVERSE), "slab C2C inv");
    else
      SB_CUFFT(cufftExecZ2Z(st->yz, (cufftDoubleComplex*)w, (cufftDoubleComplex*)w, CUFFT_INVERSE), "slab Z2Z inv");
    e = sb_launch_flat(d.q, SlabGatherOp<T>{(C2<T>*)recv, w, twz, twy, d.rb, c * d.rows, p->nz, p->ny, d.nzl, d.q},
                       stream, "slab_gather");
    if (e) return e;
  }
  return 0;
}

template <typename T>
static int cufft_slab_backward_t(sb200_poisson* p, void* solution, int ncomp, const void* send, void* stream) {
  auto* st = (SbCufftSlabState*)p->backend_state;
  const SbCufftSlabDims d = cufft_slab_dims(p, ncomp);
  const long long smy = p->ny + 2 * p->gs, smx = p->nx + 2 * p->gs, svol = (d.nzl + 2LL * p->gs) * smy * smx;
  C2<T>* xc = (C2<T>*)st->work;
  T* xo = (T*)((char*)st->work + st->xo_off);
  SB_CUFFT(cufftSetStream(st->xi, (cudaStream_t)stream), "set stream");
  for (int c = 0; c < ncomp; ++c) {
    int e = sb_launch_flat(d.rows * (p->nx + 1),
                           SlabBlocksOp<T, false>{xc, (C2<T>*)send, d.rb, c * d.rows, p->nx + 1}, stream,
                           "slab_unpack");
    if (e) return e;
    if (sizeof(T) == 4)
      SB_CUFFT(cufftExecC2R(st->xi, (cufftComplex*)xc, (cufftReal*)xo), "slab C2R");
    else
      SB_CUFFT(cufftExecZ2D(st->xi, (cufftDoubleComplex*)xc, (cufftDoubleReal*)xo), "slab Z2D");
    e = sb_launch_flat(d.rows * p->nx, SlabCropOp<T>{(T*)solution + c * svol, xo, p->ny, p->nx, p->gs, smy, smx},
                       stream, "slab_crop");
    if (e) return e;
  }
  return 0;
}

int sb_poisson_cufft_slab_forward(sb200_poisson* p, const void* rhs, int ncomp, void* send_buf, void* stream) {
  SB_DISPATCH_DTYPE(p->dtype, return cufft_slab_forward_t<T>(p, rhs, ncomp, send_buf, stream));
}
int sb_poisson_cufft_slab_spectral(sb200_poisson* p, void* recv_buf, int ncomp, void* stream) {
  SB_DISPATCH_DTYPE(p->dtype, return cufft_slab_spectral_t<T>(p, recv_buf, ncomp, stream));
}
int sb_poisson_cufft_slab_backward(sb200_poisson* p, void* solution, int ncomp, const void* send_buf,
                                   void* stream) {
  SB_DISPATCH_DTYPE(p->dtype, return cufft_slab_backward_t<T>(p, solution, ncomp, send_buf, stream));
}
#else
int sb_poisson_cufft_create(sb200_poisson*, void*) { sb_set_error("cuFFT backend unavailable in emulation"); return -1; }
int sb_poisson_cufft_destroy(sb200_poisson*) { return 0; }
int64_t sb_poisson_cufft_bytes(const sb200_poisson*) { return 0; }
int sb_poisson_cufft_solve(sb200_poisson*, void*, const void*, int, void*) { return -1; }
int sb_poisson_cufft_slab_forward(sb200_poisson*, const void*, int, void*, void*) { return -1; }
int sb_poisson_cufft_slab_spectral(sb200_poisson*, void*, int, void*) { return -1; }
int sb_poisson_cufft_slab_backward(sb200_poisson*, void*, int, const void*, void*) { return -1; }
#endif
