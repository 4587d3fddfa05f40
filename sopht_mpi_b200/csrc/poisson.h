// Internal definition of the opaque Poisson handle.
#pragma once
#include "sb200_common.h"

struct sb200_poisson {
  int dim, dtype;
  int nz, ny, nx;  // global interior grid (2D: nz = 1)
  int gs;
  int rank, nranks;
  int backend;     // 0 = cuFFT generic, 1 = pruned in-kernel FFT pipeline (power-of-two grids)
  double x_range, y_range, z_range;
  double dx;       // value of real_t(x_range / nx)
  void* backend_state;
};

#ifndef SB200_EMU
#define SB_RN_MUL_F(a, b) __fmul_rn(a, b)
#define SB_RN_ADD_F(a, b) __fadd_rn(a, b)
#define SB_RN_MUL_D(a, b) __dmul_rn(a, b)
#define SB_RN_ADD_D(a, b) __dadd_rn(a, b)
#else
#define SB_RN_MUL_F(a, b) ((a) * (b))
#define SB_RN_ADD_F(a, b) ((a) + (b))
#define SB_RN_MUL_D(a, b) ((a) * (b))
#define SB_RN_ADD_D(a, b) ((a) + (b))
#endif
// individually rounded ops (no FMA contraction) so G matches numpy bit for bit
SB_D float rn_mul(float a, float b) { return SB_RN_MUL_F(a, b); }
SB_D float rn_add(float a, float b) { return SB_RN_ADD_F(a, b); }
SB_D double rn_mul(double a, double b) { return SB_RN_MUL_D(a, b); }
SB_D double rn_add(double a, double b) { return SB_RN_ADD_D(a, b); }

// Free-space Green's function on the doubled grid, evaluated in real_t like the reference
// (UnboundedPoissonSolverMPI3D.py:82-114, UnboundedPoissonSolverMPI2D.py:73-101).
template <typename T>
struct SbGreens {
  const T* xl;  // coordinate lines of the doubled grid (device), lengths 2nx, 2ny, 2nz
  const T* yl;
  const T* zl;
  int dim;
  T two_xr, two_yr, two_zr, four_pi, two_pi, g0;
  SB_D T operator()(long long z, long long y, long long x) const {
    if (x == 0 && y == 0 && z == 0) return g0;
    const T xv = xl[x], yv = yl[y];
    const T ex = fmin(xv, two_xr - xv), ey = fmin(yv, two_yr - yv);
    T r2 = rn_add(rn_mul(ex, ex), rn_mul(ey, ey));
    if (dim == 3) {
      const T zv = zl[z];
      const T ez = fmin(zv, two_zr - zv);
      r2 = rn_add(r2, rn_mul(ez, ez));
      return (T(1) / sqrt(r2)) / four_pi;
    }
    return -log(sqrt(r2)) / two_pi;
  }
};
// Build the evaluator; `*lines_dev` receives a device allocation the caller frees with
// sb_poisson_free_greens_lines after the kernels using it have completed.
template <typename T>
int sb_poisson_make_greens(const sb200_poisson* p, SbGreens<T>* out, void** lines_dev, void* stream);
void sb_poisson_free_greens_lines(void* lines_dev);

// Fill `dst` (device, (2nz,2ny,2nx) reals, contiguous) with the free-space Green's
// function on the doubled grid, evaluated in real_t exactly like the reference
// (UnboundedPoissonSolverMPI3D.py:82-114 / UnboundedPoissonSolverMPI2D.py:73-101).
int sb_poisson_fill_greens(const sb200_poisson* p, void* dst, void* stream);

// The exchange format of the z-slab solve, shared by both backends.
// Rows of kx bins either contiguous (pitch elements per row) or, for the x-slab transpose of the
// distributed solve, split into blocks of kxl bins: bin k of row `line` lives at
//   (k / kxl) * blk + line * kxl + k % kxl        (one block per destination / source rank)
// kx bins per rank of the x-slab decomposition: ceil((nx + 1) / nranks) rounded up to a multiple of
// 4 so that every row of a block starts on a 32-byte sector
static inline int sb_slab_kxl(int nx, int nranks) { return ((nx + 1 + nranks - 1) / nranks + 3) & ~3; }

struct SbRowBlocks {
  int kxl = 0;          // 0: contiguous rows
  unsigned magic = 0;   // ceil(2^32 / kxl): k / kxl == umulhi(k, magic) for k * kxl < 2^32
  long long dblk = 0;   // block stride minus kxl
  // element offset of bin k relative to the start of its row in block 0
  SB_D long long rel(int k) const {
#ifdef SB200_EMU
    const int b = k / kxl;
#else
    const int b = (int)__umulhi((unsigned)k, magic);
#endif
    return (long long)b * dblk + k;
  }
  SB_D long long row(long long line, long long pitch) const { return line * (kxl ? (long long)kxl : pitch); }
};
static inline SbRowBlocks sb_row_blocks(int kxl, long long blk) {
  SbRowBlocks rb;
  rb.kxl = kxl;
  rb.magic = kxl ? (unsigned)((0x100000000ULL + (unsigned long long)kxl - 1) / (unsigned long long)kxl) : 0;
  rb.dblk = blk - kxl;
  return rb;
}

int sb_poisson_cufft_create(sb200_poisson* p, void* stream);
int sb_poisson_cufft_destroy(sb200_poisson* p);
int sb_poisson_cufft_solve(sb200_poisson* p, void* solution, const void* rhs, int ncomp, void* stream);
int64_t sb_poisson_cufft_bytes(const sb200_poisson* p);
// z-slab stages of a distributed cuFFT handle (any grid size, any rank count that divides nz)
int sb_poisson_cufft_slab_forward(sb200_poisson* p, const void* rhs, int ncomp, void* send_buf, void* stream);
int sb_poisson_cufft_slab_spectral(sb200_poisson* p, void* recv_buf, int ncomp, void* stream);
int sb_poisson_cufft_slab_backward(sb200_poisson* p, void* solution, int ncomp, const void* send_buf,
                                   void* stream);

int sb_poisson_fft_create(sb200_poisson* p, void* stream);
int sb_poisson_fft_destroy(sb200_poisson* p);
int sb_poisson_fft_solve(sb200_poisson* p, void* solution, const void* rhs, int ncomp, void* stream);
int64_t sb_poisson_fft_bytes(const sb200_poisson* p);
