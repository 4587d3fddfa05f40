// Unbounded Poisson solve, hot-path backend: zero-padding-PRUNED three-pass transform with
// in-kernel FFTs (fft_device.h).  Per component and cell (W = bytes per real):
//   x pass   r2c   : read 1W  write 2W      (rows of nx reals -> nx+1 bins, half-length FFT)
//   y pass   fwd   : read 2W  write 4W      (ny -> 2ny, upper half of the input is zero)
//   z pass   fused : read 4W  write 4W      (nz -> 2nz fwd, x Ghat, inverse, keep nz) in place
//   y pass   inv   : read 4W  write 2W
//   x pass   c2r   : read 2W  write 1W      (straight into the padded solution field)
// = 26 W, plus the Green's spectrum stored REAL and mirror-compressed to (nz+1)(ny+1)(nx+1)
// (~1 W per cell per component).  No doubled-domain buffer is ever materialised.
// Reference semantics: UnboundedPoissonSolverMPI3D.py:133-167 (+ fft_mpi_3d.py:34-48):
// psi = irfftn(rfftn(pad0(omega)) * rfftn(G) * dx^3)[:nz,:ny,:nx].
#include "fft_device.h"
#include "poisson.h"

#include <cstdlib>
#include <vector>

// lines per block of the 32-point-per-thread kernels (16 lines measured slower at n = 512)
#define SB_P32_LINES(log2n) 8


#ifndef SB200_EMU
#define SB_DEV_ALLOC(ptr, bytes) (cudaMalloc((void**)&(ptr), (bytes)) == cudaSuccess)
#define SB_DEV_FREE(ptr) cudaFree(ptr)
#define SB_DEV_UPLOAD(dst, src, bytes, stream) \
  cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, (cudaStream_t)(stream))
#define SB_STREAM_SYNC(stream) cudaStreamSynchronize((cudaStream_t)(stream))
#else
#define SB_DEV_ALLOC(ptr, bytes) (((ptr) = (decltype(ptr))malloc(bytes)) != nullptr)
#define SB_DEV_FREE(ptr) free(ptr)
#define SB_DEV_UPLOAD(dst, src, bytes, stream) memcpy(dst, src, bytes)
#define SB_STREAM_SYNC(stream) (void)0
#endif

// A batch of lines.  Line (i, o1, o2) starts at element
//     i + (o1 & (2^o1_shift - 1)) * s1 + (o1 >> o1_shift) * s1_hi + o2 * s2
// and point k of it lives a further k * pt elements on.  o1_shift / s1_hi split the o1 axis into
// blocks (the per-source-rank blocks of the slab transposes); the default o1_shift = 30 is one block.
// The grid is (ceil(inner / lines_per_block), n1, n2): no index division.
struct SbLines {
  int inner, n1, n2;
  long long s1, s2;
  long long pt;
  int o1_shift = 30;
  long long s1_hi = 0;
  // grouped lines (tile-contiguous layout of the fused z pass): line i sits at (i & (2^gsh - 1)) inside
  // group i >> gsh, groups are s_grp elements apart.  gsh = 31: plain (line i at element i).
  int gsh = 31;
  long long s_grp = 0;
  // rot = 7: the 8 lines of a group are rotated by (o1 >> 1) & 7 slots inside their 64-byte row (o1 = z in
  // the y passes), which makes the column reads of the one-line-per-warp z kernel bank-conflict free
  int rot = 0;
  SB_HD long long base(int i, int o1, int o2) const {
    return ((i + ((o1 >> 1) & rot)) & ((1u << gsh) - 1)) + (long long)(i >> gsh) * s_grp +
           (long long)(o1 & ((1 << o1_shift) - 1)) * s1 + (long long)(o1 >> o1_shift) * s1_hi + o2 * s2;
  }
};

// ------------------------------------------------------------- row sources (x pass)
// rows are addressed (y, z, c) = (blockIdx.x group, blockIdx.y, blockIdx.z)
template <typename T>
struct FieldRows {
  T* f;  // padded field(s) (ncomp, mz, my, mx)
  int ny, gs, dim;
  long long my, mx, vol;
  SB_D T* row(int c, int z, int y) const {
    return f + (dim == 3 ? c * vol + ((long long)(z + gs) * my + (y + gs)) * mx + gs
                         : c * vol + (long long)(y + gs) * mx + gs);
  }
  SB_D C2<T> load(int c, int z, int y, int m) const {
    const T* p = row(c, z, y) + 2 * m;
    if ((gs & 1) == 0) return *reinterpret_cast<const C2<T>*>(p);  // rows start on an even element
    return C2<T>{p[0], p[1]};
  }
};
template <typename T>
struct GreensRows {
  SbGreens<T> g;
  int ny;  // rows per z (= 2 ny of the solver)
  SB_D C2<T> load(int, int z, int y, int m) const { return C2<T>{g(z, y, 2 * m), g(z, y, 2 * m + 1)}; }
};

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

// ------------------------------------------------------------------ x pass: r2c
// Real rows of length 2N (second half zero when PRUNED) -> N+1 bins through ONE complex FFT
// of length N on z[m] = x[2m] + i x[2m+1]:
//   X[k] = (Z[k] + conj Z[N-k])/2 - i W_2N^k (Z[k] - conj Z[N-k])/2
template <typename T, typename Rows, bool PRUNED, int LOG2N, int LINES>
__global__ void __launch_bounds__(LOG2N > 0 ? LINES * (1 << LOG2N) / SB_FFT_R : 512)
    sb_fft_x_r2c_kernel(SbFftPlan plan, int lines_rt, Rows rows, C2<T>* out, long long out_pitch,
                        const C2<T>* __restrict__ tw, const C2<T>* __restrict__ wpost, SbRowBlocks rb) {
  SB_DYN_SMEM(smem_raw);
  C2<T>* sm = reinterpret_cast<C2<T>*>(smem_raw);
  const int Tn = LOG2N > 0 ? (1 << LOG2N) / SB_FFT_R : plan.threads, N = LOG2N > 0 ? (1 << LOG2N) : plan.n;
  const int lines_per_block = LOG2N > 0 ? LINES : lines_rt;
  const int l = threadIdx.x / Tn, t = threadIdx.x - l * Tn;
  const int y = blockIdx.x * lines_per_block + l;
  const int z = blockIdx.y, c = blockIdx.z;
  const bool valid = y < rows.ny;
  const int yc = valid ? y : rows.ny - 1;  // clamp: every thread runs the FFT, only stores are masked
  const SbSmemLine<T, false> sl = sb_smem_line<T, false>(sm, l, 0, sb_fft_npad(N));
  constexpr int IN = PRUNED ? SB_FFT_R / 2 : SB_FFT_R;
  C2<T> v[SB_FFT_R];
#pragma unroll
  for (int p = 0; p < SB_FFT_R; ++p) v[p] = p < IN ? rows.load(c, z, yc, t + p * Tn) : C2<T>{T(0), T(0)};
  if constexpr (LOG2N > 0)
    sb_fft_forward_c<T, LOG2N, false, LINES>(v, t, tw, SbFftLineC<T, LOG2N, false, LINES>::line(sm, l));
  else
    sb_fft_forward<T, false>(v, plan, t, tw, sl);
#pragma unroll
  for (int p = 0; p < SB_FFT_R; ++p) sl.at(t + p * Tn) = v[p];
  __syncthreads();
  if (valid) {
    const long long line = ((long long)c * gridDim.y + z) * rows.ny + y;
    C2<T>* row = out + rb.row(line, out_pitch);
    C2<T> r[SB_FFT_R];
#pragma unroll
    for (int p = 0; p < SB_FFT_R; ++p) {
      const int k = t + p * Tn;
      const C2<T> zk = v[p];
      const C2<T> zc = cconj(sl.at((N - k) & (N - 1)));
      const C2<T> wd = cmul(wpost[k], csub(zk, zc));
      const C2<T> s = cadd(zk, zc);
      r[p] = C2<T>{T(0.5) * (s.x + wd.y), T(0.5) * (s.y - wd.x)};
    }
    const C2<T> last{v[0].x - v[0].y, T(0)};
    if (rb.kxl == 0) {  // (block-uniform branch hoisted out of the unrolled stores)
#pragma unroll
      for (int p = 0; p < SB_FFT_R; ++p) row[t + p * Tn] = r[p];
      if (t == 0) row[N] = last;
    } else {
#pragma unroll
      for (int p = 0; p < SB_FFT_R; ++p) row[rb.rel(t + p * Tn)] = r[p];
      if (t == 0) row[rb.rel(N)] = last;
    }
  }
}

// ------------------------------------------------------------------ x pass: c2r
// N+1 Hermitian bins -> first N reals of the (unnormalised) inverse of length 2N:
//   Z[k] = (X[k] + conj X[N-k]) + i W_2N^-k (X[k] - conj X[N-k]),  z = ifft_N(Z),
//   x[2m] = Re z[m], x[2m+1] = Im z[m]   for m < N/2
template <typename T, int LOG2N, int LINES>
__global__ void __launch_bounds__(LOG2N > 0 ? LINES * (1 << LOG2N) / SB_FFT_R : 512)
    sb_fft_x_c2r_kernel(SbFftPlan plan, int lines_rt, const C2<T>* in, long long in_pitch,
                        FieldRows<T> rows, const C2<T>* __restrict__ tw, const C2<T>* __restrict__ wpost,
                        SbRowBlocks rb) {
  SB_DYN_SMEM(smem_raw);
  C2<T>* sm = reinterpret_cast<C2<T>*>(smem_raw);
  const int Tn = LOG2N > 0 ? (1 << LOG2N) / SB_FFT_R : plan.threads, N = LOG2N > 0 ? (1 << LOG2N) : plan.n;
  const int lines_per_block = LOG2N > 0 ? LINES : lines_rt;
  const int l = threadIdx.x / Tn, t = threadIdx.x - l * Tn;
  const int y = blockIdx.x * lines_per_block + l;
  const int z = blockIdx.y, c = blockIdx.z;
  const bool valid = y < rows.ny;
  const int yc = valid ? y : rows.ny - 1;
  const SbSmemLine<T, false> sl = sb_smem_line<T, false>(sm, l, 0, sb_fft_npad(N));
  const long long line = ((long long)c * gridDim.y + z) * rows.ny + yc;
  const C2<T>* row = in + rb.row(line, in_pitch);
  C2<T> v[SB_FFT_R];
  if (rb.kxl == 0) {  // (block-uniform branch hoisted out of the unrolled loads)
#pragma unroll
    for (int p = 0; p < SB_FFT_R; ++p) v[p] = row[t + p * Tn];
    if (t == 0) sl.at(N) = row[N];
  } else {
#pragma unroll
    for (int p = 0; p < SB_FFT_R; ++p) v[p] = row[rb.rel(t + p * Tn)];
    if (t == 0) sl.at(N) = row[rb.rel(N)];
  }
#pragma unroll
  for (int p = 0; p < SB_FFT_R; ++p) sl.at(t + p * Tn) = v[p];
  __syncthreads();
#pragma unroll
  for (int p = 0; p < SB_FFT_R; ++p) {
    const int k = t + p * Tn;
    const C2<T> xk = sl.at(k);
    const C2<T> xc = cconj(sl.at(N - k));
    const C2<T> wd = cmul(cconj(wpost[k]), csub(xk, xc));
    const C2<T> s = cadd(xk, xc);
    v[p] = C2<T>{s.x - wd.y, s.y + wd.x};
  }
  __syncthreads();
  if constexpr (LOG2N > 0)
    sb_fft_inverse_c<T, LOG2N, false, LINES>(v, t, tw, SbFftLineC<T, LOG2N, false, LINES>::line(sm, l));
  else
    sb_fft_inverse<T, false>(v, plan, t, tw, sl);
  if (valid) {
    T* orow = rows.row(c, z, y);
#pragma unroll
    for (int p = 0; p < SB_FFT_R / 2; ++p) {
      const int m = t + p * Tn;
      if ((rows.gs & 1) == 0) {
        *reinterpret_cast<C2<T>*>(orow + 2 * m) = v[p];
      } else {
        orow[2 * m] = v[p].x;
        orow[2 * m + 1] = v[p].y;
      }
    }
  }
}

constexpr int sb_lb_threads(int log2n, int lines) { return log2n > 0 ? lines * ((1 << log2n) / SB_FFT_R) : 512; }
constexpr int sb_lb_blocks(int log2n, int lines, size_t elem) {
  return (log2n > 0 && elem == 4) ? 1024 / sb_lb_threads(log2n, lines) : 1;
}

// the fused forward+Green+inverse kernel: 256-thread blocks (n <= 512) run 3 per SM at <= 80
// registers, 512-thread blocks (n = 1024) 2 per SM at 64 registers (measured best on B200:
// profiles/r01_fft_tuning.md)
constexpr int sb_lb_blocks_conv(int log2n, int lines, size_t elem) {
  if (!(log2n > 0 && elem == 4)) return 1;
  const int nt = sb_lb_threads(log2n, lines);
  return nt <= 256 ? 768 / nt : nt <= 512 ? 1024 / nt : 1;
}

// -------------------------------------------------------------- strided line pass
// MODE 0: forward, pruned input (n/2 points read, n written)            -- y forward
// MODE 1: forward, x real Green's table, inverse, pruned in and out     -- z (2D: y) fused
// MODE 2: inverse, pruned output (n read, n/2 written)                   -- y inverse
// MODE 3: forward, nothing pruned                                        -- Green's set-up
template <typename T>
struct SbGreensTable {
  const T* g;  // [n_pt_half+1][n1_half+1][pitch] reals (mirror compressed)
  long long g_pt, g_s1;
  int n1_full = 1;  // full length of the o1 (ky) axis of the table
  int o1_off = 0;   // global ky of this batch's o1 = 0 (slab decomposition)
  // thread-order copy for the specialised fused z kernel (see GreensThreadOrderOp):
  // [m1][kx group][t][line][16 bins of thread t], so a thread's 16 factors are 64 contiguous bytes
  const T* g2 = nullptr;
  // x-slab decomposition: line i of the batch is global kx = kx0 + i (clamped to the last column
  // of the table for the zero-filled padding lines)
  int kx0 = 0, kx_last = 1 << 30;
};

// 16-byte asynchronous global -> shared copy (LDGSTS.128); the issuing thread reads its own slot
// back after sb_cp_async_wait_all(), so no barrier is involved
SB_D void sb_cp_async16(void* smem_dst, const void* gsrc) {
#ifdef SB200_EMU
  memcpy(smem_dst, gsrc, 16);
#else
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)),
               "l"(gsrc)
               : "memory");
#endif
}
SB_D void sb_cp_async_wait_all() {
#ifndef SB200_EMU
  asm volatile("cp.async.wait_all;" ::: "memory");
#endif
}

// specialised float kernels are held to <= 64 registers so that 1024 threads stay resident per SM.
// Every thread walks its 16 points with one running pointer (64-bit add per point, no multiplies).
// G2: the fused pass scales by the thread-order Green's table (gt.g2) instead of the compressed one
template <typename T, int MODE, int LOG2N, int LINES, bool G2>
__global__ void __launch_bounds__(sb_lb_threads(LOG2N, LINES), MODE == 1 ? sb_lb_blocks_conv(LOG2N, LINES, sizeof(T)) : sb_lb_blocks(LOG2N, LINES, sizeof(T)))
    sb_fft_strided_kernel(SbFftPlan plan, int lb_shift_rt, const C2<T>* in, SbLines lin, C2<T>* out, SbLines lout,
                          const C2<T>* __restrict__ tw, SbGreensTable<T> gt) {
  SB_DYN_SMEM(smem_raw);
  C2<T>* sm = reinterpret_cast<C2<T>*>(smem_raw);
  const int Tn = LOG2N > 0 ? (1 << LOG2N) / SB_FFT_R : plan.threads, n = LOG2N > 0 ? (1 << LOG2N) : plan.n;
  constexpr int LINES_SHIFT = LINES == 16 ? 4 : LINES == 8 ? 3 : LINES == 4 ? 2 : LINES == 2 ? 1 : 0;
  const int lb_shift = LOG2N > 0 ? LINES_SHIFT : lb_shift_rt;
  const int l = threadIdx.x & ((1 << lb_shift) - 1), t = threadIdx.x >> lb_shift;
  // grid (kx group, o1, o2); the fused kernel with the thread-order table runs (o2, kx group, o1)
  // so that the components of one (kx, ky) tile are neighbours and share the table rows in L2
  static_assert(!G2 || (MODE == 1 && LOG2N > 0 && sizeof(T) == 4), "thread-order table: fused float kernel");
  const int ib = G2 ? blockIdx.y : blockIdx.x;
  const int i = (ib << lb_shift) + l;
  const int o1 = G2 ? blockIdx.z : blockIdx.y, o2 = G2 ? blockIdx.x : blockIdx.z;
  const bool valid = i < lin.inner;
  const int ic = valid ? i : lin.inner - 1;
  const SbSmemLine<T, true> sl = sb_smem_line<T, true>(sm, l, lb_shift, sb_fft_npad(n));
  // staging slots of the Green's factors: chunk k of thread tid at float4 index k * NT + tid
  float4* gstage = nullptr;
  if constexpr (G2) {
    constexpr int NT = LINES * ((1 << LOG2N) / SB_FFT_R);
    gstage = reinterpret_cast<float4*>(sm + LINES * SbFftC<LOG2N>::npad) + threadIdx.x;
    const int g1 = o1 + gt.o1_off;
    const int m1 = g1 <= (gt.n1_full >> 1) ? g1 : gt.n1_full - g1;
    const float4* src = reinterpret_cast<const float4*>(gt.g2) +
                        (((long long)m1 * gridDim.y + ib) * NT + threadIdx.x) * 4;
#pragma unroll
    for (int k = 0; k < 4; ++k) sb_cp_async16(gstage + k * NT, src + k);
  }
  constexpr int IN = (MODE == 0 || MODE == 1) ? SB_FFT_R / 2 : SB_FFT_R;
  constexpr int OUT = (MODE == 1 || MODE == 2) ? SB_FFT_R / 2 : SB_FFT_R;
  C2<T> v[SB_FFT_R];
  {
    const C2<T>* gp = in + lin.base(ic, o1, o2);
    const long long sp = (long long)Tn * lin.pt;
    gp += (long long)t * lin.pt;
#pragma unroll
    for (int p = 0; p < SB_FFT_R; ++p) {
      if (p < IN) {
        v[p] = *gp;
        gp += sp;
      } else {
        v[p] = C2<T>{T(0), T(0)};
      }
    }
  }
  if constexpr (MODE != 2) {
    if constexpr (LOG2N > 0)
      sb_fft_forward_c<T, LOG2N, true, LINES>(v, t, tw, SbFftLineC<T, LOG2N, true, LINES>::line(sm, l));
    else
      sb_fft_forward<T, true>(v, plan, t, tw, sl);
  }
  if constexpr (G2) {
    constexpr int NT = LINES * ((1 << LOG2N) / SB_FFT_R);
    sb_cp_async_wait_all();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float4 gv = gstage[k * NT];
      v[4 * k] = cscale(v[4 * k], gv.x);
      v[4 * k + 1] = cscale(v[4 * k + 1], gv.y);
      v[4 * k + 2] = cscale(v[4 * k + 2], gv.z);
      v[4 * k + 3] = cscale(v[4 * k + 3], gv.w);
    }
  } else if constexpr (MODE == 1) {
    // real, mirror-compressed table: bin k = t + p Tn reads row min(k, n - k); for p < 8 that is
    // k itself (k < n/2), for p >= 8 it is (n - t) - p Tn -> two running pointers, no selects
    const int g1 = o1 + gt.o1_off;
    const int m1 = g1 <= (gt.n1_full >> 1) ? g1 : gt.n1_full - g1;
    const int kxg = ic + gt.kx0 < gt.kx_last ? ic + gt.kx0 : gt.kx_last;
    const T* g = gt.g + ((long long)m1 * gt.g_s1 + kxg);
    const long long gs = (long long)Tn * gt.g_pt;
    const T* ga = g + (long long)t * gt.g_pt;
    const T* gb = g + (long long)(n - t - (SB_FFT_R / 2) * Tn) * gt.g_pt;
#pragma unroll
    for (int p = 0; p < SB_FFT_R / 2; ++p) {
      v[p] = cscale(v[p], *ga);
      v[p + SB_FFT_R / 2] = cscale(v[p + SB_FFT_R / 2], *gb);
      ga += gs;
      gb -= gs;
    }
  }
  if constexpr (MODE == 1 || MODE == 2) {
    if constexpr (LOG2N > 0)
      sb_fft_inverse_c<T, LOG2N, true, LINES>(v, t, tw, SbFftLineC<T, LOG2N, true, LINES>::line(sm, l));
    else
      sb_fft_inverse<T, true>(v, plan, t, tw, sl);
  }
  if (valid) {
    C2<T>* gp = out + lout.base(i, o1, o2);
    const long long sp = (long long)Tn * lout.pt;
    gp += (long long)t * lout.pt;
#pragma unroll
    for (int p = 0; p < OUT; ++p) {
      *gp = v[p];
      gp += sp;
    }
  }
}

// ---------------------------------------------------------------- strided pass, 32 points per thread
// Same passes (MODE 0 / 1 / 2) for n = 512 and 1024 with ONE shared-memory exchange per transform
// (fft_device.h, sb_fft32_*): a line is n / 32 threads, a block 8 lines.  MODE 1 reads the compressed
// Green's table: the 3D float z pass at these lengths is the fused z kernel below, so this one runs
// the 2D y pass.
constexpr int sb_p32_min_blocks(int log2n, int lines) {
  const int nt = lines * ((1 << log2n) / SB_FFT_P32);
  return 512 / nt > 0 ? 512 / nt : 1;  // <= 128 registers per thread
}

template <typename T, int MODE, int LOG2N, int LINES>
__global__ void __launch_bounds__(LINES*((1 << LOG2N) / SB_FFT_P32), sb_p32_min_blocks(LOG2N, LINES))
    sb_fft_strided32_kernel(const C2<T>* in, SbLines lin, C2<T>* out, SbLines lout,
                            const C2<T>* __restrict__ tw, SbGreensTable<T> gt) {
  SB_DYN_SMEM(smem_raw);
  using FC = SbFft32C<LOG2N>;
  constexpr int PT = SB_FFT_P32, Tn = FC::Tn;
  constexpr int LINES_SHIFT = LINES == 16 ? 4 : LINES == 8 ? 3 : LINES == 4 ? 2 : LINES == 2 ? 1 : 0;
  constexpr int IN = (MODE == 0 || MODE == 1) ? PT / 2 : PT;
  constexpr int OUT = (MODE == 1 || MODE == 2) ? PT / 2 : PT;
  C2<T>* sm = reinterpret_cast<C2<T>*>(smem_raw);
  const int l = threadIdx.x & (LINES - 1), t = threadIdx.x >> LINES_SHIFT;
  const int i = (blockIdx.x << LINES_SHIFT) + l;
  const int o1 = blockIdx.y, o2 = blockIdx.z;
  const bool valid = i < lin.inner;
  const int ic = valid ? i : lin.inner - 1;
  C2<T>* sline = sm + l;
  C2<T> v[PT];
  {
    const C2<T>* gp = in + lin.base(ic, o1, o2);
    const long long sp = (long long)Tn * lin.pt;
    gp += (long long)t * lin.pt;
#pragma unroll
    for (int p = 0; p < PT; ++p) {
      if (p < IN) {
        v[p] = *gp;
        gp += sp;
      } else {
        v[p] = C2<T>{T(0), T(0)};
      }
    }
  }
  if constexpr (MODE != 2) sb_fft32_forward_c<T, LOG2N, LINES, MODE == 1>(v, t, tw, sline);
  if constexpr (MODE == 1) {
    const int g1 = o1 + gt.o1_off;
    const int m1 = g1 <= (gt.n1_full >> 1) ? g1 : gt.n1_full - g1;
    const int kxg = ic + gt.kx0 < gt.kx_last ? ic + gt.kx0 : gt.kx_last;
    const T* g = gt.g + ((long long)m1 * gt.g_s1 + kxg);
    const long long gs = (long long)Tn * gt.g_pt;
    const T* ga = g + (long long)t * gt.g_pt;
    const T* gb = g + (long long)(FC::n - t - (PT / 2) * Tn) * gt.g_pt;
#pragma unroll
    for (int p = 0; p < PT / 2; ++p) {
      v[p] = cscale(v[p], *ga);
      v[p + PT / 2] = cscale(v[p + PT / 2], *gb);
      ga += gs;
      gb -= gs;
    }
  }
  if constexpr (MODE == 1 || MODE == 2) sb_fft32_inverse_c<T, LOG2N, LINES, false>(v, t, tw, sline);
  if (valid) {
    C2<T>* gp = out + lout.base(i, o1, o2);
    const long long sp = (long long)Tn * lout.pt;
    gp += (long long)t * lout.pt;
#pragma unroll
    for (int p = 0; p < OUT; ++p) {
      *gp = v[p];
      gp += sp;
    }
  }
}

// ------------------------------------------------------ fused z pass, persistent + bulk-copy prefetch
// The same transform as sb_fft_strided32_kernel<MODE 1> (forward FFT of the zero-padded z line, x real
// Green's spectrum, inverse FFT, first half kept, in place) on a TILE-CONTIGUOUS layout
//     Bt[c][kx group][ky][z][8 lines]            (one tile = nz x 8 complex = 16 / 32 KB contiguous)
// so that a whole tile moves with ONE bulk asynchronous copy (cp.async.bulk, the 1D TMA path, completion
// on an mbarrier).  Blocks are persistent: while a tile is transformed, the next tile of the block is
// already landing in shared memory, so the HBM latency that the one-tile-per-block kernel exposes at
// the start of every block (2-4 resident blocks per SM cannot hide it) leaves the critical path.
// Tiles are numbered (ky, kx group, component) with the component fastest: the three components of one
// (kx group, ky) are in flight together and share the Green's table rows in L2.
#ifndef SB200_EMU
SB_D unsigned sb_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
SB_D void sb_mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(sb_smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// arm the barrier with the byte count and start the copy (one thread)
SB_D void sb_bulk_load(void* smem_dst, const void* gsrc, unsigned bytes, unsigned long long* bar) {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sb_smem_u32(bar)), "r"(bytes)
               : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   sb_smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(sb_smem_u32(bar))
               : "memory");
}
// wait for phase `parity` of the barrier to complete, for a CONVERGED warp: the retry branch is taken on a
// warp vote, i.e. uniformly, so ptxas keeps treating the warp as converged (a per-thread retry loop in front
// of a __syncwarp makes it emit the out-of-line reconvergence path, with ~300 bytes of spills around it in
// the fused z kernel)
SB_D void sb_mbar_wait_warp(unsigned long long* bar, unsigned parity) {
  unsigned ok;
  do {
    asm volatile(
        "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(sb_smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!__all_sync(0xffffffffu, ok));
}
// arm + copy for one thread of a converged warp, PREDICATED instead of branched (a divergent branch in
// front of a __syncwarp makes ptxas emit its out-of-line reconvergence path); several copies may follow
// one arming with the total byte count
SB_D void sb_mbar_expect_if(bool pred, unsigned long long* bar, unsigned bytes) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.u32 p, %0, 0;\n"
      "@p fence.proxy.async.shared::cta;\n"
      "@p mbarrier.arrive.expect_tx.shared::cta.b64 _, [%2], %1;\n}" ::"r"((unsigned)pred),
      "r"(bytes), "r"(sb_smem_u32(bar))
      : "memory");
}
SB_D void sb_bulk_copy_if(bool pred, void* smem_dst, const void* gsrc, unsigned bytes, unsigned long long* bar) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.u32 p, %0, 0;\n"
      "@p cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%1], [%2], %3, [%4];\n}" ::"r"(
          (unsigned)pred),
      "r"(sb_smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(sb_smem_u32(bar))
      : "memory");
}
SB_D void sb_mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(sb_smem_u32(bar)) : "memory");
}
// generic-proxy writes to shared memory -> visible to the bulk-copy engine
SB_D void sb_fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// shared -> global bulk copy (one thread), completion tracked by the thread's bulk group
SB_D void sb_bulk_store(void* gdst, const void* smem_src, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(sb_smem_u32(smem_src)),
               "r"(bytes)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
SB_D void sb_bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
SB_D void sb_bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
#else
// emulation: the barrier word is [completed phases : 32][bytes / 16 in flight : 16][arrival count : 8][pending : 8]
SB_D void sb_mbar_init(unsigned long long* bar, unsigned count) {
  __atomic_store_n(bar, ((unsigned long long)count << 8) | count, __ATOMIC_SEQ_CST);
}
// pending -= arrivals, in-flight += tx16 (may be negative); the phase completes when both reach zero
SB_D void sb_mbar_update(unsigned long long* bar, unsigned arrivals, long long tx16) {
  unsigned long long e = __atomic_load_n(bar, __ATOMIC_SEQ_CST);
  for (;;) {
    const unsigned long long cnt = (e >> 8) & 0xffu, pend = (e & 0xffu) - arrivals;
    const unsigned long long tx = (unsigned long long)((long long)((e >> 16) & 0xffffu) + tx16) & 0xffffu;
    unsigned long long d = (e & 0xffffffff00000000ULL) | (tx << 16) | (cnt << 8) | pend;
    if (pend == 0 && tx == 0) d = (((e >> 32) + 1) << 32) | (cnt << 8) | cnt;
    if (__atomic_compare_exchange_n(bar, &e, d, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST)) return;
  }
}
SB_D void sb_mbar_arrive(unsigned long long* bar) { sb_mbar_update(bar, 1, 0); }
SB_D void sb_mbar_expect_if(bool pred, unsigned long long* bar, unsigned bytes) {
  if (pred) sb_mbar_update(bar, 1, bytes / 16);
}
SB_D void sb_bulk_copy_if(bool pred, void* smem_dst, const void* gsrc, unsigned bytes, unsigned long long* bar) {
  if (!pred) return;
  memcpy(smem_dst, gsrc, bytes);
  sb_mbar_update(bar, 0, -(long long)(bytes / 16));
}
SB_D void sb_bulk_load(void* smem_dst, const void* gsrc, unsigned bytes, unsigned long long* bar) {
  sb_mbar_expect_if(true, bar, bytes);
  sb_bulk_copy_if(true, smem_dst, gsrc, bytes, bar);
}
SB_D void sb_mbar_wait_warp(unsigned long long* bar, unsigned parity) {
  while (((__atomic_load_n(bar, __ATOMIC_SEQ_CST) >> 32) & 1u) == parity) std::this_thread::yield();
}
SB_D void sb_fence_async_smem() { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
SB_D void sb_bulk_store(void* gdst, const void* smem_src, unsigned bytes) { memcpy(gdst, smem_src, bytes); }
SB_D void sb_bulk_wait_read() {}
SB_D void sb_bulk_wait_all() {}
#endif

// ------------------------------------------------------ fused z pass, one line per warp
// A line's n / 32 threads sit inside ONE warp (fft_device.h, sb_fft32w_forward), so that no warp ever
// waits for another one inside the transform: the kernel is bound by FP32 issue, and block barriers
// between the exchange stages leave that pipe idle (DESIGN.md, "Fused z pass").  So:
//   * the register-stage exchange is warp local (__syncwarp only);
//   * a warp reads its line from the landed tile and writes the result back to the SAME slots: the tile
//     buffer needs no block barrier either.  Reading column l of the [z][8] tile would be an 8- to 16-way
//     bank conflict, therefore the y passes store the tile with its 64-byte rows rotated by (z >> 1) & 7
//     slots (SbLines::rot): a warp's 32 (16) consecutive z then fall on distinct banks;
//   * tiles move in AND out with bulk copies (cp.async.bulk, mbarrier / bulk-group completion); two tile
//     buffers per block alternate; the warp that writes the LAST line of a tile (shared-memory arrival
//     counter) stores the tile and re-arms the buffer with the tile after next, nobody waits for it;
//   * the Green's factors (g5[m1][kx group][line][n] floats, natural bin order) are staged per warp by a
//     bulk copy into the warp's own exchange line, which is idle between the two transforms; the copy
//     overlaps the second register stage of the forward transform.
template <int LOG2N>
struct SbZw {
  using FC = SbFft32C<LOG2N>;
  static constexpr int Tn = FC::Tn, LINES = 8, NT = LINES * Tn, NW = NT / 32, NZ = FC::n / 2;
  static constexpr unsigned TILE = NZ * LINES;  // complex elements of a tile
  static constexpr int XL = SbFft32W<LOG2N>::XL;
  static constexpr int BLOCKS = LOG2N >= 10 ? 2 : 4;
  static constexpr size_t smem = 2 * TILE * sizeof(C2<float>) + (size_t)LINES * XL * sizeof(float) + 128;
  static_assert((2 + NW) * 8 + 2 * 4 + 2 * 4 <= 128, "barriers, arrival counters, tile ids");
};

template <int LOG2N>
__global__ void __launch_bounds__(SbZw<LOG2N>::NT, SbZw<LOG2N>::BLOCKS)
    sb_fft_zconvw_kernel(C2<float>* B, int ntiles, int ncomp, int ng, int nky, const C2<float>* __restrict__ tw,
                         const float* __restrict__ g5, int n1_full, int* next_tile) {
  using Z = SbZw<LOG2N>;
  constexpr int PT = SB_FFT_P32, Tn = Z::Tn, N = Z::FC::n;
  constexpr unsigned TILE = Z::TILE, TILE_BYTES = TILE * sizeof(C2<float>);
  SB_DYN_SMEM(smem_raw);
  C2<float>* tbuf = reinterpret_cast<C2<float>*>(smem_raw);  // two tiles [nz][8]
  float* xch = reinterpret_cast<float*>(tbuf + 2 * TILE);    // exchange lines
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(xch + Z::LINES * Z::XL);  // full[2], green[NW]
  unsigned* cnt = reinterpret_cast<unsigned*>(bars + 2 + Z::NW);  // lines written per tile buffer
  int* tile_of = reinterpret_cast<int*>(cnt + 2);                  // tile held by each buffer
  const int tid = threadIdx.x, l = tid / Tn, t = tid % Tn, lane = tid & 31, warp = tid >> 5;
  float* xl = xch + l * Z::XL;
  const int slot = (l + (t >> 1)) & 7;  // (z >> 1) & 7 == (t >> 1) & 7 for every z = t + p Tn of this thread
  auto tile_offset = [&](int tile) {
    const int c = tile % ncomp, r = tile / ncomp;
    return (((long long)c * ng + r % ng) * nky + r / ng) * (long long)TILE;
  };
  // Tiles are handed out by a global counter (not a fixed stride): a block that starts late, because its
  // SM was still busy with the exchange kernel of the neighbouring component, simply processes fewer.
  // One thread fetches the tile for a buffer, records it, and either starts its copy or, when the tiles
  // have run out, completes the buffer's barrier by hand so that the waiting warps see the end.
  auto arm = [&](int b) {
    const int tile = atomicAdd(next_tile, 1);
    tile_of[b] = tile;
    if (tile < ntiles)
      sb_bulk_load(tbuf + b * TILE, B + tile_offset(tile), TILE_BYTES, bars + b);
    else
      sb_mbar_arrive(bars + b);
  };
  if (tid == 0) {
    sb_mbar_init(bars + 0, 1);
    sb_mbar_init(bars + 1, 1);
    for (int w = 0; w < Z::NW; ++w) sb_mbar_init(bars + 2 + w, 1);
    cnt[0] = cnt[1] = 0;
  }
  __syncthreads();
  if (tid == 0) {
    arm(0);
    arm(1);
  }
  for (int k = 0;; ++k) {
    const int b = k & 1;
    C2<float>* tb = tbuf + b * TILE + slot;
    sb_mbar_wait_warp(bars + b, (unsigned)(k >> 1) & 1u);
    if (tile_of[b] >= ntiles) break;
    C2<float> v[PT];
#pragma unroll
    for (int p = 0; p < PT / 2; ++p) v[p] = tb[(t + p * Tn) * Z::LINES];
    sb_fft32w_forward<LOG2N, true>(v, t, tw, xl);
    // the exchange buffer is idle until the next transform: stage this warp's Green's factors in it
    // (n floats per line, natural bin order) while the second register stage runs
    __syncwarp();
    {
      const int r = tile_of[b] / ncomp, kxg = r % ng, ky = r / ng;  // (re-read: registers are scarce)
      const int m1 = ky <= (n1_full >> 1) ? ky : n1_full - ky;
      constexpr int LW = 32 / Tn;  // lines per warp
      const float* src = g5 + (((long long)m1 * ng + kxg) * Z::LINES + warp * LW) * N;
      sb_mbar_expect_if(lane == 0, bars + 2 + warp, LW * N * sizeof(float));
#pragma unroll
      for (int i = 0; i < LW; ++i)
        sb_bulk_copy_if(lane == 0, xch + (warp * LW + i) * Z::XL, src + i * N, N * sizeof(float), bars + 2 + warp);
    }
    sb_fft32w_second<LOG2N>(v, t, tw);
    sb_mbar_wait_warp(bars + 2 + warp, (unsigned)k & 1u);
    // x Green's factor, and the conjugation that turns the second forward transform into the inverse
#pragma unroll
    for (int p = 0; p < PT; ++p) v[p] = cscale_conj(v[p], xl[t + p * Tn]);
    sb_fft32w_forward<LOG2N, false>(v, t, tw, xl);
    sb_fft32w_second<LOG2N>(v, t, tw);
#pragma unroll
    for (int p = 0; p < PT / 2; ++p) tb[(t + p * Tn) * Z::LINES] = C2<float>{v[p].x, -v[p].y};
    sb_fence_async_smem();
    __syncwarp();
    if (lane == 0) {
      __threadfence_block();
      if ((atomicAdd(cnt + b, 1u) + 1) % Z::NW == 0) {  // last line of the tile: store it, re-arm the buffer
        __threadfence_block();
        sb_bulk_store(B + tile_offset(tile_of[b]), tbuf + b * TILE, TILE_BYTES);
        sb_bulk_wait_read();
        arm(b);
      }
    }
  }
  if (lane == 0) sb_bulk_wait_all();
}

// Re(spectrum) * scale -> mirror-compressed table
template <typename T>
struct GreensExtractOp {
  T* g;
  const C2<T>* full;
  long long pitch, n2y, hy1;  // hy1 = ny + 1 rows kept
  T scale;
  SB_D void operator()(long long i) const {
    const long long kx = i % pitch, r = i / pitch;
    const long long ky = r % hy1, kz = r / hy1;
    g[i] = full[(kz * n2y + ky) * pitch + kx].x * scale;
  }
};

// compressed table g[mk][m1][kx] -> thread order g2[m1][ib][t][l][p]  (bin k = t + p Tn of the line
// kx = ib LINES + l with 16 bins per thread, sb_fft_strided_kernel; mk = min(k, n - k)); kx beyond the
// pitch reads as zero
template <typename T>
struct GreensThreadOrderOp {
  T* g2;
  const T* g;
  long long g_pt, g_s1;
  int n, Tn, lines, nib, pitch;
  int kx0, inner;  // first global kx of this rank's lines, number of lines
  int warp_order = 0;  // 1: g5[m1][ib][l][n] (natural bin order per line, sb_fft_zconvw_kernel)
  SB_D void operator()(long long idx) const {
    int p, l, t;
    long long r;
    if (warp_order) {
      const int k = (int)(idx % n), mk = k <= (n >> 1) ? k : n - k;
      r = idx / n;
      l = (int)(r % lines);
      r /= lines;
      const int ib = (int)(r % nib), i = ib * lines + l, kx = kx0 + i;
      const long long m1 = r / nib;
      g2[idx] = (i < inner && kx < pitch) ? g[mk * g_pt + m1 * g_s1 + kx] : T(0);
      return;
    } else {
      p = (int)(idx % SB_FFT_R);
      r = idx / SB_FFT_R;
      l = (int)(r % lines);
      r /= lines;
      t = (int)(r % Tn);
      r /= Tn;
    }
    const int ib = (int)(r % nib);
    const long long m1 = r / nib;
    const int k = t + p * Tn, mk = k <= (n >> 1) ? k : n - k, i = ib * lines + l, kx = kx0 + i;
    g2[idx] = (i < inner && kx < pitch) ? g[mk * g_pt + m1 * g_s1 + kx] : T(0);
  }
};

// --------------------------------------------------------------------- host state
// The kx side of a handle: where the x passes put their output and which kx lines the y / z passes
// transform.  A single-GPU solve is the one-rank case: all nz planes, rows of nx + 1 bins with pitch nx + 2.
// A z-slab rank r of P runs the x passes on its nz / P planes and writes each row as P blocks of kxl bins,
// one per destination rank; after the all-to-all it owns kx bins [r kxl, (r + 1) kxl) of ALL planes,
// blocked by source rank: R[zb][c][zl][y][kx].
struct SbKxSide {
  int planes;       // planes of the x passes
  int inner;        // kx lines of the y / z passes
  long long pitch;  // row pitch of the x-pass output and of B[c][nz][2ny][pitch]
  SbRowBlocks rb;   // blocks of the x-pass rows (contiguous on a single GPU)
  SbLines lx;       // the x-pass output as lines (kx, z, c) along y
  int kx0;          // global kx of line 0 (column of the Green's table)
};
static SbKxSide sb_kx_side(const sb200_poisson* p, int ncomp) {
  const int nranks = p->nranks, nz = p->dim == 3 ? p->nz : 1, ny = p->ny;
  SbKxSide k;
  k.planes = nz / nranks;
  k.inner = nranks > 1 ? sb_slab_kxl(p->nx, nranks) : p->nx + 1;
  k.pitch = nranks > 1 ? k.inner : p->nx + 2;
  k.kx0 = nranks > 1 ? p->rank * k.inner : 0;
  const long long blk = (long long)ncomp * k.planes * ny * k.pitch;  // one destination / source block
  k.lx = SbLines{k.inner, nz, ncomp, ny * k.pitch, k.planes * ny * k.pitch, k.pitch};
  if (nranks > 1) {
    k.rb = sb_row_blocks(k.inner, blk);
    k.lx.o1_shift = 0;
    while ((1 << k.lx.o1_shift) < k.planes) ++k.lx.o1_shift;
    k.lx.s1_hi = blk;
  }
  return k;
}

template <typename T>
struct SbFftState {
  SbFftPlan px, py, pz;
  C2<T>*twx = nullptr, *twy = nullptr, *twz = nullptr, *wpost = nullptr;
  C2<T>* A = nullptr;  // [ncomp][nz][ny][P]  (single GPU)
  C2<T>* B = nullptr;  // [ncomp][nz][2ny][pitch]  (SbKxSide)
  T* G = nullptr;      // [nz+1][ny+1][P]  (2D: [ny+1][P])
  T* G2 = nullptr;     // thread-order copy of G for the specialised fused z kernel (float, 3D)
  long long P = 0;
  size_t bytes = 0;
  // tile-contiguous layout of B + persistent bulk-copy z kernel (float, 3D, 2nz = 512 / 1024)
  bool zconv = false;
  int ng = 0;  // kx groups of 8 lines
  int* tile_counter = nullptr;  // work counter of the persistent z kernel
  // optional per-launch timing (sb200_poisson_set_profiling): events around the five launches
  bool profile = false, have_times = false;
#ifndef SB200_EMU
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
#endif
  void mark(int i, void* stream) {
#ifndef SB200_EMU
    if (profile) cudaEventRecord(ev[i], (cudaStream_t)stream);
#else
    (void)i; (void)stream;
#endif
  }
};

template <typename T>
static C2<T>* make_twiddles(int n, int count, double denom, void* stream) {
  // W[k] = exp(-2 pi i k / denom), k < count
  std::vector<C2<T>> h(count);
  for (int k = 0; k < count; ++k) {
    const double a = -2.0 * M_PI * (double)k / denom;
    h[k] = C2<T>{(T)std::cos(a), (T)std::sin(a)};
  }
  C2<T>* d = nullptr;
  if (!SB_DEV_ALLOC(d, sizeof(C2<T>) * count)) return nullptr;
  SB_DEV_UPLOAD(d, h.data(), sizeof(C2<T>) * count, stream);
  SB_STREAM_SYNC(stream);
  (void)n;
  return d;
}

static int lines_per_block_for(int threads_per_line, size_t elem, bool strided) {
  int lb = strided ? (elem == 4 ? 8 : 4) : 1;  // >= 64 B contiguous per point for strided passes
  while (lb * threads_per_line < 128) lb *= 2;
  while (lb > 1 && lb * threads_per_line > 512) lb /= 2;
  return lb;
}

// lines per block of the compile-time specialised kernels
template <typename T>
constexpr int sb_strided_lines(int log2n, int mode) {
  (void)mode;
  return (sizeof(T) == 4 && log2n <= 10) ? 8 : 4;
}
constexpr int sb_xpass_lines(int log2n) { return log2n <= 7 ? 16 : log2n == 8 ? 8 : log2n == 9 ? 4 : log2n == 10 ? 2 : 1; }

template <typename T, typename Rows, bool PRUNED, int LOG2N>
static int launch_x_r2c_c(const SbFftPlan& plan, int ny, int nz, int ncomp, const Rows& rows, C2<T>* out,
                          long long pitch, const C2<T>* tw, const C2<T>* wpost, void* stream,
                          const SbRowBlocks& rb) {
  constexpr int LINES = LOG2N > 0 ? sb_xpass_lines(LOG2N) : 0;
  const int lb = LOG2N > 0 ? LINES : lines_per_block_for(plan.threads, sizeof(T), false);
  const size_t smem = (size_t)lb * sb_fft_npad(plan.n) * sizeof(C2<T>);
  SB_KERNEL_ATTR_SMEM((sb_fft_x_r2c_kernel<T, Rows, PRUNED, LOG2N, LINES>), smem);
  const dim3 grid((unsigned)((ny + lb - 1) / lb), (unsigned)nz, (unsigned)ncomp);
  SB_LAUNCH_COOP((sb_fft_x_r2c_kernel<T, Rows, PRUNED, LOG2N, LINES>), grid, dim3(lb * plan.threads), smem,
                 stream, plan, lb, rows, out, pitch, tw, wpost, rb);
  SB_CHECK_LAUNCH("fft_x_r2c");
  return 0;
}
template <typename T, typename Rows, bool PRUNED>
static int launch_x_r2c(const SbFftPlan& plan, int ny, int nz, int ncomp, const Rows& rows, C2<T>* out,
                        long long pitch, const C2<T>* tw, const C2<T>* wpost, void* stream,
                        const SbRowBlocks& rb = SbRowBlocks()) {
  if constexpr (PRUNED) {  // compile-time specialised lengths, float and double
    switch (plan.log2n) {
      case 8: return launch_x_r2c_c<T, Rows, PRUNED, 8>(plan, ny, nz, ncomp, rows, out, pitch, tw, wpost, stream, rb);
      case 9: return launch_x_r2c_c<T, Rows, PRUNED, 9>(plan, ny, nz, ncomp, rows, out, pitch, tw, wpost, stream, rb);
      case 10: return launch_x_r2c_c<T, Rows, PRUNED, 10>(plan, ny, nz, ncomp, rows, out, pitch, tw, wpost, stream, rb);
      default: break;
    }
  }
  return launch_x_r2c_c<T, Rows, PRUNED, 0>(plan, ny, nz, ncomp, rows, out, pitch, tw, wpost, stream, rb);
}

template <typename T, int LOG2N>
static int launch_x_c2r_c(const SbFftPlan& plan, int ny, int nz, int ncomp, const C2<T>* in, long long pitch,
                          const FieldRows<T>& dst, const C2<T>* tw, const C2<T>* wpost, void* stream,
                          const SbRowBlocks& rb) {
  constexpr int LINES = LOG2N > 0 ? sb_xpass_lines(LOG2N) : 0;
  const int lb = LOG2N > 0 ? LINES : lines_per_block_for(plan.threads, sizeof(T), false);
  const size_t smem = (size_t)lb * sb_fft_npad(plan.n) * sizeof(C2<T>);
  SB_KERNEL_ATTR_SMEM((sb_fft_x_c2r_kernel<T, LOG2N, LINES>), smem);
  const dim3 grid((unsigned)((ny + lb - 1) / lb), (unsigned)nz, (unsigned)ncomp);
  SB_LAUNCH_COOP((sb_fft_x_c2r_kernel<T, LOG2N, LINES>), grid, dim3(lb * plan.threads), smem, stream, plan, lb,
                 in, pitch, dst, tw, wpost, rb);
  SB_CHECK_LAUNCH("fft_x_c2r");
  return 0;
}
template <typename T>
static int launch_x_c2r(const SbFftPlan& plan, int ny, int nz, int ncomp, const C2<T>* in, long long pitch,
                        const FieldRows<T>& dst, const C2<T>* tw, const C2<T>* wpost, void* stream,
                        const SbRowBlocks& rb = SbRowBlocks()) {
  {
    switch (plan.log2n) {
      case 8: return launch_x_c2r_c<T, 8>(plan, ny, nz, ncomp, in, pitch, dst, tw, wpost, stream, rb);
      case 9: return launch_x_c2r_c<T, 9>(plan, ny, nz, ncomp, in, pitch, dst, tw, wpost, stream, rb);
      case 10: return launch_x_c2r_c<T, 10>(plan, ny, nz, ncomp, in, pitch, dst, tw, wpost, stream, rb);
      default: break;
    }
  }
  return launch_x_c2r_c<T, 0>(plan, ny, nz, ncomp, in, pitch, dst, tw, wpost, stream, rb);
}

// 32 points per thread (one exchange per transform) for n = 512 / 1024 in float, in the passes where it
// measured fastest on B200 (profiles/r01_fft_tuning.md): n = 1024 all three, n = 512 the forward and the
// fused pass
constexpr bool sb_use_p32(int mode, int log2n) {
  return (log2n == 10 && mode <= 2) || (log2n == 9 && mode <= 1);
}

template <typename T, int MODE, int LOG2N>
static int launch_strided32(const C2<T>* in, const SbLines& lin, C2<T>* out, const SbLines& lout,
                            const C2<T>* tw, const SbGreensTable<T>& gt, void* stream) {
  constexpr int LINES = SB_P32_LINES(LOG2N), NT = LINES * ((1 << LOG2N) / SB_FFT_P32);
  const size_t smem = sizeof(C2<T>) * (size_t)LINES * SbFft32C<LOG2N>::npad;
  const dim3 grid((unsigned)((lin.inner + LINES - 1) / LINES), (unsigned)lin.n1, (unsigned)lin.n2);
  SB_KERNEL_ATTR_SMEM((sb_fft_strided32_kernel<T, MODE, LOG2N, LINES>), smem);
  SB_LAUNCH_COOP((sb_fft_strided32_kernel<T, MODE, LOG2N, LINES>), grid, dim3(NT), smem, stream, in, lin, out, lout,
                 tw, gt);
  SB_CHECK_LAUNCH("fft_strided32");
  return 0;
}

template <typename T, int MODE, int LOG2N>
static int launch_strided_c(const SbFftPlan& plan, const C2<T>* in, const SbLines& lin, C2<T>* out,
                            const SbLines& lout, const C2<T>* tw, const SbGreensTable<T>& gt, void* stream) {
  constexpr int LINES = LOG2N > 0 ? sb_strided_lines<T>(LOG2N, MODE) : 0;
  if constexpr (sizeof(T) == 4 && sb_use_p32(MODE, LOG2N)) {
    return launch_strided32<T, MODE, LOG2N>(in, lin, out, lout, tw, gt, stream);
  } else {
    const int lb = LOG2N > 0 ? LINES : lines_per_block_for(plan.threads, sizeof(T), true);
    const size_t smem = (size_t)lb * sb_fft_npad(plan.n) * sizeof(C2<T>);
    int lb_shift = 0;
    while ((1 << lb_shift) < lb) ++lb_shift;
    const unsigned nib = (unsigned)((lin.inner + lb - 1) / lb);
    if constexpr (MODE == 1 && LOG2N > 0 && sizeof(T) == 4) {
      if (gt.g2) {
        // + 64 bytes per thread of staged Green's factors; grid (component, kx group, o1)
        const size_t smem2 = smem + (size_t)lb * plan.threads * 64;
        const dim3 grid2((unsigned)lin.n2, nib, (unsigned)lin.n1);
        SB_KERNEL_ATTR_SMEM((sb_fft_strided_kernel<T, MODE, LOG2N, LINES, true>), smem2);
        SB_LAUNCH_COOP((sb_fft_strided_kernel<T, MODE, LOG2N, LINES, true>), grid2, dim3(lb * plan.threads), smem2,
                       stream, plan, lb_shift, in, lin, out, lout, tw, gt);
        SB_CHECK_LAUNCH("fft_strided");
        return 0;
      }
    }
    const dim3 grid(nib, (unsigned)lin.n1, (unsigned)lin.n2);
    SB_KERNEL_ATTR_SMEM((sb_fft_strided_kernel<T, MODE, LOG2N, LINES, false>), smem);
    SB_LAUNCH_COOP((sb_fft_strided_kernel<T, MODE, LOG2N, LINES, false>), grid, dim3(lb * plan.threads), smem, stream,
                   plan, lb_shift, in, lin, out, lout, tw, gt);
    SB_CHECK_LAUNCH("fft_strided");
    return 0;
  }
}
template <typename T, int MODE>
static int launch_strided(const SbFftPlan& plan, const C2<T>* in, const SbLines& lin, C2<T>* out,
                          const SbLines& lout, const C2<T>* tw, const SbGreensTable<T>& gt, void* stream) {
  if constexpr (MODE != 3) {  // compile-time specialised lengths (float: 256..2048, double: 256..1024)
    switch (plan.log2n) {
      case 8: return launch_strided_c<T, MODE, 8>(plan, in, lin, out, lout, tw, gt, stream);
      case 9: return launch_strided_c<T, MODE, 9>(plan, in, lin, out, lout, tw, gt, stream);
      case 10: return launch_strided_c<T, MODE, 10>(plan, in, lin, out, lout, tw, gt, stream);
      case 11:
        if constexpr (sizeof(T) == 4) return launch_strided_c<T, MODE, 11>(plan, in, lin, out, lout, tw, gt, stream);
        break;
      default: break;
    }
  }
  return launch_strided_c<T, MODE, 0>(plan, in, lin, out, lout, tw, gt, stream);
}

template <int LOG2N>
static int launch_zconvw(C2<float>* B, int ncomp, int ng, int nky, const C2<float>* tw, const float* g3,
                         int n1_full, int* tile_counter, void* stream) {
  using Z = SbZw<LOG2N>;
  SB_REQUIRE(tile_counter != nullptr, "fft_zconvw: no tile counter");
  sb_memset_async(tile_counter, 0, sizeof(int), stream);
  SB_KERNEL_ATTR_SMEM((sb_fft_zconvw_kernel<LOG2N>), Z::smem);
  const long long ntiles = (long long)ncomp * ng * nky;
  long long resident = 148LL * Z::BLOCKS;
#ifndef SB200_EMU
  {
    static int sms = 0, per_sm = 0;
    if (sms == 0) {
      int dev = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sb_fft_zconvw_kernel<LOG2N>, Z::NT, Z::smem);
      if (per_sm < 1) per_sm = 1;
    }
    resident = (long long)sms * per_sm;
  }
#else
  resident = 3;  // a few persistent "blocks", several tiles each
#endif
  const unsigned grid = (unsigned)(ntiles < resident ? ntiles : resident);
  SB_LAUNCH_COOP((sb_fft_zconvw_kernel<LOG2N>), dim3(grid), dim3(Z::NT), Z::smem, stream, B, (int)ntiles, ncomp, ng,
                 nky, tw, g3, n1_full, tile_counter);
  SB_CHECK_LAUNCH("fft_zconvw");
  return 0;
}
// fused z pass on the tile-contiguous layout (float, 2nz = 512 / 1024: SbFftState::zconv)
template <typename T>
static int launch_zconv(int log2n, C2<T>* B, int ncomp, int ng, int nky, const C2<T>* tw, const T* g2, int n1_full,
                        int* tile_counter, void* stream) {
  if constexpr (sizeof(T) == 4) {
    if (log2n == 9) return launch_zconvw<9>(B, ncomp, ng, nky, tw, g2, n1_full, tile_counter, stream);
    if (log2n == 10) return launch_zconvw<10>(B, ncomp, ng, nky, tw, g2, n1_full, tile_counter, stream);
  }
  sb_set_error("fft_zconv: unsupported transform length");
  return -1;
}

template <typename T>
static int fft_create_t(sb200_poisson* p, void* stream) {
  auto* st = new SbFftState<T>();
  p->backend_state = st;
  const int nz = p->nz, ny = p->ny, nx = p->nx;
  SB_REQUIRE(sb_fft_make_plan(nx, &st->px) == 0 && sb_fft_make_plan(2 * ny, &st->py) == 0 &&
                 (p->dim == 2 || sb_fft_make_plan(2 * nz, &st->pz) == 0),
             "fft backend needs power-of-two grid sizes (nx >= 16, ny >= 8, nz >= 8)");
  SB_REQUIRE(nx <= 4096 && ny <= 2048 && nz <= 2048, "fft backend: grid too large for one line per block");
  st->P = nx + 2;
  const long long P = st->P;
  st->twx = make_twiddles<T>(nx, nx, (double)nx, stream);
  st->wpost = make_twiddles<T>(nx, nx, 2.0 * nx, stream);
  st->twy = make_twiddles<T>(2 * ny, 2 * ny, 2.0 * ny, stream);
  if (p->dim == 3) st->twz = make_twiddles<T>(2 * nz, 2 * nz, 2.0 * nz, stream);
  SB_REQUIRE(st->twx && st->wpost && st->twy && (p->dim == 2 || st->twz), "fft backend: twiddle allocation");
  if (p->nranks > 1) {
    SB_REQUIRE(p->dim == 3, "fft backend: slab decomposition is implemented for 3D grids");
    SB_REQUIRE(p->nranks == 2 || p->nranks == 4 || p->nranks == 8,
               "fft backend: slab decomposition needs 2, 4 or 8 ranks");
    SB_REQUIRE(nz % p->nranks == 0 && nz / p->nranks >= 2 * p->gs, "fft backend: nz must split into slabs");
  }
  const SbKxSide kx = sb_kx_side(p, 3);
  const size_t a_bytes = p->nranks == 1 ? sizeof(C2<T>) * 3 * (size_t)(p->dim == 3 ? nz : 1) * ny * P : 0;
  st->ng = (kx.inner + 7) / 8;
  st->zconv = sizeof(T) == 4 && p->dim == 3 && (st->pz.log2n == 9 || st->pz.log2n == 10);
  if (st->zconv) SB_REQUIRE(SB_DEV_ALLOC(st->tile_counter, 64), "fft backend: cannot allocate the tile counter");
  // B: tile-contiguous (zconv) or [c][nz][2ny][pitch]
  const size_t b_bytes = p->dim != 3 ? 0
                         : sizeof(C2<T>) * 3 * (size_t)nz * 2 * ny * (st->zconv ? 8LL * st->ng : kx.pitch);
  const size_t g_bytes = sizeof(T) * (p->dim == 3 ? (nz + 1) : 1) * (ny + 1) * P;
  if (a_bytes) SB_REQUIRE(SB_DEV_ALLOC(st->A, a_bytes), "fft backend: cannot allocate x-pass buffer");
  if (b_bytes) SB_REQUIRE(SB_DEV_ALLOC(st->B, b_bytes), "fft backend: cannot allocate y-pass buffer");
  // (the padding lines of the last kx group are transformed along with the others: keep them finite)
  if (b_bytes && st->zconv) sb_memset_async(st->B, 0, b_bytes, stream);
  SB_REQUIRE(SB_DEV_ALLOC(st->G, g_bytes), "fft backend: cannot allocate Green's table");
  st->bytes = a_bytes + b_bytes + g_bytes;

  // ---- Green's spectrum: full (un-pruned) transform of G on the doubled grid, real part kept
  const long long n2z = p->dim == 3 ? 2LL * nz : 1, n2y = 2LL * ny;
  C2<T>* full = nullptr;
  SB_REQUIRE(SB_DEV_ALLOC(full, sizeof(C2<T>) * n2z * n2y * P), "fft backend: cannot allocate Green's scratch");
  GreensRows<T> gl;
  void* lines_dev = nullptr;
  int e = sb_poisson_make_greens<T>(p, &gl.g, &lines_dev, stream);
  if (e) return e;
  gl.ny = (int)n2y;
  // doubled rows have 2nx reals = nx complex points, none pruned
  if ((e = launch_x_r2c<T, GreensRows<T>, false>(st->px, (int)n2y, (int)n2z, 1, gl, full, P, st->twx, st->wpost,
                                                 stream)))
    return e;
  SbGreensTable<T> none{nullptr, 0, 0};
  {
    SbLines ly{nx + 1, (int)n2z, 1, n2y * P, 0, P};  // lines (kx, z), points along y
    if ((e = launch_strided<T, 3>(st->py, full, ly, full, ly, st->twy, none, stream))) return e;
  }
  if (p->dim == 3) {
    SbLines lz{nx + 1, (int)n2y, 1, P, 0, n2y * P};  // lines (kx, ky), points along z
    if ((e = launch_strided<T, 3>(st->pz, full, lz, full, lz, st->twz, none, stream))) return e;
  }
  double dxp = 1.0;
  for (int d = 0; d < p->dim; ++d) dxp *= p->dx;
  const double scale = dxp / ((double)n2z * (double)n2y * 2.0 * (double)nx);
  const long long hz1 = p->dim == 3 ? nz + 1 : 1;
  e = sb_launch_flat(hz1 * (ny + 1) * P, GreensExtractOp<T>{st->G, full, P, n2y, (long long)ny + 1, (T)scale},
                     stream, "greens_extract");
  if constexpr (sizeof(T) == 4) {
    if (!e && p->dim == 3 && st->pz.log2n >= 8 && st->pz.log2n <= 11) {
      // reordered copy for the fused z pass: line order for the z kernel (zconv), thread order for the
      // strided kernel (16 bins per thread)
      const int lines = st->zconv ? SB_P32_LINES(st->pz.log2n) : sb_strided_lines<T>(st->pz.log2n, 1);
      const int nib = (kx.inner + lines - 1) / lines;
      const long long count = (long long)(ny + 1) * nib * lines * 2 * nz;  // (both orders: n floats per line)
      SB_REQUIRE(SB_DEV_ALLOC(st->G2, sizeof(T) * count), "fft backend: cannot allocate the thread-order table");
      st->bytes += sizeof(T) * count;
      e = sb_launch_flat(count, GreensThreadOrderOp<T>{st->G2, st->G, (long long)(ny + 1) * P, P, 2 * nz,
                                                       2 * nz / SB_FFT_R, lines, nib, (int)P, kx.kx0, kx.inner,
                                                       st->zconv},
                         stream, "greens_thread_order");
    }
  }
  SB_STREAM_SYNC(stream);
  sb_poisson_free_greens_lines(lines_dev);
  SB_DEV_FREE(full);
  return e;
}

// ------------------------------------------ the three stages of a solve, single GPU and z-slab alike
// X is the x-pass output: the buffer A of a single-GPU solve, the caller's exchange buffers of a z-slab
// rank (SbKxSide).  Profiling marks 2 and 3 sit inside the spectral stage (they only record on a
// single-rank handle).
template <typename T>
static FieldRows<T> sb_field_rows(const sb200_poisson* p, const SbKxSide& kx, const void* f) {
  const long long my = p->ny + 2 * p->gs, mx = p->nx + 2 * p->gs;
  const long long vol = (p->dim == 3 ? kx.planes + 2LL * p->gs : 1) * my * mx;
  return FieldRows<T>{(T*)f, p->ny, p->gs, p->dim, my, mx, vol};
}
template <typename T>
static int fft_x_forward_t(sb200_poisson* p, const void* rhs, int ncomp, C2<T>* X, void* stream) {
  auto* st = (SbFftState<T>*)p->backend_state;
  const SbKxSide kx = sb_kx_side(p, ncomp);
  return launch_x_r2c<T, FieldRows<T>, true>(st->px, p->ny, kx.planes, ncomp, sb_field_rows<T>(p, kx, rhs), X,
                                             kx.pitch, st->twx, st->wpost, stream, kx.rb);
}
template <typename T>
static int fft_spectral_t(sb200_poisson* p, C2<T>* X, int ncomp, void* stream) {
  auto* st = (SbFftState<T>*)p->backend_state;
  const SbKxSide kx = sb_kx_side(p, ncomp);
  const int nz = p->nz, ny = p->ny;
  const long long P = st->P, pitch = kx.pitch;
  SbGreensTable<T> none{nullptr, 0, 0};
  SbGreensTable<T> gt{st->G, (p->dim == 3 ? ny + 1LL : 1LL) * P, P, 2 * ny, 0};
  gt.g2 = st->G2;
  gt.kx0 = kx.kx0;
  gt.kx_last = (int)P - 1;
  int e;
  if (p->dim == 2) {  // fused forward / x Ghat / inverse along y, in place on X
    st->mark(2, stream);
    if ((e = launch_strided<T, 1>(st->py, X, kx.lx, X, kx.lx, st->twy, gt, stream))) return e;
    st->mark(3, stream);
    return 0;
  }
  // y forward X -> B, z pass in place on B, y inverse B -> X.  B is either tile-contiguous for the
  // persistent z kernel, Bt[c][kx group][ky][z][8] addressed through grouped lines, or B[c][z][ky][pitch]
  const long long nky = 2LL * ny, tile = (long long)nz * 8;
  SbLines lb{kx.inner, nz, ncomp, nky * pitch, nz * nky * pitch, pitch};
  if (st->zconv) {
    lb = SbLines{kx.inner, nz, ncomp, 8, st->ng * nky * tile, tile};
    lb.gsh = 3;
    lb.s_grp = nky * tile;
    lb.rot = 7;
  }
  if ((e = launch_strided<T, 0>(st->py, X, kx.lx, st->B, lb, st->twy, none, stream))) return e;
  st->mark(2, stream);
  if (st->zconv) {
    e = launch_zconv<T>(st->pz.log2n, st->B, ncomp, st->ng, (int)nky, st->twz, st->G2, 2 * ny, st->tile_counter,
                        stream);
  } else {  // lines (kx, ky, c), points along z
    SbLines lz{kx.inner, 2 * ny, ncomp, pitch, nz * nky * pitch, nky * pitch};
    e = launch_strided<T, 1>(st->pz, st->B, lz, st->B, lz, st->twz, gt, stream);
  }
  if (e) return e;
  st->mark(3, stream);
  return launch_strided<T, 2>(st->py, st->B, lb, X, kx.lx, st->twy, none, stream);
}
template <typename T>
static int fft_x_backward_t(sb200_poisson* p, void* solution, int ncomp, const C2<T>* X, void* stream) {
  auto* st = (SbFftState<T>*)p->backend_state;
  const SbKxSide kx = sb_kx_side(p, ncomp);
  return launch_x_c2r<T>(st->px, p->ny, kx.planes, ncomp, X, kx.pitch, sb_field_rows<T>(p, kx, solution), st->twx,
                         st->wpost, stream, kx.rb);
}

template <typename T>
static int fft_solve_t(sb200_poisson* p, void* solution, const void* rhs, int ncomp, void* stream) {
  auto* st = (SbFftState<T>*)p->backend_state;
  SB_REQUIRE(ncomp >= 1 && ncomp <= 3, "poisson_solve: ncomp must be 1..3");
  int e;
  st->mark(0, stream);
  if ((e = fft_x_forward_t<T>(p, rhs, ncomp, st->A, stream))) return e;
  st->mark(1, stream);
  if ((e = fft_spectral_t<T>(p, st->A, ncomp, stream))) return e;
  st->mark(4, stream);
  e = fft_x_backward_t<T>(p, solution, ncomp, st->A, stream);
  st->mark(5, stream);
  st->have_times = st->profile && e == 0;
  return e;
}

template <typename T>
static int fft_set_profiling_t(sb200_poisson* p, int enable) {
  auto* st = (SbFftState<T>*)p->backend_state;
#ifndef SB200_EMU
  if (enable && !st->ev[0])
    for (auto& ev : st->ev) SB_REQUIRE(cudaEventCreate(&ev) == cudaSuccess, "poisson profiling: cudaEventCreate");
#endif
  st->profile = enable != 0;
  st->have_times = false;
  return 0;
}
template <typename T>
static int fft_last_stage_ms_t(sb200_poisson* p, float* ms_out, int n) {
  auto* st = (SbFftState<T>*)p->backend_state;
  SB_REQUIRE(st->have_times, "poisson profiling: no profiled solve yet");
  for (int i = 0; i < n && i < 5; ++i) {
#ifndef SB200_EMU
    if (i == 0) SB_REQUIRE(cudaEventSynchronize(st->ev[5]) == cudaSuccess, "poisson profiling: event sync");
    SB_REQUIRE(cudaEventElapsedTime(&ms_out[i], st->ev[i], st->ev[i + 1]) == cudaSuccess,
               "poisson profiling: elapsed time");
#else
    ms_out[i] = 0.f;
#endif
  }
  return 0;
}
extern "C" int sb200_poisson_set_profiling(sb200_poisson_t* p, int enable) {
  SB_REQUIRE(p && p->backend == 1 && p->backend_state && p->nranks == 1,
             "poisson profiling needs a single-rank handle of the fft backend");
  SB_DISPATCH_DTYPE(p->dtype, return fft_set_profiling_t<T>(p, enable));
}
extern "C" int sb200_poisson_last_stage_ms(sb200_poisson_t* p, float* ms_out, int n) {
  SB_REQUIRE(p && p->backend == 1 && p->backend_state && ms_out && n >= 1,
             "poisson profiling needs a handle of the fft backend");
  SB_DISPATCH_DTYPE(p->dtype, return fft_last_stage_ms_t<T>(p, ms_out, n));
}

template <typename T>
static void fft_destroy_t(sb200_poisson* p) {
  auto* st = (SbFftState<T>*)p->backend_state;
  if (!st) return;
  SB_DEV_FREE(st->twx);
  SB_DEV_FREE(st->twy);
  if (st->twz) SB_DEV_FREE(st->twz);
  SB_DEV_FREE(st->wpost);
  if (st->A) SB_DEV_FREE(st->A);
  if (st->B) SB_DEV_FREE(st->B);
  if (st->G) SB_DEV_FREE(st->G);
  if (st->G2) SB_DEV_FREE(st->G2);
  if (st->tile_counter) SB_DEV_FREE(st->tile_counter);
#ifndef SB200_EMU
  for (auto& ev : st->ev)
    if (ev) cudaEventDestroy(ev);
#endif
  delete st;
  p->backend_state = nullptr;
}

int sb_poisson_fft_create(sb200_poisson* p, void* stream) {
  SB_DISPATCH_DTYPE(p->dtype, return fft_create_t<T>(p, stream));
}

// ------------------------------------------------------------------ z-slab entry points
// rank r of P holds planes [r nz/P, (r+1) nz/P).  The transpose happens where the data is smallest
// (2 W per cell instead of 4 W after the y pass):
//   forward : x r2c of the local planes, written as P blocks of kxl = ceil((nx+1)/P) kx bins, one
//             per destination rank:                      S[kxb][c][zl][y][kx_in]
//   all-to-all -> every rank owns its kx block of ALL planes: R[zb][c][zl][y][kx_in]
//   spectral: y forward R -> B[c][z][ky][kx_in], fused z pass in place on B (Green's table columns
//             kx0 + kx_in), y inverse B -> R (same blocked-by-z layout)
//   all-to-all back, backward: x c2r of the local planes from S.
// The three stages are the ones of the single-GPU solve (fft_solve_t) on the caller's buffers.
// Bins beyond nx (the padding of the last block) are never written: the buffers must be
// zero-initialised once by the caller.
static int slab_check(const sb200_poisson* p, int ncomp) {
  SB_REQUIRE(p && p->backend == 1 && p->nranks > 1 && p->backend_state,
             "poisson slab entry points need a distributed handle of the fft backend");
  SB_REQUIRE(ncomp >= 1 && ncomp <= 3, "poisson slab: ncomp must be 1..3");
  return 0;
}
extern "C" int64_t sb200_poisson_slab_buffer_bytes(const sb200_poisson_t* p, int ncomp) {
  if (!p || p->nranks < 1) return 0;
  const int64_t w = p->dtype == SB200_F32 ? 4 : 8;
  const int64_t kxl = sb_slab_kxl(p->nx, p->nranks);
  return 2 * w * ncomp * (int64_t)(p->nz / p->nranks) * p->ny * kxl * p->nranks;
}
extern "C" int sb200_poisson_slab_forward(sb200_poisson_t* p, const void* rhs, int ncomp, void* send_buf,
                                          void* stream) {
  if (int e = slab_check(p, ncomp)) return e;
  SB_DISPATCH_DTYPE(p->dtype, return fft_x_forward_t<T>(p, rhs, ncomp, (C2<T>*)send_buf, stream));
}
extern "C" int sb200_poisson_slab_spectral(sb200_poisson_t* p, void* recv_buf, int ncomp, void* stream) {
  if (int e = slab_check(p, ncomp)) return e;
  SB_DISPATCH_DTYPE(p->dtype, return fft_spectral_t<T>(p, (C2<T>*)recv_buf, ncomp, stream));
}
extern "C" int sb200_poisson_slab_backward(sb200_poisson_t* p, void* solution, int ncomp, const void* send_buf,
                                           void* stream) {
  if (int e = slab_check(p, ncomp)) return e;
  SB_DISPATCH_DTYPE(p->dtype, return fft_x_backward_t<T>(p, solution, ncomp, (const C2<T>*)send_buf, stream));
}
int sb_poisson_fft_destroy(sb200_poisson* p) {
  if (p->dtype == SB200_F32) fft_destroy_t<float>(p); else fft_destroy_t<double>(p);
  return 0;
}
int sb_poisson_fft_solve(sb200_poisson* p, void* solution, const void* rhs, int ncomp, void* stream) {
  SB_DISPATCH_DTYPE(p->dtype, return fft_solve_t<T>(p, solution, rhs, ncomp, stream));
}
int64_t sb_poisson_fft_bytes(const sb200_poisson* p) {
  if (!p->backend_state) return 0;
  return p->dtype == SB200_F32 ? (int64_t)((SbFftState<float>*)p->backend_state)->bytes
                               : (int64_t)((SbFftState<double>*)p->backend_state)->bytes;
}
extern "C" int sb200_poisson_fft_available(void) { return 1; }
