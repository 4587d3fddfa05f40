// In-kernel FFT building blocks for the pruned Poisson pipeline.
//
// A line of length n = 2^k is transformed by T = n/16 threads; every thread keeps 16
// complex points in registers at positions  t + p*T  (p = 0..15).  That position set is the
// same for every Stockham stage, so global loads, global stores and the shared-memory
// re-reads are all unit-stride across threads, and zero-padding pruning is "skip p >= 8".
// Stages of radix 16/8/4/2 run entirely in registers; between stages the line is exchanged
// through (padded) shared memory.  Index algebra prototyped in tools/fft_prototype.py.
#pragma once
#include "sb200_rt.h"

template <typename T>
struct alignas(2 * sizeof(T)) C2 {
  T x, y;
};

// device table W[k] = exp(-2 pi i k / denom), k < count (poisson_fft.cu); nullptr when the allocation fails
template <typename T>
C2<T>* make_twiddles(int n, int count, double denom, void* stream);

template <typename T>
SB_HD C2<T> cmul(C2<T> a, C2<T> b) {
  return C2<T>{a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x};
}
template <typename T>
SB_HD C2<T> cadd(C2<T> a, C2<T> b) { return C2<T>{a.x + b.x, a.y + b.y}; }
template <typename T>
SB_HD C2<T> csub(C2<T> a, C2<T> b) { return C2<T>{a.x - b.x, a.y - b.y}; }
template <typename T>
SB_HD C2<T> cscale(C2<T> a, T s) { return C2<T>{a.x * s, a.y * s}; }
template <typename T>
SB_HD C2<T> cconj(C2<T> a) { return C2<T>{a.x, -a.y}; }
// conj(a) * s
template <typename T>
SB_HD C2<T> cscale_conj(C2<T> a, T s) { return C2<T>{a.x * s, a.y * -s}; }
// multiply by -i  (forward quarter turn)
template <typename T>
SB_HD C2<T> cmul_mi(C2<T> a) { return C2<T>{a.y, -a.x}; }

#if defined(__CUDACC__) && !defined(SB200_EMU)
// float complex arithmetic on the packed sm_100 FP32 forms (add/sub/mul/fma .f32x2 -> FADD2 /
// FMUL2 / FFMA2): one issue slot per complex add, two per complex multiply.  ptxas folds the lane
// swaps, negations and scalar broadcasts below into operand modifiers (.LO_HI, .NP, .F32), so
// cconj / cmul_mi cost nothing.  FP32 lane throughput is unchanged (tools/ubench/f32x2.cu), the
// gain is issue slots for the address / shared-memory / load instructions between the butterflies.
#define SB_PACKED_F32 1
typedef unsigned long long sb_u64;
SB_D sb_u64 sb_pk(float lo, float hi) {
  sb_u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
SB_D C2<float> sb_up(sb_u64 v) {
  C2<float> r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
  return r;
}
SB_D sb_u64 sb_add2(sb_u64 a, sb_u64 b) {
  sb_u64 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
SB_D sb_u64 sb_sub2(sb_u64 a, sb_u64 b) {
  sb_u64 d;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
SB_D sb_u64 sb_mul2(sb_u64 a, sb_u64 b) {
  sb_u64 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
SB_D sb_u64 sb_fma2(sb_u64 a, sb_u64 b, sb_u64 c) {
  sb_u64 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
SB_HD C2<float> cadd(C2<float> a, C2<float> b) {
#ifdef __CUDA_ARCH__
  return sb_up(sb_add2(sb_pk(a.x, a.y), sb_pk(b.x, b.y)));
#else
  return C2<float>{a.x + b.x, a.y + b.y};
#endif
}
SB_HD C2<float> csub(C2<float> a, C2<float> b) {
#ifdef __CUDA_ARCH__
  return sb_up(sb_sub2(sb_pk(a.x, a.y), sb_pk(b.x, b.y)));
#else
  return C2<float>{a.x - b.x, a.y - b.y};
#endif
}
SB_HD C2<float> cscale(C2<float> a, float s) {
#ifdef __CUDA_ARCH__
  return sb_up(sb_mul2(sb_pk(a.x, a.y), sb_pk(s, s)));
#else
  return C2<float>{a.x * s, a.y * s};
#endif
}
SB_HD C2<float> cscale_conj(C2<float> a, float s) {
#ifdef __CUDA_ARCH__
  return sb_up(sb_mul2(sb_pk(a.x, a.y), sb_pk(s, -s)));
#else
  return C2<float>{a.x * s, a.y * -s};
#endif
}
SB_HD C2<float> cmul(C2<float> a, C2<float> b) {
#ifdef __CUDA_ARCH__
  // (ax bx - ay by, ay bx + ax by) = (ax, ay) * (bx, bx) + (ay, ax) * (-by, by)
  return sb_up(sb_fma2(sb_pk(a.x, a.y), sb_pk(b.x, b.x), sb_mul2(sb_pk(a.y, a.x), sb_pk(-b.y, b.y))));
#else
  return C2<float>{a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x};
#endif
}
#endif

#define SB_FFT_R 16        // points per thread
#define SB_FFT_MAXSTAGES 4

struct SbFftPlan {
  int n;        // transform length (power of two, >= 16)
  int log2n;
  int threads;  // n / 16 threads per line
  int nstages;
  int radix[SB_FFT_MAXSTAGES];
};

static inline int sb_fft_make_plan(int n, SbFftPlan* p) {
  if (n < 16 || (n & (n - 1))) return -1;
  p->n = n;
  p->log2n = 0;
  while ((1 << p->log2n) < n) ++p->log2n;
  p->threads = n / SB_FFT_R;
  p->nstages = 0;
  int m = n;
  while (m > 1) {
    int r = m >= 16 ? 16 : m;
    if (p->nstages >= SB_FFT_MAXSTAGES) return -1;
    p->radix[p->nstages++] = r;
    m /= r;
  }
  return 0;
}

// ---------------------------------------------------------------- small DFTs (forward)
template <typename T>
SB_D void dft2(C2<T>& a, C2<T>& b) {
  const C2<T> s = cadd(a, b), d = csub(a, b);
  a = s;
  b = d;
}
template <typename T>
SB_D void dft4(C2<T>& a0, C2<T>& a1, C2<T>& a2, C2<T>& a3) {
  const C2<T> t0 = cadd(a0, a2), t1 = csub(a0, a2), t2 = cadd(a1, a3), t3 = cmul_mi(csub(a1, a3));
  a0 = cadd(t0, t2);
  a1 = cadd(t1, t3);
  a2 = csub(t0, t2);
  a3 = csub(t1, t3);
}
// a[0..R) -> DFT in natural order, R in {2,4,8,16}
template <typename T, int R>
SB_D void dft_small(C2<T>* a) {
  if (R == 2) {
    dft2(a[0], a[1]);
  } else if (R == 4) {
    dft4(a[0], a[1], a[2], a[3]);
  } else if (R == 8) {
    // 8 = 4 (inner, over n1, stride 2) x 2 (outer, over n2)
    const T h = T(0.70710678118654752440);
    C2<T> e[4] = {a[0], a[2], a[4], a[6]}, o[4] = {a[1], a[3], a[5], a[7]};
    dft4(e[0], e[1], e[2], e[3]);
    dft4(o[0], o[1], o[2], o[3]);
    // twiddle W8^k1 on the odd branch
    o[1] = cscale(cadd(o[1], cmul_mi(o[1])), h);         // (1 - i)/sqrt2
    o[2] = cmul_mi(o[2]);
    o[3] = cscale(csub(cmul_mi(o[3]), o[3]), h);         // (-1 - i)/sqrt2
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      a[k] = cadd(e[k], o[k]);
      a[k + 4] = csub(e[k], o[k]);
    }
  } else {
    // 16 = 4 (inner over n1, stride 4) x 4 (outer over n2); X[k1 + 4 k2]
    const T c1 = T(0.92387953251128675613), s1 = T(0.38268343236508977173);
    const T h = T(0.70710678118654752440);
    C2<T> b[4][4];  // b[n2][k1]
#pragma unroll
    for (int n2 = 0; n2 < 4; ++n2) {
      b[n2][0] = a[n2];
      b[n2][1] = a[n2 + 4];
      b[n2][2] = a[n2 + 8];
      b[n2][3] = a[n2 + 12];
      dft4(b[n2][0], b[n2][1], b[n2][2], b[n2][3]);
    }
    // twiddles W16^(n2*k1) = exp(-2 pi i n2 k1 / 16)
    const C2<T> w1{c1, -s1}, w2{h, -h}, w3{s1, -c1}, w6{-h, -h}, w9{-c1, s1};
    b[1][1] = cmul(b[1][1], w1);
    b[1][2] = cmul(b[1][2], w2);
    b[1][3] = cmul(b[1][3], w3);
    b[2][1] = cmul(b[2][1], w2);
    b[2][2] = cmul_mi(b[2][2]);  // W16^4 = -i
    b[2][3] = cmul(b[2][3], w6);
    b[3][1] = cmul(b[3][1], w3);
    b[3][2] = cmul(b[3][2], w6);
    b[3][3] = cmul(b[3][3], w9);
#pragma unroll
    for (int k1 = 0; k1 < 4; ++k1) {
      dft4(b[0][k1], b[1][k1], b[2][k1], b[3][k1]);
      a[k1] = b[0][k1];
      a[k1 + 4] = b[1][k1];
      a[k1 + 8] = b[2][k1];
      a[k1 + 12] = b[3][k1];
    }
  }
}

// ------------------------------------------------------------------ shared memory view
// Element i of a line lives at padded position i + (i >> 4) (one pad per 16 elements keeps
// the radix-16 scatter conflict-free).  LINE_FASTEST interleaves the lines of a block
// (element-major) so that strided passes read/write whole line groups contiguously; the
// number of lines per block is a power of two there (shift `ls`).
SB_HD int sb_fft_npad(int n) { return n + (n >> 4) + 1; }

template <typename T, bool LINE_FASTEST>
struct SbSmemLine {
  C2<T>* base;  // points at element 0 of this thread's line
  int ls;       // log2(lines per block) when LINE_FASTEST, else 0
  SB_D C2<T>& at_padded(int ip) const { return base[LINE_FASTEST ? (ip << ls) : ip]; }
  SB_D C2<T>& at(int i) const { return at_padded(i + (i >> 4)); }
};
template <typename T, bool LINE_FASTEST>
SB_D SbSmemLine<T, LINE_FASTEST> sb_smem_line(C2<T>* sm, int l, int lines_shift, int npad) {
  SbSmemLine<T, LINE_FASTEST> s;
  s.base = sm + (LINE_FASTEST ? l : l * npad);
  s.ls = LINE_FASTEST ? lines_shift : 0;
  return s;
}

// twiddles w^1..w^(R-1) of one butterfly from log2(R) exact table entries (w^1, w^2, w^4, w^8);
// the rest are products of at most three of them.
template <typename T, int R>
SB_D void sb_twiddle_apply(C2<T>* a, const C2<T>* __restrict__ tw, int step) {
  const C2<T> w1 = tw[step];
  a[1] = cmul(a[1], w1);
  if (R >= 4) {
    const C2<T> w2 = tw[2 * step];
    const C2<T> w3 = cmul(w1, w2);
    a[2] = cmul(a[2], w2);
    a[3] = cmul(a[3], w3);
    if (R >= 8) {
      const C2<T> w4 = tw[4 * step];
      const C2<T> w5 = cmul(w1, w4), w6 = cmul(w2, w4), w7 = cmul(w3, w4);
      a[4] = cmul(a[4], w4);
      a[5] = cmul(a[5], w5);
      a[6] = cmul(a[6], w6);
      a[7] = cmul(a[7], w7);
      if (R >= 16) {
        const C2<T> w8 = tw[8 * step];
        a[8] = cmul(a[8], w8);
        a[9] = cmul(a[9], cmul(w1, w8));
        a[10] = cmul(a[10], cmul(w2, w8));
        a[11] = cmul(a[11], cmul(w3, w8));
        a[12] = cmul(a[12], cmul(w4, w8));
        a[13] = cmul(a[13], cmul(w5, w8));
        a[14] = cmul(a[14], cmul(w6, w8));
        a[15] = cmul(a[15], cmul(w7, w8));
      }
    }
  }
}

// Base twiddles (w^1, w^2, w^4, w^8: log2(R) of them) of one butterfly, loaded ahead of use.
template <int R>
struct SbTwBase {
  static constexpr int N = R == 16 ? 4 : R == 8 ? 3 : R == 4 ? 2 : 1;
};
template <typename T, int R>
SB_D void sb_twiddle_load(C2<T>* pw, const C2<T>* __restrict__ tw, int step) {
  pw[0] = tw[step];
  if (R >= 4) pw[1] = tw[2 * step];
  if (R >= 8) pw[2] = tw[4 * step];
  if (R >= 16) pw[3] = tw[8 * step];
}
template <typename T, int R>
SB_D void sb_twiddle_apply_base(C2<T>* a, const C2<T>* pw) {
  const C2<T> w1 = pw[0];
  a[1] = cmul(a[1], w1);
  if (R >= 4) {
    const C2<T> w2 = pw[1];
    const C2<T> w3 = cmul(w1, w2);
    a[2] = cmul(a[2], w2);
    a[3] = cmul(a[3], w3);
    if (R >= 8) {
      const C2<T> w4 = pw[2];
      const C2<T> w5 = cmul(w1, w4), w6 = cmul(w2, w4), w7 = cmul(w3, w4);
      a[4] = cmul(a[4], w4);
      a[5] = cmul(a[5], w5);
      a[6] = cmul(a[6], w6);
      a[7] = cmul(a[7], w7);
      if (R >= 16) {
        const C2<T> w8 = pw[3];
        a[8] = cmul(a[8], w8);
        a[9] = cmul(a[9], cmul(w1, w8));
        a[10] = cmul(a[10], cmul(w2, w8));
        a[11] = cmul(a[11], cmul(w3, w8));
        a[12] = cmul(a[12], cmul(w4, w8));
        a[13] = cmul(a[13], cmul(w5, w8));
        a[14] = cmul(a[14], cmul(w6, w8));
        a[15] = cmul(a[15], cmul(w7, w8));
      }
    }
  }
}

// One radix-R stage for the butterflies owned by thread t.
//   v[p] <-> element t + p*T.  Ns = 2^ns_shift = product of the radices already applied
//   (always a power of 16 here: non-final stages are radix 16).
// last == false (R == 16 only): results go to shared memory at their Stockham positions,
// the caller syncs and re-reads; last == true: results return to v[].
template <typename T, int R, bool LINE_FASTEST>
SB_D void sb_fft_stage(C2<T>* v, int t, int threads, int log2n, int ns_shift, bool last,
                       const C2<T>* __restrict__ tw, const SbSmemLine<T, LINE_FASTEST>& sl) {
  constexpr int M = SB_FFT_R / R;  // butterflies per thread
  constexpr int LOG2R = R == 16 ? 4 : R == 8 ? 3 : R == 4 ? 2 : 1;
  const int Ns = 1 << ns_shift;
#pragma unroll
  for (int m = 0; m < M; ++m) {
    C2<T> a[R];
#pragma unroll
    for (int q = 0; q < R; ++q) a[q] = v[m + M * q];
    const int j = t + m * threads;
    const int k = j & (Ns - 1);
    if (ns_shift > 0) sb_twiddle_apply<T, R>(a, tw, k << (log2n - ns_shift - LOG2R));
    dft_small<T, R>(a);
    if (last) {
#pragma unroll
      for (int q = 0; q < R; ++q) v[m + M * q] = a[q];
    } else {
      // j0 = (j / Ns) * Ns * R + k ; element j0 + q*Ns ; padded: ip0 + q * stride
      const int j0 = ((j >> ns_shift) << (ns_shift + LOG2R)) + k;
      const int ip0 = j0 + (j0 >> 4);
      const int stride = ns_shift == 0 ? 1 : Ns + (Ns >> 4);
#pragma unroll
      for (int q = 0; q < R; ++q) sl.at_padded(ip0 + q * stride) = a[q];
    }
  }
}

// Forward FFT of the line held in v[] (all threads of the block must call this; the
// __syncthreads inside are block-wide).  On return v[p] = X[t + p*T].
template <typename T, bool LINE_FASTEST>
SB_D void sb_fft_forward(C2<T>* v, const SbFftPlan& plan, int t, const C2<T>* __restrict__ tw,
                         const SbSmemLine<T, LINE_FASTEST>& sl) {
  int ns_shift = 0;
  const int log2n = plan.log2n, Tn = plan.threads;
  for (int s = 0; s < plan.nstages; ++s) {
    const int r = plan.radix[s];
    const bool last = s == plan.nstages - 1;
    if (r == 16)
      sb_fft_stage<T, 16, LINE_FASTEST>(v, t, Tn, log2n, ns_shift, last, tw, sl);
    else if (r == 8)
      sb_fft_stage<T, 8, LINE_FASTEST>(v, t, Tn, log2n, ns_shift, true, tw, sl);
    else if (r == 4)
      sb_fft_stage<T, 4, LINE_FASTEST>(v, t, Tn, log2n, ns_shift, true, tw, sl);
    else
      sb_fft_stage<T, 2, LINE_FASTEST>(v, t, Tn, log2n, ns_shift, true, tw, sl);
    if (!last) {
      __syncthreads();
      if (Tn >= 16) {
        const int ip0 = t + (t >> 4), stride = Tn + (Tn >> 4);
#pragma unroll
        for (int p = 0; p < SB_FFT_R; ++p) v[p] = sl.at_padded(ip0 + p * stride);
      } else {
#pragma unroll
        for (int p = 0; p < SB_FFT_R; ++p) v[p] = sl.at(t + p * Tn);
      }
      __syncthreads();
    }
    ns_shift += r == 16 ? 4 : r == 8 ? 3 : r == 4 ? 2 : 1;
  }
}

// Unnormalised inverse through conj(fft(conj(x))).
template <typename T, bool LINE_FASTEST>
SB_D void sb_fft_inverse(C2<T>* v, const SbFftPlan& plan, int t, const C2<T>* __restrict__ tw,
                         const SbSmemLine<T, LINE_FASTEST>& sl) {
#pragma unroll
  for (int p = 0; p < SB_FFT_R; ++p) v[p].y = -v[p].y;
  sb_fft_forward<T, LINE_FASTEST>(v, plan, t, tw, sl);
#pragma unroll
  for (int p = 0; p < SB_FFT_R; ++p) v[p].y = -v[p].y;
}

// =========================================================================================
// Compile-time specialised transform: n = 2^LOG2N, LINES = lines per block (power of two) when
// LINE_FASTEST.  Every stride below is a constant, so shared-memory addresses fold into
// base + immediate and the 16-point register file never moves between code paths.
template <int LOG2N>
struct SbFftC {
  static constexpr int n = 1 << LOG2N;
  static constexpr int Tn = n / SB_FFT_R;
  static constexpr int nfull = LOG2N / 4;       // radix-16 stages
  static constexpr int rem = LOG2N % 4;         // final radix 2^rem stage (if any)
  static constexpr int npad = n + (n >> 4) + 1;
};

template <typename T, int LOG2N, bool LINE_FASTEST, int LINES>
struct SbFftLineC {
  using P = SbFftC<LOG2N>;
  static constexpr int MUL = LINE_FASTEST ? LINES : 1;
  // pointer to padded element 0 of local line l
  static SB_D C2<T>* line(C2<T>* sm, int l) { return sm + (LINE_FASTEST ? l : l * P::npad); }
  static SB_HD size_t smem_bytes() { return sizeof(C2<T>) * (size_t)LINES * P::npad; }
};

// base twiddles of the (16 / R) butterflies thread t runs in the radix-R stage that follows Ns points:
// issued BEFORE the exchange barriers in front of that stage, while the 16 data registers are dead
// (the points sit in shared memory), so the L1 / L2 latency of the table hides behind the exchange
template <typename T, int LOG2N, int R, int NS_SHIFT>
SB_D void sb_fft_stage_twiddles_c(C2<T>* pw, int t, const C2<T>* __restrict__ tw) {
  using P = SbFftC<LOG2N>;
  constexpr int M = SB_FFT_R / R;
  constexpr int LOG2R = R == 16 ? 4 : R == 8 ? 3 : R == 4 ? 2 : 1;
  constexpr int Ns = 1 << NS_SHIFT;
#pragma unroll
  for (int m = 0; m < M; ++m) {
    const int k = (t + m * P::Tn) & (Ns - 1);
    sb_twiddle_load<T, R>(pw + m * SbTwBase<R>::N, tw, k << (LOG2N - NS_SHIFT - LOG2R));
  }
}

template <typename T, int LOG2N, bool LINE_FASTEST, int LINES, int R, int NS_SHIFT, bool LAST>
SB_D void sb_fft_stage_c(C2<T> (&v)[SB_FFT_R], int t, const C2<T>* pw, C2<T>* sl) {
  using P = SbFftC<LOG2N>;
  constexpr int MUL = LINE_FASTEST ? LINES : 1;
  constexpr int M = SB_FFT_R / R;
  constexpr int LOG2R = R == 16 ? 4 : R == 8 ? 3 : R == 4 ? 2 : 1;
  constexpr int Ns = 1 << NS_SHIFT;
#pragma unroll
  for (int m = 0; m < M; ++m) {
    C2<T> a[R];
#pragma unroll
    for (int q = 0; q < R; ++q) a[q] = v[m + M * q];
    const int j = t + m * P::Tn;
    const int k = j & (Ns - 1);
    if constexpr (NS_SHIFT > 0) sb_twiddle_apply_base<T, R>(a, pw + m * SbTwBase<R>::N);
    dft_small<T, R>(a);
    if constexpr (LAST) {
#pragma unroll
      for (int q = 0; q < R; ++q) v[m + M * q] = a[q];
    } else {
      const int j0 = ((j >> NS_SHIFT) << (NS_SHIFT + LOG2R)) + k;
      C2<T>* dst = sl + (j0 + (j0 >> 4)) * MUL;
      constexpr int stride = (NS_SHIFT == 0 ? 1 : Ns + (Ns >> 4)) * MUL;
#pragma unroll
      for (int q = 0; q < R; ++q) dst[q * stride] = a[q];
    }
  }
}

// shared-memory re-read of the thread's 16 points (positions t + p*Tn)
template <typename T, int LOG2N, bool LINE_FASTEST, int LINES>
SB_D void sb_fft_reread_c(C2<T> (&v)[SB_FFT_R], int t, const C2<T>* sl) {
  using P = SbFftC<LOG2N>;
  constexpr int MUL = LINE_FASTEST ? LINES : 1;
  if constexpr (P::Tn >= 16) {
    const C2<T>* src = sl + (t + (t >> 4)) * MUL;
    constexpr int stride = (P::Tn + (P::Tn >> 4)) * MUL;
#pragma unroll
    for (int p = 0; p < SB_FFT_R; ++p) v[p] = src[p * stride];
  } else {
#pragma unroll
    for (int p = 0; p < SB_FFT_R; ++p) {
      const int i = t + p * P::Tn;
      v[p] = sl[(i + (i >> 4)) * MUL];
    }
  }
}

template <typename T, int LOG2N, bool LINE_FASTEST, int LINES>
SB_D void sb_fft_forward_c(C2<T> (&v)[SB_FFT_R], int t, const C2<T>* __restrict__ tw, C2<T>* sl) {
  using P = SbFftC<LOG2N>;
  static_assert(LOG2N >= 4 && LOG2N <= 12, "supported lengths: 16 .. 4096");
  constexpr int RLAST = 1 << P::rem;  // closing radix (1: none)
  C2<T> pw[8];                        // base twiddles of the next stage (at most 8 complex)
  // radix of the stage that follows `done` radix-16 stages
#define SB_NEXT_TWIDDLES(done)                                                                   \
  do {                                                                                           \
    if constexpr (P::nfull > (done))                                                             \
      sb_fft_stage_twiddles_c<T, LOG2N, 16, 4 * (done)>(pw, t, tw);                              \
    else if constexpr (P::rem > 0)                                                               \
      sb_fft_stage_twiddles_c<T, LOG2N, RLAST, 4 * (done)>(pw, t, tw);                           \
  } while (0)
  // stage 0
  if constexpr (P::nfull >= 1) {
    constexpr bool last = P::nfull == 1 && P::rem == 0;
    sb_fft_stage_c<T, LOG2N, LINE_FASTEST, LINES, 16, 0, last>(v, t, pw, sl);
    if constexpr (!last) {
      SB_NEXT_TWIDDLES(1);
      __syncthreads();
      sb_fft_reread_c<T, LOG2N, LINE_FASTEST, LINES>(v, t, sl);
      __syncthreads();
    }
  }
  if constexpr (P::nfull >= 2) {
    constexpr bool last = P::nfull == 2 && P::rem == 0;
    sb_fft_stage_c<T, LOG2N, LINE_FASTEST, LINES, 16, 4, last>(v, t, pw, sl);
    if constexpr (!last) {
      SB_NEXT_TWIDDLES(2);
      __syncthreads();
      sb_fft_reread_c<T, LOG2N, LINE_FASTEST, LINES>(v, t, sl);
      __syncthreads();
    }
  }
  if constexpr (P::nfull >= 3) {
    constexpr bool last = P::rem == 0;
    sb_fft_stage_c<T, LOG2N, LINE_FASTEST, LINES, 16, 8, last>(v, t, pw, sl);
    if constexpr (!last) {
      SB_NEXT_TWIDDLES(3);
      __syncthreads();
      sb_fft_reread_c<T, LOG2N, LINE_FASTEST, LINES>(v, t, sl);
      __syncthreads();
    }
  }
#undef SB_NEXT_TWIDDLES
  if constexpr (P::rem == 1) sb_fft_stage_c<T, LOG2N, LINE_FASTEST, LINES, 2, 4 * P::nfull, true>(v, t, pw, sl);
  if constexpr (P::rem == 2) sb_fft_stage_c<T, LOG2N, LINE_FASTEST, LINES, 4, 4 * P::nfull, true>(v, t, pw, sl);
  if constexpr (P::rem == 3) sb_fft_stage_c<T, LOG2N, LINE_FASTEST, LINES, 8, 4 * P::nfull, true>(v, t, pw, sl);
}

template <typename T, int LOG2N, bool LINE_FASTEST, int LINES>
SB_D void sb_fft_inverse_c(C2<T> (&v)[SB_FFT_R], int t, const C2<T>* __restrict__ tw, C2<T>* sl) {
#if defined(__CUDA_ARCH__)
  // launder the table pointer: in the fused forward/inverse kernel the compiler would otherwise keep
  // the forward transform's twiddles live in registers for re-use here (24 registers that cost a
  // resident block); re-loading them hits L1
  asm volatile("" : "+l"(tw));
#endif
#pragma unroll
  for (int p = 0; p < SB_FFT_R; ++p) v[p].y = -v[p].y;
  sb_fft_forward_c<T, LOG2N, LINE_FASTEST, LINES>(v, t, tw, sl);
#pragma unroll
  for (int p = 0; p < SB_FFT_R; ++p) v[p].y = -v[p].y;
}

// =========================================================================================
// 32 points per thread: n = 32 * m with m in {8, 16, 32} is ONE radix-32 stage, ONE shared-memory
// exchange and one radix-m stage (the 16-point variant above needs two exchanges for n >= 512).
// Half the shared-memory traffic and barriers per transform for the same FP32 work; the price is
// 64 data registers per thread (<= 128 registers, half the resident threads).  Lines are
// interleaved element-major (LINES per block) like the LINE_FASTEST layout above; element e sits at
// padded position e + (e >> 5), which keeps the radix-32 scatter (thread stride 33) and the re-read
// (unit thread stride) conflict-free for 64-bit accesses.
#define SB_FFT_P32 32

template <typename T>
SB_D void dft32(C2<T>* a) {
  // 32 = 2 x 16: E = DFT16(even), O = DFT16(odd), X[k] = E[k] + W32^k O[k], X[k+16] = E[k] - W32^k O[k]
  C2<T> e[16], o[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    e[k] = a[2 * k];
    o[k] = a[2 * k + 1];
  }
  dft_small<T, 16>(e);
  dft_small<T, 16>(o);
  constexpr double c[16] = {1.0, 0.98078528040323044913, 0.92387953251128675613, 0.83146961230254523708,
                            0.70710678118654752440, 0.55557023301960222474, 0.38268343236508977173,
                            0.19509032201612826785, 0.0, -0.19509032201612826785, -0.38268343236508977173,
                            -0.55557023301960222474, -0.70710678118654752440, -0.83146961230254523708,
                            -0.92387953251128675613, -0.98078528040323044913};
  constexpr double sn[16] = {0.0, 0.19509032201612826785, 0.38268343236508977173, 0.55557023301960222474,
                             0.70710678118654752440, 0.83146961230254523708, 0.92387953251128675613,
                             0.98078528040323044913, 1.0, 0.98078528040323044913, 0.92387953251128675613,
                             0.83146961230254523708, 0.70710678118654752440, 0.55557023301960222474,
                             0.38268343236508977173, 0.19509032201612826785};
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    C2<T> w;
    if (k == 0)
      w = o[0];
    else if (k == 8)
      w = cmul_mi(o[8]);
    else
      w = cmul(o[k], C2<T>{T(c[k]), T(-sn[k])});
    a[k] = cadd(e[k], w);
    a[k + 16] = csub(e[k], w);
  }
}

template <typename T, int R>
SB_D void dft_small32(C2<T>* a) {
  if constexpr (R == 32)
    dft32<T>(a);
  else
    dft_small<T, R>(a);
}

// twiddles w^1 .. w^(R-1) from the log2(R) base values w^1, w^2, w^4, (w^8, w^16)
template <typename T, int R>
SB_D void sb_twiddle_apply_base32(C2<T>* a, const C2<T>* pw) {
  if constexpr (R <= 16) {
    sb_twiddle_apply_base<T, R>(a, pw);
  } else {
    C2<T> w[16];  // w^0 .. w^15 (w[0] unused)
    w[1] = pw[0];
    w[2] = pw[1];
    w[3] = cmul(w[1], w[2]);
    w[4] = pw[2];
    w[5] = cmul(w[1], w[4]);
    w[6] = cmul(w[2], w[4]);
    w[7] = cmul(w[3], w[4]);
    w[8] = pw[3];
#pragma unroll
    for (int i = 1; i < 8; ++i) w[8 + i] = cmul(w[i], w[8]);
    const C2<T> w16 = pw[4];
    a[16] = cmul(a[16], w16);
#pragma unroll
    for (int i = 1; i < 16; ++i) {
      a[i] = cmul(a[i], w[i]);
      a[16 + i] = cmul(a[16 + i], cmul(w[i], w16));
    }
  }
}

template <int LOG2N>
struct SbFft32C {
  static constexpr int n = 1 << LOG2N;
  static constexpr int Tn = n / SB_FFT_P32;          // threads per line
  static constexpr int R2 = n / SB_FFT_P32;          // radix of the second stage (8, 16 or 32)
  static constexpr int M = SB_FFT_P32 / R2;          // second-stage butterflies per thread
  static constexpr int NB = R2 == 32 ? 5 : R2 == 16 ? 4 : 3;  // base twiddles per butterfly
  static constexpr int npad = n + (n >> 5) + 1;
  static_assert(LOG2N >= 8 && LOG2N <= 10, "32-point-per-thread transforms: n = 256, 512, 1024");
};

// forward transform of the line held in v[] (v[p] <-> element t + p Tn on entry and on return);
// sl = padded element 0 of this thread's line, lines interleaved LINES-wide
// TRAIL: barrier after the re-read, needed only when the exchange buffer is written again afterwards
template <typename T, int LOG2N, int LINES, bool TRAIL = true>
SB_D void sb_fft32_forward_c(C2<T> (&v)[SB_FFT_P32], int t, const C2<T>* __restrict__ tw, C2<T>* sl) {
  using P = SbFft32C<LOG2N>;
  dft32<T>(v);
  {
    C2<T>* dst = sl + (33 * t) * LINES;  // position 32 t + q, padded 33 t + q
#pragma unroll
    for (int q = 0; q < SB_FFT_P32; ++q) dst[q * LINES] = v[q];
  }
  // base twiddles of the second stage, in flight across the exchange (the data registers are dead)
  C2<T> pw[P::M * P::NB];
#pragma unroll
  for (int m = 0; m < P::M; ++m) {
    const int k = t + m * P::Tn;  // butterfly index j < 32 = Ns, twiddle W_n^(k q)
#pragma unroll
    for (int b = 0; b < P::NB; ++b) pw[m * P::NB + b] = tw[k << b];
  }
  __syncthreads();
#pragma unroll
  for (int p = 0; p < SB_FFT_P32; ++p) {
    // element t + p Tn; its padding (e >> 5) does not depend on t because t < Tn <= 32
    const int pad = (p * P::Tn) >> 5;
    v[p] = sl[(t + p * P::Tn + pad) * LINES];
  }
  if constexpr (TRAIL) __syncthreads();
#pragma unroll
  for (int m = 0; m < P::M; ++m) {
    C2<T> a[P::R2];
#pragma unroll
    for (int q = 0; q < P::R2; ++q) a[q] = v[m + P::M * q];
    sb_twiddle_apply_base32<T, P::R2>(a, pw + m * P::NB);
    dft_small32<T, P::R2>(a);
#pragma unroll
    for (int q = 0; q < P::R2; ++q) v[m + P::M * q] = a[q];
  }
}

template <typename T, int LOG2N, int LINES, bool TRAIL = true>
SB_D void sb_fft32_inverse_c(C2<T> (&v)[SB_FFT_P32], int t, const C2<T>* __restrict__ tw, C2<T>* sl) {
#if defined(__CUDA_ARCH__)
  asm volatile("" : "+l"(tw));  // see sb_fft_inverse_c
#endif
#pragma unroll
  for (int p = 0; p < SB_FFT_P32; ++p) v[p].y = -v[p].y;
  sb_fft32_forward_c<T, LOG2N, LINES, TRAIL>(v, t, tw, sl);
#pragma unroll
  for (int p = 0; p < SB_FFT_P32; ++p) v[p].y = -v[p].y;
}

// ------------------------------------------------------------------ one line per warp (float)
// The same 32-point-per-thread transform with the line's n / 32 threads INSIDE one warp (lanes t of a
// warp for n = 1024, half a warp for n = 512): the exchange between the two register stages is warp
// local, so the only synchronisation is __syncwarp and the warps of a block never wait for each other.
// The exchange buffer holds ONE float per element (real parts first, then the imaginary parts through the
// same words): half the shared memory of the complex exchange, 32-bit accesses at thread stride 33 /
// unit stride are conflict-free.

// DFT-16 of a[0..7] with a[8..15] = 0 (zero-padded line): the first radix-4 layer needs half its adds
template <typename T>
SB_D void dft16_upper_zero(C2<T>* a) {
  const T c1 = T(0.92387953251128675613), s1 = T(0.38268343236508977173);
  const T h = T(0.70710678118654752440);
  C2<T> b[4][4];  // b[n2][k1]
#pragma unroll
  for (int n2 = 0; n2 < 4; ++n2) {
    const C2<T> a0 = a[n2], a1 = a[n2 + 4], m = cmul_mi(a1);
    b[n2][0] = cadd(a0, a1);
    b[n2][1] = cadd(a0, m);
    b[n2][2] = csub(a0, a1);
    b[n2][3] = csub(a0, m);
  }
  const C2<T> w1{c1, -s1}, w2{h, -h}, w3{s1, -c1}, w6{-h, -h}, w9{-c1, s1};
  b[1][1] = cmul(b[1][1], w1);
  b[1][2] = cmul(b[1][2], w2);
  b[1][3] = cmul(b[1][3], w3);
  b[2][1] = cmul(b[2][1], w2);
  b[2][2] = cmul_mi(b[2][2]);
  b[2][3] = cmul(b[2][3], w6);
  b[3][1] = cmul(b[3][1], w3);
  b[3][2] = cmul(b[3][2], w6);
  b[3][3] = cmul(b[3][3], w9);
#pragma unroll
  for (int k1 = 0; k1 < 4; ++k1) {
    dft4(b[0][k1], b[1][k1], b[2][k1], b[3][k1]);
    a[k1] = b[0][k1];
    a[k1 + 4] = b[1][k1];
    a[k1 + 8] = b[2][k1];
    a[k1 + 12] = b[3][k1];
  }
}

// DFT-32 of a[0..15] with a[16..31] = 0 on entry (UPPER_ZERO), all 32 outputs
template <typename T, bool UPPER_ZERO>
SB_D void dft32_p(C2<T>* a) {
  if constexpr (!UPPER_ZERO) {
    dft32<T>(a);
  } else {
    C2<T> e[16], o[16];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      e[k] = a[2 * k];
      o[k] = a[2 * k + 1];
    }
    dft16_upper_zero<T>(e);
    dft16_upper_zero<T>(o);
    constexpr double c[16] = {1.0, 0.98078528040323044913, 0.92387953251128675613, 0.83146961230254523708,
                              0.70710678118654752440, 0.55557023301960222474, 0.38268343236508977173,
                              0.19509032201612826785, 0.0, -0.19509032201612826785, -0.38268343236508977173,
                              -0.55557023301960222474, -0.70710678118654752440, -0.83146961230254523708,
                              -0.92387953251128675613, -0.98078528040323044913};
    constexpr double sn[16] = {0.0, 0.19509032201612826785, 0.38268343236508977173, 0.55557023301960222474,
                               0.70710678118654752440, 0.83146961230254523708, 0.92387953251128675613,
                               0.98078528040323044913, 1.0, 0.98078528040323044913, 0.92387953251128675613,
                               0.83146961230254523708, 0.70710678118654752440, 0.55557023301960222474,
                               0.38268343236508977173, 0.19509032201612826785};
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      C2<T> w;
      if (k == 0)
        w = o[0];
      else if (k == 8)
        w = cmul_mi(o[8]);
      else
        w = cmul(o[k], C2<T>{T(c[k]), T(-sn[k])});
      a[k] = cadd(e[k], w);
      a[k + 16] = csub(e[k], w);
    }
  }
}

// scheduling fence on the 64 data registers: everything before it is complete and nothing after it has
// started, which keeps ptxas from interleaving two register stages (and spilling)
SB_D void sb_reg_fence(C2<float> (&v)[SB_FFT_P32]) {
#if defined(__CUDA_ARCH__)
#pragma unroll
  for (int p = 0; p < SB_FFT_P32; ++p) asm volatile("" : "+f"(v[p].x), "+f"(v[p].y));
#else
  (void)v;
#endif
}

template <int LOG2N>
struct SbFft32W {
  using P = SbFft32C<LOG2N>;
  // floats per exchange line: n + n/32 pads, rounded so that lines start on 16 bytes (they also stage the
  // line's Green's factors, a bulk copy) and, for n = 512 (two lines per warp), sit 16 banks apart
  static constexpr int XL = P::Tn == 32 ? P::n + P::n / 32 + 4 : P::n + P::n / 32;
  static_assert(XL % 4 == 0 && (P::Tn == 32 || (XL % 32) == 16), "exchange line stride");
};

// forward transform, v[p] <-> element t + p Tn on entry and on return; xl = this line's exchange floats
// (element e at padded position e + (e >> 5): scatter at thread stride 33, re-read at unit stride).
// UPPER_ZERO: v[16..31] are zero on entry (and need not be initialised).
template <int LOG2N, bool UPPER_ZERO>
SB_D void sb_fft32w_forward(C2<float> (&v)[SB_FFT_P32], int t, const C2<float>* __restrict__ tw, float* xl) {
  using P = SbFft32C<LOG2N>;
  dft32_p<float, UPPER_ZERO>(v);
  (void)tw;
  float* dst = xl + 33 * t;
  __syncwarp();  // the previous readers of this buffer are done
#pragma unroll
  for (int q = 0; q < SB_FFT_P32; ++q) dst[q] = v[q].x;
  __syncwarp();
#pragma unroll
  for (int p = 0; p < SB_FFT_P32; ++p) v[p].x = xl[t + p * P::Tn + ((p * P::Tn) >> 5)];
  __syncwarp();
#pragma unroll
  for (int q = 0; q < SB_FFT_P32; ++q) dst[q] = v[q].y;
  __syncwarp();
#pragma unroll
  for (int p = 0; p < SB_FFT_P32; ++p) v[p].y = xl[t + p * P::Tn + ((p * P::Tn) >> 5)];
}
// ... second register stage (after the exchange); split from the first so that the caller can reuse the
// exchange buffer in between
template <int LOG2N>
SB_D void sb_fft32w_second(C2<float> (&v)[SB_FFT_P32], int t, const C2<float>* __restrict__ tw) {
  using P = SbFft32C<LOG2N>;
#pragma unroll
  for (int m = 0; m < P::M; ++m) {
    C2<float> pw[P::NB];
    const int k = t + m * P::Tn;
#pragma unroll
    for (int b = 0; b < P::NB; ++b) pw[b] = tw[k << b];
    C2<float> a[P::R2];
#pragma unroll
    for (int q = 0; q < P::R2; ++q) a[q] = v[m + P::M * q];
    sb_twiddle_apply_base32<float, P::R2>(a, pw);
    dft_small32<float, P::R2>(a);
#pragma unroll
    for (int q = 0; q < P::R2; ++q) v[m + P::M * q] = a[q];
  }
}
