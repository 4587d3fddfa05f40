// Fused vorticity update: one streaming pass over (omega, u) instead of the reference's
// cross product + curl update + three diffusion-flux/add sweeps
// (reference simulator/flow/flow_simulators_mpi_3d.py:395-411):
//     buf    = u x omega                      (every cell)
//     omega2 = omega + p * curl(buf)          (cells the MPI wrapper writes)
//     out    = omega2 + d * lap7(omega2)      (same cells, zero flux on the physical ring)
// 2.5D scheme: a CTA owns a (TY x TX) tile of the (y,x) plane and marches along z; the
// cross product is staged on the tile + 2 halo cells, omega2 on tile + 1, both in rings of
// three planes in shared memory, so every input plane is read from HBM once (plus the
// in-plane halo overlap, served by L2) and the output written once: ~9 W per cell instead of
// 33 W.  Each thread owns a fixed set of cells of every region: shared/global offsets and the
// (y,x) part of the wrapper masks are computed once, the z part is uniform per plane, and the
// next plane's omega/u are prefetched into registers while the current one is processed.
#include "sb200_common.h"

template <int TY, int TX, int NT>
struct FusedTile {
  static constexpr int P2 = TX + 4, R2 = (TY + 4) * P2;  // tile + halo 2
  static constexpr int P1 = TX + 2, R1 = (TY + 2) * P1;  // tile + halo 1
  static constexpr int R0 = TY * TX;
  static constexpr int C2N = (R2 + NT - 1) / NT;  // cells per thread in each region
  static constexpr int C1N = (R1 + NT - 1) / NT;
  static constexpr int C0N = (R0 + NT - 1) / NT;
  // reals: buf ring 3 planes x 3 comps (R2), omega ring 2 x 3 (R1), omega2 ring 3 x 3 (R1)
  static constexpr int ELEMS = 9 * R2 + 6 * R1 + 9 * R1;
};

// (y,x) part of the support-1 wrapper mask:
//   bit0 = A: written whenever 1 <= z < mz-1           (x slabs, y slabs)
//   bit1 = B: written whenever z is in the interior / z-slab range
//   bit2 = inside the array, bit3 = on the physical ring because of y or x
SB_D int sb_yx_mask(const SbGeom& g, int y, int x) {
  if (y < 0 || y >= g.my || x < 0 || x >= g.mx) return 0;
  const int gs = g.gs;
  const bool xs = (x == gs) || (x == g.mx - gs - 1);
  const bool xi = x > gs && x < g.mx - gs - 1;
  const bool ys = (y == gs) || (y == g.my - gs - 1);
  const bool yi = y > gs && y < g.my - gs - 1;
  const bool yfull = y >= 1 && y < g.my - 1;
  const int w = gs + 1;
  const bool ring = (g.phys[4] && x < w) || (g.phys[5] && x >= g.mx - w) || (g.phys[2] && y < w) ||
                    (g.phys[3] && y >= g.my - w);
  return ((xs && yfull) || (xi && ys) ? 1 : 0) | (xi && yi ? 2 : 0) | 4 | (ring ? 8 : 0);
}

template <typename T, int TY, int TX, int NT>
__global__ void __launch_bounds__(NT)
    sb_vorticity_fused_kernel(SbGeom g, T* __restrict__ out, const T* __restrict__ w, const T* __restrict__ u,
                              T p, T d, int zchunk, int z_begin, int z_end) {
  using FT = FusedTile<TY, TX, NT>;
  SB_DYN_SMEM(smem_raw);
  T* sbuf = reinterpret_cast<T*>(smem_raw);  // [3][3][R2]
  T* sw1 = sbuf + 9 * FT::R2;                // [2][3][R1]
  T* sw2 = sw1 + 6 * FT::R1;                 // [3][3][R1]
  const int tid = threadIdx.x;
  const int y0 = blockIdx.y * TY, x0 = blockIdx.x * TX;
  const int zb = z_begin + blockIdx.z * zchunk;
  const int ze = zb + zchunk < z_end ? zb + zchunk : z_end;
  const long long vol = g.vol, plane = g.plane;
  const int zlo = g.phys[0] ? g.gs : 1, zhi = g.phys[1] ? g.mz - g.gs : g.mz - 1;
  const int zring_lo = g.phys[0] ? g.gs + 1 : 0, zring_hi = g.phys[1] ? g.mz - g.gs - 1 : g.mz;

  // ---- per-thread cell bookkeeping (z invariant)
  int a_goff[FT::C2N], a_j[FT::C2N];  // region 2: global (y,x) offset (-1 = none), region-1 slot (-1)
  int b_i[FT::C1N], b_m[FT::C1N];     // region 1: region-2 slot, mask
  int c_j[FT::C0N], c_goff[FT::C0N], c_m[FT::C0N];
#pragma unroll
  for (int k = 0; k < FT::C2N; ++k) {
    const int i = tid + k * NT;
    const int ry = i / FT::P2, rx = i - ry * FT::P2;
    const int y = y0 + ry - 2, x = x0 + rx - 2;
    const bool in = i < FT::R2 && y >= 0 && y < g.my && x >= 0 && x < g.mx;
    a_goff[k] = in ? y * g.mx + x : -1;
    a_j[k] = (i < FT::R2 && ry >= 1 && ry <= TY + 2 && rx >= 1 && rx <= TX + 2)
                 ? (ry - 1) * FT::P1 + (rx - 1)
                 : -1;
  }
#pragma unroll
  for (int k = 0; k < FT::C1N; ++k) {
    const int j = tid + k * NT;
    const int ry = j / FT::P1, rx = j - ry * FT::P1;
    b_i[k] = (ry + 1) * FT::P2 + (rx + 1);
    b_m[k] = j < FT::R1 ? sb_yx_mask(g, y0 + ry - 1, x0 + rx - 1) : 0;
  }
#pragma unroll
  for (int k = 0; k < FT::C0N; ++k) {
    const int c = tid + k * NT;
    const int ty = c / TX, tx = c - ty * TX;
    const int y = y0 + ty, x = x0 + tx;
    c_j[k] = (ty + 1) * FT::P1 + (tx + 1);
    c_m[k] = c < FT::R0 ? sb_yx_mask(g, y, x) : 0;
    c_goff[k] = y * g.mx + x;
  }

  // ---- register prefetch of plane zf: omega (3) and u (3) for this thread's region-2 cells
  T rw[FT::C2N][3], ru[FT::C2N][3];
  auto prefetch = [&](int z) {
    const bool zin = z >= 0 && z < g.mz;
    const long long zoff = (long long)z * plane;
#pragma unroll
    for (int k = 0; k < FT::C2N; ++k) {
      if (zin && a_goff[k] >= 0) {
        const long long gi = zoff + a_goff[k];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          rw[k][c] = w[gi + c * vol];
          ru[k][c] = u[gi + c * vol];
        }
      } else {
#pragma unroll
        for (int c = 0; c < 3; ++c) rw[k][c] = ru[k][c] = T(0);
      }
    }
  };
  prefetch(zb - 2);

  for (int zf = zb - 2; zf <= ze + 1; ++zf) {
    // ---- A: cross product of plane zf on tile + 2, omega of plane zf on tile + 1
    {
      T* b = sbuf + ((zf + 3) % 3) * 3 * FT::R2;
      T* s1 = sw1 + ((zf + 2) & 1) * 3 * FT::R1;
#pragma unroll
      for (int k = 0; k < FT::C2N; ++k) {
        const int i = tid + k * NT;
        if (i < FT::R2) {
          const T w0 = rw[k][0], w1 = rw[k][1], w2 = rw[k][2];
          const T u0 = ru[k][0], u1 = ru[k][1], u2 = ru[k][2];
          b[i] = u1 * w2 - u2 * w1;
          b[FT::R2 + i] = u2 * w0 - u0 * w2;
          b[2 * FT::R2 + i] = u0 * w1 - u1 * w0;
          const int j = a_j[k];
          if (j >= 0) {
            s1[j] = w0;
            s1[FT::R1 + j] = w1;
            s1[2 * FT::R1 + j] = w2;
          }
        }
      }
    }
    if (zf + 1 <= ze + 1) prefetch(zf + 1);  // in flight during phases B and C
    __syncthreads();
    // ---- B: omega2 of plane zc = zf - 1 on tile + 1
    const int zc = zf - 1;
    if (zc >= 0 && zc < g.mz) {
      const T* bm = sbuf + ((zc + 2) % 3) * 3 * FT::R2;  // plane zc - 1
      const T* b0 = sbuf + (zc % 3) * 3 * FT::R2;
      const T* bp = sbuf + ((zc + 1) % 3) * 3 * FT::R2;
      const T* s1 = sw1 + (zc & 1) * 3 * FT::R1;
      T* s2 = sw2 + (zc % 3) * 3 * FT::R1;
      const int zmask = ((zc >= 1 && zc < g.mz - 1) ? 1 : 0) | ((zc >= zlo && zc < zhi) ? 2 : 0);
#pragma unroll
      for (int k = 0; k < FT::C1N; ++k) {
        const int j = tid + k * NT;
        if (j < FT::R1) {
          T c0 = s1[j], c1 = s1[FT::R1 + j], c2 = s1[2 * FT::R1 + j];
          if (b_m[k] & zmask & 3) {
            const int i = b_i[k];
            const T* by0 = b0 + FT::R2;
            const T* bz0 = b0 + 2 * FT::R2;
            c0 += p * (bz0[i + FT::P2] - bz0[i - FT::P2] - bp[FT::R2 + i] + bm[FT::R2 + i]);
            c1 += p * (bp[i] - bm[i] - bz0[i + 1] + bz0[i - 1]);
            c2 += p * (by0[i + 1] - by0[i - 1] - b0[i + FT::P2] + b0[i - FT::P2]);
          }
          s2[j] = c0;
          s2[FT::R1 + j] = c1;
          s2[2 * FT::R1 + j] = c2;
        }
      }
    }
    __syncthreads();
    // ---- C: diffusion of plane zo = zf - 2 on the tile, write out
    const int zo = zf - 2;
    if (zo >= zb && zo < ze) {
      const T* qm = sw2 + ((zo + 2) % 3) * 3 * FT::R1;
      const T* q0 = sw2 + (zo % 3) * 3 * FT::R1;
      const T* qp = sw2 + ((zo + 1) % 3) * 3 * FT::R1;
      const int zmask = ((zo >= 1 && zo < g.mz - 1) ? 1 : 0) | ((zo >= zlo && zo < zhi) ? 2 : 0);
      const bool zring = zo < zring_lo || zo >= zring_hi;
      const long long zoff = (long long)zo * plane;
#pragma unroll
      for (int k = 0; k < FT::C0N; ++k) {
        const int m = c_m[k];
        if (m & 4) {
          const int j = c_j[k];
          const bool lap = (m & zmask & 3) && !(m & 8) && !zring;
          const long long gi = zoff + c_goff[k];
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            const T* q = q0 + c * FT::R1;
            T v = q[j];
            if (lap) {
              const T s = q[j + 1] + q[j - 1] + q[j + FT::P1] + q[j - FT::P1] + qp[c * FT::R1 + j] +
                          qm[c * FT::R1 + j];
              v += d * (s - T(6) * q[j]);
            }
            out[gi + c * vol] = v;
          }
        }
      }
    }
    // (the barrier after phase A of the next iteration orders C against the next B)
  }
}

// ----------------------------------------------------------------------------------------------
// Float version 2: the same update with vectorised global access and far fewer instructions per cell.
// A warp owns one row of 64 cells (32 lanes x a strip of 2 cells: 8-byte loads / stores, 256 contiguous
// bytes per warp), a block R consecutive rows, and the block marches along z.  z neighbours are carried
// in registers (two planes of history), x neighbours come from the strip itself or from the adjacent
// lanes (shuffles), and only the y neighbours go through shared memory (5 arrays, double buffered, ONE
// barrier per plane).  Every thread evaluates all three levels on its own cells: u x omega on the whole
// block footprint, omega2 on footprint - 1, the result on footprint - 2, so a block stores (R - 4) rows
// x 60 cells.  Blocks whose footprint lies inside the region written by the reference's interior
// call skip the per-cell wrapper masks (FAST); the others evaluate them exactly as version 1 does.
template <int R>
struct FusedV2 {
  static constexpr int NT = 32 * R;
  static constexpr int TXU = 60, TYU = R - 4;        // cells stored per block
  static constexpr int ROW = 64;                     // floats per row in shared memory
  static constexpr int ARR = (R + 2) * ROW;          // one array: R rows + a guard row at each end
  static constexpr int ELEMS = 2 * 5 * ARR;          // double buffered: buf_x, buf_z, omega2 x 3
};

struct alignas(8) F2 {
  float x, y;
};
SB_D F2 sb_ld2(const float* p) { return *reinterpret_cast<const F2*>(p); }
SB_D void sb_st2(float* p, F2 v) { *reinterpret_cast<F2*>(p) = v; }

template <int R, bool FAST>
SB_D void sb_vorticity_fused_v2_body(const SbGeom& g, float* __restrict__ out, const float* __restrict__ w,
                                     const float* __restrict__ u, float p, float d, int zchunk, int z_begin,
                                     int z_end, float* smem) {
  using FV = FusedV2<R>;
  const int lane = threadIdx.x & 31, row = threadIdx.x >> 5;
  const int x = (int)blockIdx.x * FV::TXU - 2 + 2 * lane;  // first cell of the strip (even)
  const int y = (int)blockIdx.y * FV::TYU - 2 + row;
  const int zb = z_begin + blockIdx.z * zchunk;
  const int ze = zb + zchunk < z_end ? zb + zchunk : z_end;
  const long long vol = g.vol, plane = g.plane;
  const int zlo = g.phys[0] ? g.gs : 1, zhi = g.phys[1] ? g.mz - g.gs : g.mz - 1;
  const int zring_lo = g.phys[0] ? g.gs + 1 : 0, zring_hi = g.phys[1] ? g.mz - g.gs - 1 : g.mz;
  // per-cell (y,x) masks (z invariant): bit0 A, bit1 B, bit2 inside the array, bit3 physical ring
  int m0 = 6, m1 = 6;
  bool in0 = true, in1 = true;
  if (!FAST) {
    m0 = sb_yx_mask(g, y, x);
    m1 = sb_yx_mask(g, y, x + 1);
    in0 = (m0 & 4) != 0;
    in1 = (m1 & 4) != 0;
  }
  // a strip is loaded / stored as one 8-byte access when both cells are inside the array
  const bool pair = in0 && in1;
  const long long goff = (long long)y * g.mx + x;
  const bool st_row = row >= 2 && row < R - 2 && lane >= 1 && lane <= 30;  // cells this thread stores
  float* sA = smem;  // [parity][array][row + 1][64]
  const int soff = (row + 1) * FV::ROW + 2 * lane;

  // zero the guard rows once (rows 0 and R + 1 of every array are only read by the edge rows, whose
  // results are never stored; keep them finite)
  for (int i = threadIdx.x; i < FV::ELEMS; i += FV::NT) smem[i] = 0.f;
  __syncthreads();

  auto load_plane = [&](int z, F2 (&wl)[3], F2 (&ul)[3]) {
    const bool zin = z >= 0 && z < g.mz;
    if (zin && (FAST || pair)) {
      const long long gi = (long long)z * plane + goff;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        wl[c] = sb_ld2(w + gi + c * vol);
        ul[c] = sb_ld2(u + gi + c * vol);
      }
    } else {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        wl[c] = F2{0.f, 0.f};
        ul[c] = F2{0.f, 0.f};
      }
      if (!FAST && zin) {
        const long long gi = (long long)z * plane + goff;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          if (in0) {
            wl[c].x = w[gi + c * vol];
            ul[c].x = u[gi + c * vol];
          }
          if (in1) {
            wl[c].y = w[gi + 1 + c * vol];
            ul[c].y = u[gi + 1 + c * vol];
          }
        }
      }
    }
  };
  // One plane of the march.  The z history lives in registers that ROTATE through the roles (the
  // march is unrolled six times below, the period of the 3-deep omega / buf / omega2 and the 2-deep u
  // rotations), so no register is ever copied:
  //   wnext/unext: plane zf + 1 (loads in flight)   wcur/ucur: plane zf   wprev: plane zf - 1
  //   b0 = buf(zf) (written here), b1 = buf(zf - 1), b2 = buf(zf - 2)
  //   q1 = omega2(zf - 1) (written here), q2 = omega2(zf - 2), q3 = omega2(zf - 3)
  auto step = [&](int zf, F2 (&wnext)[3], F2 (&unext)[3], const F2 (&wc)[3], const F2 (&uc)[3], const F2 (&wp)[3],
                  F2 (&b0)[3], const F2 (&b1)[3], const F2 (&b2)[3], F2 (&q1)[3], const F2 (&q2)[3],
                  const F2 (&q3)[3]) {
    const int par = zf & 1;
    float* sw = sA + par * 5 * FV::ARR;               // written this iteration
    const float* sr = sA + (par ^ 1) * 5 * FV::ARR;   // written by the previous iteration
    if (zf + 1 <= ze + 1) load_plane(zf + 1, wnext, unext);
    b0[0] = F2{uc[1].x * wc[2].x - uc[2].x * wc[1].x, uc[1].y * wc[2].y - uc[2].y * wc[1].y};
    b0[1] = F2{uc[2].x * wc[0].x - uc[0].x * wc[2].x, uc[2].y * wc[0].y - uc[0].y * wc[2].y};
    b0[2] = F2{uc[0].x * wc[1].x - uc[1].x * wc[0].x, uc[0].y * wc[1].y - uc[1].y * wc[0].y};

    // ---- omega2 of plane zc = zf - 1 (needs buf(zf), buf(zf - 2) own; buf(zf - 1) neighbours)
    const int zc = zf - 1;
    {
      const F2 bxu = sb_ld2(sr + 0 * FV::ARR + soff + FV::ROW), bxd = sb_ld2(sr + 0 * FV::ARR + soff - FV::ROW);
      const F2 bzu = sb_ld2(sr + 1 * FV::ARR + soff + FV::ROW), bzd = sb_ld2(sr + 1 * FV::ARR + soff - FV::ROW);
      // x neighbours of buf_y, buf_z at plane zc: inside the strip or from the adjacent lane
      const float byl = __shfl_up_sync(0xffffffffu, b1[1].y, 1), byr = __shfl_down_sync(0xffffffffu, b1[1].x, 1);
      const float bzl = __shfl_up_sync(0xffffffffu, b1[2].y, 1), bzr = __shfl_down_sync(0xffffffffu, b1[2].x, 1);
      const int zmask = ((zc >= 1 && zc < g.mz - 1) ? 1 : 0) | ((zc >= zlo && zc < zhi) ? 2 : 0);
      const bool wr0 = FAST ? (zmask & 2) != 0 : (m0 & zmask & 3) != 0;
      const bool wr1 = FAST ? (zmask & 2) != 0 : (m1 & zmask & 3) != 0;
      // curl_x = d(buf_z)/dy - d(buf_y)/dz ; curl_y = d(buf_x)/dz - d(buf_z)/dx ; curl_z = d(buf_y)/dx - d(buf_x)/dy
      q1[0] = wp[0];
      q1[1] = wp[1];
      q1[2] = wp[2];
      if (wr0) {
        q1[0].x += p * (bzu.x - bzd.x - b0[1].x + b2[1].x);
        q1[1].x += p * (b0[0].x - b2[0].x - b1[2].y + bzl);
        q1[2].x += p * (b1[1].y - byl - bxu.x + bxd.x);
      }
      if (wr1) {
        q1[0].y += p * (bzu.y - bzd.y - b0[1].y + b2[1].y);
        q1[1].y += p * (b0[0].y - b2[0].y - bzr + b1[2].x);
        q1[2].y += p * (byr - b1[1].x - bxu.y + bxd.y);
      }
    }
    // ---- result of plane zo = zf - 2 (needs omega2(zf - 1), omega2(zf - 3) own; omega2(zf - 2) neighbours)
    const int zo = zf - 2;
    if (zo >= zb && zo < ze) {
      const int zmask = ((zo >= 1 && zo < g.mz - 1) ? 1 : 0) | ((zo >= zlo && zo < zhi) ? 2 : 0);
      const bool zring = zo < zring_lo || zo >= zring_hi;
      const bool lap0 = (FAST ? (zmask & 2) != 0 : ((m0 & zmask & 3) != 0 && !(m0 & 8))) && !zring;
      const bool lap1 = (FAST ? (zmask & 2) != 0 : ((m1 & zmask & 3) != 0 && !(m1 & 8))) && !zring;
      F2 r[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const F2 qu = sb_ld2(sr + (2 + c) * FV::ARR + soff + FV::ROW);
        const F2 qd = sb_ld2(sr + (2 + c) * FV::ARR + soff - FV::ROW);
        const float ql = __shfl_up_sync(0xffffffffu, q2[c].y, 1), qr = __shfl_down_sync(0xffffffffu, q2[c].x, 1);
        r[c] = q2[c];
        if (lap0) {
          const float sum = q2[c].y + ql + qu.x + qd.x + q1[c].x + q3[c].x;
          r[c].x += d * (sum - 6.f * q2[c].x);
        }
        if (lap1) {
          const float sum = qr + q2[c].x + qu.y + qd.y + q1[c].y + q3[c].y;
          r[c].y += d * (sum - 6.f * q2[c].y);
        }
      }
      if (st_row) {
        const long long gi = (long long)zo * plane + goff;
        if (FAST || pair) {
#pragma unroll
          for (int c = 0; c < 3; ++c) sb_st2(out + gi + c * vol, r[c]);
        } else {
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            if (in0) out[gi + c * vol] = r[c].x;
            if (in1) out[gi + 1 + c * vol] = r[c].y;
          }
        }
      }
    }
    // ---- publish this iteration's planes for the y neighbours of the next one
    sb_st2(sw + 0 * FV::ARR + soff, b0[0]);
    sb_st2(sw + 1 * FV::ARR + soff, b0[2]);
    sb_st2(sw + 2 * FV::ARR + soff, q1[0]);
    sb_st2(sw + 3 * FV::ARR + soff, q1[1]);
    sb_st2(sw + 4 * FV::ARR + soff, q1[2]);
    __syncthreads();
  };

  F2 W[3][3] = {}, U[2][3] = {}, B[3][3] = {}, Q[3][3] = {};
  load_plane(zb - 2, W[0], U[0]);
  const int zlast = ze + 1;
  // step k of a period: current plane in W[k % 3] / U[k % 2], results into B[k % 3] / Q[k % 3]
#define SB_FUSED_STEP(k)                                                                                     \
  step(zf, W[((k) + 1) % 3], U[((k) + 1) % 2], W[(k) % 3], U[(k) % 2], W[((k) + 2) % 3], B[(k) % 3],         \
       B[((k) + 2) % 3], B[((k) + 1) % 3], Q[(k) % 3], Q[((k) + 2) % 3], Q[((k) + 1) % 3]);                  \
  if (++zf > zlast) break;
  for (int zf = zb - 2;;) {
    SB_FUSED_STEP(0)
    SB_FUSED_STEP(1)
    SB_FUSED_STEP(2)
    SB_FUSED_STEP(3)
    SB_FUSED_STEP(4)
    SB_FUSED_STEP(5)
  }
#undef SB_FUSED_STEP
}

template <int R>
__global__ void __launch_bounds__(32 * R)
    sb_vorticity_fused_v2_kernel(SbGeom g, float* __restrict__ out, const float* __restrict__ w,
                                 const float* __restrict__ u, float p, float d, int zchunk, int z_begin,
                                 int z_end) {
  using FV = FusedV2<R>;
  SB_DYN_SMEM(smem_raw);
  float* smem = reinterpret_cast<float*>(smem_raw);
  // the block's footprint: x in [x0 - 2, x0 + 62), y in [y0 - 2, y0 + R - 2); omega2 is evaluated on
  // footprint - 1: FAST when that region lies where the reference's interior call writes (mask B, no ring)
  const int x0 = (int)blockIdx.x * FV::TXU, y0 = (int)blockIdx.y * FV::TYU;
  const bool fast = x0 - 1 >= g.gs + 1 && x0 + FV::TXU <= g.mx - g.gs - 2 && y0 - 1 >= g.gs + 1 &&
                    y0 + FV::TYU <= g.my - g.gs - 2 && x0 + 62 <= g.mx && y0 + R - 2 <= g.my;
  if (fast)
    sb_vorticity_fused_v2_body<R, true>(g, out, w, u, p, d, zchunk, z_begin, z_end, smem);
  else
    sb_vorticity_fused_v2_body<R, false>(g, out, w, u, p, d, zchunk, z_begin, z_end, smem);
}

// z chunks of the marching kernels: a block marches zchunk + 4 planes (4 to prime the rings), and the grid
// of tiles x chunks runs in waves of `resident` blocks; pick the chunk count that minimises
// waves x (zchunk + 4), with chunks of at least 8 planes.  (6 chunks at 260^3 were 918 blocks = 2.07 waves
// of 444: a third wave for 30 blocks.)
struct SbZChunks {
  int chunks, zchunk;
};
static SbZChunks sb_z_chunks(long long tiles, int nzr, long long resident) {
  SbZChunks r{1, nzr};
  long long best = -1;
  for (int c = 1; c <= nzr; ++c) {
    const int zc = (nzr + c - 1) / c;
    if (zc < 8 && c > 1) break;
    const int cc = (nzr + zc - 1) / zc;  // chunks actually needed for this chunk length
    const long long waves = (tiles * cc + resident - 1) / resident;
    const long long cost = waves * (zc + 4);
    if (best < 0 || cost < best) {
      best = cost;
      r = SbZChunks{cc, zc};
    }
  }
  return r;
}

template <int R>
static int launch_fused_v2(const SbGeom& g, void* out, const void* w, const void* u, double p, double d,
                           int z0, int z1, void* stream) {
  using FV = FusedV2<R>;
  const size_t smem = sizeof(float) * FV::ELEMS;
  const unsigned gx = (g.mx + FV::TXU - 1) / FV::TXU, gy = (g.my + FV::TYU - 1) / FV::TYU;
  SB_KERNEL_ATTR_SMEM((sb_vorticity_fused_v2_kernel<R>), smem);
  long long resident = 148;
#ifndef SB200_EMU
  {
    static long long cached = 0;
    if (cached == 0) {
      int dev = 0, sms = 0, per_sm = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sb_vorticity_fused_v2_kernel<R>, FV::NT, smem);
      cached = (long long)sms * (per_sm > 0 ? per_sm : 1);
    }
    resident = cached;
  }
#endif
  const SbZChunks zc = sb_z_chunks((long long)gx * gy, z1 - z0, resident);
  SB_LAUNCH_COOP((sb_vorticity_fused_v2_kernel<R>), dim3(gx, gy, (unsigned)zc.chunks), dim3(FV::NT), smem, stream, g,
                 (float*)out, (const float*)w, (const float*)u, (float)p, (float)d, zc.zchunk, z0, z1);
  SB_CHECK_LAUNCH("vorticity_fused_v2");
  return 0;
}

template <typename T, int TY, int TX, int NT>
static int launch_fused(const SbGeom& g, void* out, const void* w, const void* u, double p, double d,
                        int z0, int z1, void* stream) {
  using FT = FusedTile<TY, TX, NT>;
  const size_t smem = sizeof(T) * FT::ELEMS;
  const unsigned gx = (g.mx + TX - 1) / TX, gy = (g.my + TY - 1) / TY;
  SB_KERNEL_ATTR_SMEM((sb_vorticity_fused_kernel<T, TY, TX, NT>), smem);
  long long resident = 148 * 3;
#ifndef SB200_EMU
  {
    static long long cached = 0;
    if (cached == 0) {
      int dev = 0, sms = 0, per_sm = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sb_vorticity_fused_kernel<T, TY, TX, NT>, NT, smem);
      cached = (long long)sms * (per_sm > 0 ? per_sm : 1);
    }
    resident = cached;
  }
#endif
  const SbZChunks zc = sb_z_chunks((long long)gx * gy, z1 - z0, resident);
  SB_LAUNCH_COOP((sb_vorticity_fused_kernel<T, TY, TX, NT>), dim3(gx, gy, (unsigned)zc.chunks), dim3(NT), smem,
                 stream, g, (T*)out, (const T*)w, (const T*)u, (T)p, (T)d, zc.zchunk, z0, z1);
  SB_CHECK_LAUNCH("vorticity_fused");
  return 0;
}

extern "C" int sb200_vorticity_rhs_fused_3d_range(const sb200_grid_t* gr, void* out, const void* vorticity,
                                                  const void* velocity, double curl_prefactor, double nu_dt_by_dx2,
                                                  int z_begin, int z_end, void* stream) {
  SbGeom g;
  SB_REQUIRE(sb_make_geom(gr, &g) == 0, "bad grid");
  SB_REQUIRE(g.dim == 3, "vorticity_rhs_fused_3d: 3D only");
  SB_REQUIRE(g.gs >= 2, "vorticity_rhs_fused_3d needs ghost_size >= 2");
  SB_REQUIRE(out && vorticity && velocity && out != vorticity, "vorticity_rhs_fused_3d: bad pointers");
  SB_REQUIRE(g.plane < (1LL << 31), "vorticity_rhs_fused_3d: plane too large");
  SB_REQUIRE(z_begin >= 0 && z_end <= g.mz, "vorticity_rhs_fused_3d: bad plane range");
  if (z_end <= z_begin) return 0;
  if (gr->dtype == SB200_F32) {
    // version 2 (24 rows per block) needs even row lengths (8-byte strips)
    if ((g.mx & 1) == 0)
      return launch_fused_v2<24>(g, out, vorticity, velocity, curl_prefactor, nu_dt_by_dx2, z_begin, z_end, stream);
    // 16 x 32 tiles, 256 threads (version 1): measured best of 8x64, 12x32, 24x32, 16x48, 16x16 in round 1
    return launch_fused<float, 16, 32, 256>(g, out, vorticity, velocity, curl_prefactor, nu_dt_by_dx2, z_begin, z_end,
                                            stream);
  }
  return launch_fused<double, 8, 32, 256>(g, out, vorticity, velocity, curl_prefactor, nu_dt_by_dx2, z_begin, z_end,
                                          stream);
}

extern "C" int sb200_vorticity_rhs_fused_3d(const sb200_grid_t* gr, void* out, const void* vorticity,
                                            const void* velocity, const void* forcing,
                                            double curl_prefactor, double nu_dt_by_dx2, void* stream) {
  SB_REQUIRE(gr, "bad grid");
  SB_REQUIRE(forcing == nullptr,
             "vorticity_rhs_fused_3d: apply the forcing update first "
             "(sb200_update_vorticity_from_sparse_forcing)");
  return sb200_vorticity_rhs_fused_3d_range(gr, out, vorticity, velocity, curl_prefactor, nu_dt_by_dx2, 0,
                                            gr->n[0] + 2 * gr->gs, stream);
}
