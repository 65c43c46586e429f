// Stand-alone operators around the fused path, sm_100a: rfgr2beff (dense field synthesis), beff2ab
// (Hargreaves A/B propagation, forward and adjoint), beff2u-phi and freeprec.  All are HBM-bound / one-shot; they exist so that every function of
// the reference's path (SURVEY 8a: a3, a5, f-1) has a native implementation behind the same C ABI.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/mrphy_b200.h"
#include "abi_common.cuh"
#include "bloch_math.cuh"
#include "grad_finalize.cuh"
#include "ptx_helpers.cuh"

namespace mrphy {

// ---- rfgr2beff (beffective.py:107-168) -------------------------------------------------------------
// Threads run along time for one spin: the three components of consecutive steps are contiguous, so a block's
// output for one spin is ONE contiguous run of 12*RB bytes.  A block owns RB = 1024 consecutive steps (4 per
// thread, waveform samples in registers) of SPB consecutive spins; per spin the 4x3 results are staged in shared
// memory (double-buffered, one barrier per spin) and leave as 128-bit stores when rows are 16-byte aligned
// (ALIGNED), as scalar stores otherwise.  The next spin's constants are fetched while the current one is stored.
// MC: several coils with a b1Map (the coil sum runs inside, rf re-read from L1); otherwise the coils are
// pre-summed (no b1Map, beffective.py:147-151) or there is one coil.
template <typename T> struct SpinK { T lx, ly, lz, bz0, br, bi; };

template <typename T>
__device__ __forceinline__ SpinK<T> load_spin_k(const mrphy_rfgr2beff_args& a, int n, int i, bool mc) {
  SpinK<T> k;
  const T* lp = (const T*)a.loc + (int64_t)n * a.loc_sn + (int64_t)i * a.loc_sm;
  k.lx = lp[0]; k.ly = lp[1]; k.lz = lp[2];
  k.bz0 = a.df.ptr ? (T)ld_param(a.df, n, i) / (T)ld_param(a.gamma, n, i) : (T)0;   // beffective.py:142
  k.br = (T)1; k.bi = (T)0;
  if (a.b1 && !mc) {
    const T* bp = (const T*)a.b1 + (int64_t)n * a.b1_sn + (int64_t)i * a.b1_sm;
    k.br = bp[0]; k.bi = bp[a.nC];
  }
  return k;
}

template <typename T, bool ALIGNED, bool MC>
__global__ void __launch_bounds__(256, sizeof(T) == 8 ? 3 : 4) rfgr2beff_kernel(const mrphy_rfgr2beff_args a, const int tblocks) {
  constexpr int SPT = 4, RB = 256 * SPT, SPB = 16;   // steps per thread, steps per block, spins per block
  constexpr int NST = ALIGNED ? 3 : 2;               // stage buffers (3 with the asynchronous bulk stores)
  extern __shared__ __align__(128) unsigned char rf_smem[];
  T(*stage)[3 * RB] = reinterpret_cast<T(*)[3 * RB]>(rf_smem);
  const int n = blockIdx.y, tid = threadIdx.x;
  const int sb = (int)(blockIdx.x / tblocks);
  const int tb0 = (int)(blockIdx.x % tblocks) * RB;
  const int cnt = min(RB, a.nT - tb0);
  T rx[SPT], ry[SPT], gx[SPT], gy[SPT], gz[SPT];
#pragma unroll
  for (int u = 0; u < SPT; ++u) {
    const int t = tb0 + u * 256 + tid;
    rx[u] = ry[u] = gx[u] = gy[u] = gz[u] = (T)0;
    if (t < a.nT) {
      const T* gr = (const T*)a.gr + (int64_t)n * a.gr_sn + (int64_t)t * a.gr_st;
      gx[u] = gr[0]; gy[u] = gr[a.gr_sx]; gz[u] = gr[2 * a.gr_sx];
      if (!MC) {
        const T* rf = (const T*)a.rf + (int64_t)n * a.rf_sn + (int64_t)t * a.rf_st;
        for (int c = 0; c < a.nC; ++c) { rx[u] += rf[c * a.rf_sc]; ry[u] += rf[a.rf_sx + c * a.rf_sc]; }
      }
    }
  }
  const int i0 = sb * SPB, i1 = min(a.nM, i0 + SPB);
  SpinK<T> k = load_spin_k<T>(a, n, i0, MC);
  for (int i = i0; i < i1; ++i) {
    const SpinK<T> kn = load_spin_k<T>(a, n, min(i + 1, i1 - 1), MC);   // in flight during this spin's math + stores
    T* st = stage[(i - i0) % NST];
#pragma unroll
    for (int u = 0; u < SPT; ++u) {
      const int j = u * 256 + tid;
      T bx, by;
      if (!MC) {
        bx = fnma_(k.bi, ry[u], k.br * rx[u]);
        by = fma_(k.bi, rx[u], k.br * ry[u]);
      } else {              // several coils with a b1Map (beffective.py:160-165)
        bx = by = (T)0;
        if (tb0 + j < a.nT) {
          const T* rf = (const T*)a.rf + (int64_t)n * a.rf_sn + (int64_t)(tb0 + j) * a.rf_st;
          const T* bp = (const T*)a.b1 + (int64_t)n * a.b1_sn + (int64_t)i * a.b1_sm;
          for (int c = 0; c < a.nC; ++c) {
            const T x = rf[c * a.rf_sc], y = rf[a.rf_sx + c * a.rf_sc], br = bp[c], bi = bp[a.nC + c];
            bx += br * x - bi * y;
            by += br * y + bi * x;
          }
        }
      }
      st[3 * j] = bx; st[3 * j + 1] = by;
      st[3 * j + 2] = fma_(k.lx, gx[u], fma_(k.ly, gy[u], fma_(k.lz, gz[u], k.bz0)));
    }
    T* out = (T*)a.Beff + (((int64_t)n * a.nM + i) * a.nT + tb0) * 3;
    if (ALIGNED) {
      // the row leaves as ONE TMA bulk store (cp.async.bulk shared -> global, 12*cnt bytes).  Three buffers: before this
      // barrier thread 0 waits until all but the latest store have finished reading shared memory, so the buffer
      // written at the next spin (last used three spins ago) is known to be free by everyone after the barrier.
      fence_proxy_async_smem();
      if (tid == 0) bulk_wait_read<1>();
      __syncthreads();
      if (tid == 0) {
        bulk_s2g(out, st, (uint32_t)(cnt * 3 * sizeof(T)));
        bulk_commit();
      }
    } else {
      __syncthreads();   // also orders buffer reuse: this buffer was last read two spins ago
      for (int q = tid; q < 3 * cnt; q += 256) out[q] = st[q];
    }
    k = kn;
  }
  if (ALIGNED && tid == 0) bulk_wait_read<0>();   // shared memory must outlive the last stores
}

// ---- adjoint of rfgr2beff: the sums over spins ------------------------------------------------------
// Threads run along time: a block owns 256 steps x one range of spins and keeps its W = 2*NC+3 running sums in
// registers; the spins' constants (b1, loc) are staged through shared memory one group of G spins at a time, two
// stages on one barrier per group.  ALIGNED (nT % 4 == 0 and a 16-byte aligned gBeff: every row is) stages the rows
// too, by the TMA engine: one 1-D bulk copy (cp.async.bulk, 3 KB = 256 steps x xyz) per spin, G spins per stage on
// mbarriers -- 24 KB in flight per block, no registers or L1 sectors spent on the strided xyz pattern; threads then
// read their own triplet from shared memory (stride 3: conflict-free).  Otherwise each thread reads its own triplet
// from global memory (the xyz triplets of 256 consecutive steps of one spin are 3 KB contiguous, so a warp's three
// strided loads cover whole lines).  Block partials go to partials[N][S][W][nT]; grad_finalize_kernel sums the S
// slices in fixed order.
template <typename T, bool ALIGNED> struct RBCfg {
  static constexpr int G = ALIGNED ? 32 / (int)sizeof(T) : 32;        // spins per stage: 8 (fp32), 4 (fp64); 32 unstaged
  static constexpr int TBK = 256;
  static constexpr size_t buf_bytes = ALIGNED ? (size_t)2 * G * 3 * TBK * sizeof(T) : 0;   // 48 KB of rows
  __host__ __device__ static constexpr size_t cst_bytes(int W) { return ((sizeof(T) * 2 * G * W + 15) / 16) * 16; }
  __host__ __device__ static constexpr size_t smem(int W) { return buf_bytes + cst_bytes(W) + 16; }   // rows, constants, 2 mbarriers
};
template <typename T, int NC, bool ALIGNED>
__global__ void __launch_bounds__(256) rfgr2beff_bwd_kernel(const mrphy_rfgr2beff_args a, const int per_split) {
  using C = RBCfg<T, ALIGNED>;
  constexpr int W = 2 * NC + 3, G = C::G, TBK = C::TBK;
  extern __shared__ __align__(128) unsigned char rb_smem[];
  T(*buf)[G][3 * TBK] = reinterpret_cast<T(*)[G][3 * TBK]>(rb_smem);
  T(*cst)[G][W] = reinterpret_cast<T(*)[G][W]>(rb_smem + C::buf_bytes);
  uint64_t* full = reinterpret_cast<uint64_t*>(rb_smem + C::buf_bytes + C::cst_bytes(W));
  const int n = blockIdx.z, split = blockIdx.y, S = gridDim.y, tid = threadIdx.x;
  const int t0 = blockIdx.x * TBK, len = min(TBK, a.nT - t0);
  const uint32_t row_bytes = (uint32_t)(len * 3 * sizeof(T));
  const bool valid = tid < len;
  const int i0 = split * per_split, i1 = min(a.nM, i0 + per_split);
  const int ngroups = (i1 - i0 + G - 1) / G;
  const T* Gb = (const T*)a.gBeff + ((size_t)n * a.nM * a.nT + t0) * 3;
  if (ALIGNED && tid == 0) {
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    fence_barrier_init();
  }
  __syncthreads();
  auto issue = [&](int g, int s) {
    const int c0 = i0 + g * G, cnt = min(G, i1 - c0);
    if (ALIGNED && tid == 0) {
      mbar_arrive_expect_tx(&full[s], row_bytes * cnt);
      for (int q = 0; q < cnt; ++q) bulk_g2s(buf[s][q], Gb + (size_t)(c0 + q) * a.nT * 3, row_bytes, &full[s]);
    }
    for (int e = tid; e < cnt * W; e += 256) {   // the group's b1 / loc (visible after the barrier closing this iteration)
      const int q = e / W, w = e - q * W, i = c0 + q;
      T v;
      if (w < 2 * NC) {
        const int c = w % NC;
        v = a.b1 ? (c < a.nC ? ((const T*)a.b1)[(int64_t)n * a.b1_sn + (int64_t)i * a.b1_sm + (w / NC) * a.nC + c] : (T)0)
                 : (w < NC ? (T)1 : (T)0);
      } else {
        v = ((const T*)a.loc)[(int64_t)n * a.loc_sn + (int64_t)i * a.loc_sm + (w - 2 * NC)];
      }
      cst[s][q][w] = v;
    }
  };
  T arx[NC], ary[NC], ag[3] = {0, 0, 0};
#pragma unroll
  for (int c = 0; c < NC; ++c) arx[c] = ary[c] = (T)0;
  if (ngroups > 0) issue(0, 0);
  __syncthreads();
  for (int g = 0; g < ngroups; ++g) {
    const int s = g & 1, cnt = min(G, i1 - (i0 + g * G));
    if (g + 1 < ngroups) issue(g + 1, s ^ 1);   // that stage was drained in iteration g-1 (barrier below)
    if (ALIGNED) mbar_wait(&full[s], (g >> 1) & 1);
    if (valid) {
#pragma unroll 4
      for (int q = 0; q < cnt; ++q) {
        const T* gp = ALIGNED ? &buf[s][q][3 * tid] : Gb + (size_t)(i0 + g * G + q) * a.nT * 3 + 3 * tid;
        const T gx = gp[0], gy = gp[1], gz = gp[2];
#pragma unroll
        for (int c = 0; c < NC; ++c) {
          const T br = cst[s][q][c], bi = cst[s][q][NC + c];
          arx[c] = fma_(br, gx, fma_(bi, gy, arx[c]));
          ary[c] = fma_(br, gy, fnma_(bi, gx, ary[c]));
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) ag[k] = fma_(cst[s][q][2 * NC + k], gz, ag[k]);
      }
    }
    __syncthreads();
  }
  if (!valid) return;
  T* P = (T*)a.partials + (((size_t)n * S + split) * W) * (size_t)a.nT + t0 + tid;
#pragma unroll
  for (int c = 0; c < NC; ++c) { P[(size_t)c * a.nT] = arx[c]; P[(size_t)(NC + c) * a.nT] = ary[c]; }
#pragma unroll
  for (int k = 0; k < 3; ++k) P[(size_t)(2 * NC + k) * a.nT] = ag[k];
}

// ---- beff2ab (beffective.py:40-104) ----------------------------------------------------------------
// One spin per thread, [A|B] = 4 column vectors in registers, same rotation + relaxation per step as the
// simulation (apply_fwd with the relaxation constants given as factors).
template <typename T, int POL>
__global__ void __launch_bounds__(128) beff2ab_kernel(const mrphy_beff2ab_args a) {
  const int n = blockIdx.y, i = blockIdx.x * 128 + threadIdx.x;
  if (i >= a.nM) return;
  const double gam = ld_param(a.gamma, n, i), dt = ld_param(a.dt, n, 0);
  const T g = (T)(6.283185307179586476925286766559 * gam * dt);
  const T E1 = (T)ld_param(a.E1, n, i), E2 = (T)ld_param(a.E2, n, i);
  const T e1 = E1 - (T)1, e2 = E2 - (T)1;
  T cx[4] = {1, 0, 0, 0}, cy[4] = {0, 1, 0, 0}, cz[4] = {0, 0, 1, 0};   // columns of [A|B]
  const T* B = (const T*)a.Beff + (int64_t)n * a.B_sn + (int64_t)i * a.B_sm;
  T* ck = a.ckpt ? (T*)a.ckpt + (size_t)n * ((a.nT - 1) / a.K) * 12 * (size_t)a.nM : nullptr;
  for (int t = 0; t < a.nT; ++t) {
    const T bx = g * B[3 * t], by = g * B[3 * t + 1], bz = g * B[3 * t + 2];
    const RotCoef<T> r = rot_coef<T, POL>(bx, by, bz);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      // rotate, then scale by (E2,E2,E1); only the B column receives the recovery term (1-E1)
      apply_fwd<T, false>(r, bx, by, bz, (T)0, (T)0, cx[q], cy[q], cz[q]);
      cx[q] = fma_(e2, cx[q], cx[q]);
      cy[q] = fma_(e2, cy[q], cy[q]);
      cz[q] = fma_(e1, cz[q], cz[q]);
    }
    cz[3] -= e1;
    const int t1 = t + 1;
    if (ck && t1 % a.K == 0 && t1 < a.nT) {   // [A|B] after t1 steps, component-major so spins coalesce
      T* cp = ck + (size_t)(t1 / a.K - 1) * 12 * (size_t)a.nM + i;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        cp[(size_t)(3 * q) * a.nM] = cx[q]; cp[(size_t)(3 * q + 1) * a.nM] = cy[q]; cp[(size_t)(3 * q + 2) * a.nM] = cz[q];
      }
    }
  }
  T* A = (T*)a.A + ((int64_t)n * a.nM + i) * 9;
  T* Bo = (T*)a.B + ((int64_t)n * a.nM + i) * 3;
#pragma unroll
  for (int q = 0; q < 3; ++q) { A[q] = cx[q]; A[3 + q] = cy[q]; A[6 + q] = cz[q]; }
  Bo[0] = cx[3]; Bo[1] = cy[3]; Bo[2] = cz[3];
}

// Adjoint of beff2ab: the four columns of [A|B] are four magnetisation vectors driven by the same field, so a
// step is apply_bwd (time-reversed state + adjoint + field gradient F) per column with the relaxation handled
// here: only the B column carries the recovery term.  States come from un-relaxing the later state, re-
// synchronised with the forward checkpoints every K steps; with K == 1 the state before the rotation is instead
// recomputed from the previous checkpoint, so nothing is ever divided by E1/E2 (valid down to E = 0).
template <typename T, int POL>
__global__ void __launch_bounds__(128) beff2ab_bwd_kernel(const mrphy_beff2ab_args a) {
  const int n = blockIdx.y, i = blockIdx.x * 128 + threadIdx.x;
  if (i >= a.nM) return;
  const int nT = a.nT, K = a.K;
  const size_t nM = (size_t)a.nM;
  const double gam = ld_param(a.gamma, n, i), dt = ld_param(a.dt, n, 0);
  const T g = (T)(6.283185307179586476925286766559 * gam * dt);
  const T E1 = (T)ld_param(a.E1, n, i), E2 = (T)ld_param(a.E2, n, i);
  const T e1 = E1 - (T)1, e2 = E2 - (T)1;
  const T iE1 = K > 1 ? (T)1 / E1 : (T)0, iE2 = K > 1 ? (T)1 / E2 : (T)0;
  const T* Ap = (const T*)a.A + ((size_t)n * nM + i) * 9;
  const T* Bp = (const T*)a.B + ((size_t)n * nM + i) * 3;
  const T* gAp = (const T*)a.gA + ((size_t)n * nM + i) * 9;
  const T* gBp = (const T*)a.gB + ((size_t)n * nM + i) * 3;
  T cx[4], cy[4], cz[4], hx[4], hy[4], hz[4];
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    cx[q] = Ap[q]; cy[q] = Ap[3 + q]; cz[q] = Ap[6 + q];
    hx[q] = gAp[q]; hy[q] = gAp[3 + q]; hz[q] = gAp[6 + q];
  }
  cx[3] = Bp[0]; cy[3] = Bp[1]; cz[3] = Bp[2];
  hx[3] = gBp[0]; hy[3] = gBp[1]; hz[3] = gBp[2];
  const T* Bf = (const T*)a.Beff + (int64_t)n * a.B_sn + (int64_t)i * a.B_sm;
  T* G = (T*)a.gBeff + ((size_t)n * nM + i) * (size_t)nT * 3;
  const T* ck = (const T*)a.ckpt + (size_t)n * ((nT - 1) / K) * 12 * nM + i;
  SpinConst<T, 1> kd;   // apply_bwd<RELAX=false> never reads it
  kd.e1 = kd.e2 = kd.e1i = (T)0; kd.iE1 = kd.iE2 = (T)1;
  T sE1 = 0, sE2 = 0, sg = 0;
  for (int t = nT - 1; t >= 0; --t) {
    const T Bx = Bf[3 * t], By = Bf[3 * t + 1], Bz = Bf[3 * t + 2];
    const T bx = g * Bx, by = g * By, bz = g * Bz;
    const RotCoef<T> r = rot_coef<T, POL>(bx, by, bz);
    T Fx = 0, Fy = 0, Fz = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      T tx, ty, tz;   // the column after the rotation, before the relaxation, of step t
      if (K == 1) {
        if (t > 0) {
          const T* cp = ck + (size_t)(t - 1) * 12 * nM;
          tx = cp[(size_t)(3 * q) * nM]; ty = cp[(size_t)(3 * q + 1) * nM]; tz = cp[(size_t)(3 * q + 2) * nM];
        } else {
          tx = q == 0; ty = q == 1; tz = q == 2;
        }
        apply_fwd<T, false>(r, bx, by, bz, (T)0, (T)0, tx, ty, tz);
      } else {
        tx = cx[q] * iE2; ty = cy[q] * iE2; tz = (q == 3 ? cz[q] + e1 : cz[q]) * iE1;
      }
      sE2 = fma_(hx[q], tx, fma_(hy[q], ty, sE2));
      sE1 = fma_(hz[q], q == 3 ? tz - (T)1 : tz, sE1);
      T gx = fma_(e2, hx[q], hx[q]), gy = fma_(e2, hy[q], hy[q]), gz = fma_(e1, hz[q], hz[q]);
      T fx, fy, fz;
      apply_bwd<T, false, 1>(kd, r, bx, by, bz, tx, ty, tz, gx, gy, gz, fx, fy, fz);
      cx[q] = tx; cy[q] = ty; cz[q] = tz;
      hx[q] = gx; hy[q] = gy; hz[q] = gz;
      Fx += fx; Fy += fy; Fz += fz;
    }
    G[3 * t] = -g * Fx; G[3 * t + 1] = -g * Fy; G[3 * t + 2] = -g * Fz;   // dL/dBeff = -g F, dL/dg = -F.Beff
    sg -= fma_(Fx, Bx, fma_(Fy, By, Fz * Bz));
    if (K > 1 && t % K == 0 && t > 0) {
      const T* cp = ck + (size_t)(t / K - 1) * 12 * nM;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        cx[q] = cp[(size_t)(3 * q) * nM]; cy[q] = cp[(size_t)(3 * q + 1) * nM]; cz[q] = cp[(size_t)(3 * q + 2) * nM];
      }
    }
  }
  T* gp = (T*)a.gP + ((size_t)n * nM + i) * 3;
  gp[0] = sE1; gp[1] = sE2; gp[2] = sg;
}

// ---- beff2u-phi (beffective.py:14-37) --------------------------------------------------------------
// U = b / max(|b|, 1e-12) (F.normalize), Phi = -|b| g; the adjoint is the autograd of exactly that.
template <typename T>
__global__ void __launch_bounds__(256) beff2uphi_kernel(const mrphy_beff2uphi_args a) {
  const int n = blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
  if (i >= a.nM) return;
  const T* bp = (const T*)a.beff + (int64_t)n * a.b_sn + (int64_t)i * a.b_sm;
  const T x = bp[0], y = bp[1], z = bp[2];
  const T g = (T)ld_param(a.g, n, i);
  const T nrm = sqrt(x * x + y * y + z * z);
  const T inv = (T)1 / max(nrm, (T)1e-12);
  const size_t o = (size_t)n * a.nM + i;
  if (!a.adjoint) {
    T* u = (T*)a.U + o * 3;
    u[0] = x * inv; u[1] = y * inv; u[2] = z * inv;
    ((T*)a.Phi)[o] = -nrm * g;
    return;
  }
  T gx = 0, gy = 0, gz = 0, gn = 0;
  if (a.gU) {
    const T* gu = (const T*)a.gU + o * 3;
    gx = gu[0] * inv; gy = gu[1] * inv; gz = gu[2] * inv;
    if (nrm > (T)1e-12) gn = -(gx * x + gy * y + gz * z) * inv;   // d(1/|b|): -(gU.b)/|b|^2
  }
  if (a.gPhi) {
    const T gp = ((const T*)a.gPhi)[o];
    gn -= gp * g;
    if (a.gg) ((T*)a.gg)[o] = -gp * nrm;
  } else if (a.gg) {
    ((T*)a.gg)[o] = 0;
  }
  const T w = nrm > (T)0 ? gn / nrm : (T)0;   // d|b|/db = b/|b|, 0 at the origin (torch.norm)
  T* out = (T*)a.gbeff + o * 3;
  out[0] = fma_(w, x, gx); out[1] = fma_(w, y, gy); out[2] = fma_(w, z, gz);
}

// ---- freeprec (sims.py:325-421) --------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) freeprec_kernel(const mrphy_freeprec_args a) {
  const int n = blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
  if (i >= a.nM) return;
  const T* mp = (const T*)a.Mi + (int64_t)n * a.Mi_sn + (int64_t)i * a.Mi_sm;
  double x = mp[0], y = mp[1], z = mp[2];
  const double dur = ld_param(a.dur, n, 0);
  double c = 1.0, s = 0.0, E1 = 1.0, E2 = 1.0, rec = 0.0;
  if (a.df.ptr) sincos(-6.283185307179586476925286766559 * ld_param(a.df, n, i) * dur, &s, &c);
  if (a.T1.ptr) {
    const double x1 = -dur / ld_param(a.T1, n, i);
    E1 = exp(x1); E2 = exp(-dur / ld_param(a.T2, n, i)); rec = -expm1(x1);
  }
  double ox, oy, oz;
  if (!a.adjoint) {       // rotate then relax (sims.py:345-369)
    ox = E2 * (c * x - s * y); oy = E2 * (s * x + c * y); oz = E1 * z + rec;
  } else {                // transposed map on the incoming gradient (sims.py:403-419)
    const double gx = E2 * x, gy = E2 * y;
    ox = c * gx + s * gy; oy = c * gy - s * gx; oz = E1 * z;
  }
  T* op = (T*)a.Mo + ((int64_t)n * a.nM + i) * 3;
  op[0] = (T)ox; op[1] = (T)oy; op[2] = (T)oz;
}

}  // namespace mrphy

using namespace mrphy;

#define BEGIN_CALL()       \
  launch_count() = 0;      \
  err_buf()[0] = 0;        \
  if (!a) return fail(MRPHY_ERR_ARG, "null args%s")
#define DTYPE_OK(a) ((a)->dtype == MRPHY_F32 || (a)->dtype == MRPHY_F64)

// Per-spin gradients of rfgr2beff (autograd of beffective.py:137-167 w.r.t. loc, df, gamma, b1Map): reductions over TIME.
// One warp per spin, lanes along time: every iteration reads 32 consecutive (gBx, gBy, gBz) = 384 contiguous bytes of the
// spin's row; the waveform samples of those steps come from L1/L2 (every warp reads the same 20 KB).  3 + 1 + 2 NC running
// sums per lane, combined with shuffles at the end.
template <typename T, int NC>
__global__ void __launch_bounds__(256) rfgr2beff_spin_grads_kernel(const mrphy_rfgr2beff_args a) {
  const int lane = threadIdx.x & 31, n = blockIdx.y;
  const int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= a.nM) return;
  const T* G = (const T*)a.gBeff + ((size_t)n * a.nM + (size_t)i) * (size_t)a.nT * 3;
  const T* rf = (const T*)a.rf + (int64_t)n * a.rf_sn;
  const T* gr = (const T*)a.gr + (int64_t)n * a.gr_sn;
  const int64_t rf_sc = (a.flags & MRPHY_RF_COIL_DIM) ? a.rf_sc : 0;
  const bool want_b1 = a.gb1 != nullptr, want_loc = a.gloc != nullptr;
  T al[3] = {0, 0, 0}, az = 0, abr[NC], abi[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) abr[c] = abi[c] = (T)0;
#pragma unroll 2
  for (int t = lane; t < a.nT; t += 32) {
    const T gx = G[3 * (size_t)t], gy = G[3 * (size_t)t + 1], gz = G[3 * (size_t)t + 2];
    az += gz;
    if (want_loc) {
#pragma unroll
      for (int x = 0; x < 3; ++x) al[x] = fma(gr[x * a.gr_sx + t * a.gr_st], gz, al[x]);
    }
    if (want_b1) {
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        if (c < a.nC) {
          const T rx = rf[t * a.rf_st + c * rf_sc], ry = rf[a.rf_sx + t * a.rf_st + c * rf_sc];
          abr[c] = fma(rx, gx, fma(ry, gy, abr[c]));
          abi[c] = fma(rx, gy, fma(-ry, gx, abi[c]));
        }
      }
    }
  }
  auto wsum = [&](T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
  };
  az = wsum(az);
  const size_t s = (size_t)n * a.nM + (size_t)i;
  if (a.gsz && lane == 0) ((T*)a.gsz)[s] = az;
  if (want_loc) {
#pragma unroll
    for (int x = 0; x < 3; ++x) {
      const T v = wsum(al[x]);
      if (lane == 0) ((T*)a.gloc)[s * 3 + x] = v;
    }
  }
  if (want_b1) {
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      if (c < a.nC) {
        const T vr = wsum(abr[c]), vi = wsum(abi[c]);
        if (lane == 0) {
          ((T*)a.gb1)[(s * 2) * a.nC + c] = vr;
          ((T*)a.gb1)[(s * 2 + 1) * a.nC + c] = vi;
        }
      }
    }
  }
}

extern "C" size_t mrphy_sizeof_args(int which) {
  switch (which) {
    case 0: return sizeof(mrphy_param);
    case 1: return sizeof(mrphy_fused_args);
    case 2: return sizeof(mrphy_beff_args);
    case 3: return sizeof(mrphy_rfgr2beff_args);
    case 4: return sizeof(mrphy_beff2ab_args);
    case 5: return sizeof(mrphy_beff2uphi_args);
    case 6: return sizeof(mrphy_freeprec_args);
    case 7: return sizeof(mrphy_reparam_args);
    case 8: return sizeof(mrphy_mask_args);
    case 9: return sizeof(mrphy_clamp_args);
    case 10: return sizeof(mrphy_readout_args);
  }
  return 0;
}

extern "C" int mrphy_rfgr2beff(const mrphy_rfgr2beff_args* a, void* cuda_stream) {
  BEGIN_CALL();
  if (!DTYPE_OK(a) || a->N < 1 || a->N > 65535 || a->nM < 1 || a->nT < 1 || a->nC < 1) return fail(MRPHY_ERR_ARG, "bad sizes or dtype%s");
  if (!a->rf || !a->gr || !a->loc || !a->Beff) return fail(MRPHY_ERR_ARG, "rf, gr, loc, Beff are required%s");
  if (a->df.ptr && !a->gamma.ptr) return fail(MRPHY_ERR_ARG, "df needs gamma%s");
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const int tblocks = (a->nT + 1023) / 1024;
  const int64_t gx = (int64_t)((a->nM + 15) / 16) * tblocks;   // 16 spins per block (SPB)
  if (gx > 2147483647LL) return fail(MRPHY_ERR_ARG, "nM*nT too large for one launch%s");
  dim3 grid((unsigned)gx, a->N);
  timing_begin(st);
  const size_t es = a->dtype == MRPHY_F64 ? 8 : 4;
  const bool aligned = ((size_t)a->nT * 3 * es) % 16 == 0 && ((uintptr_t)a->Beff) % 16 == 0;
  const bool mc = a->b1 && a->nC > 1;
#define RFGR_LAUNCH(T, AL, MCV)                                                                       \
  do {                                                                                                \
    constexpr size_t smem_ = (size_t)((AL) ? 3 : 2) * 3 * 1024 * sizeof(T);                           \
    CK(cudaFuncSetAttribute(rfgr2beff_kernel<T, AL, MCV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_)); \
    rfgr2beff_kernel<T, AL, MCV><<<grid, 256, smem_, st>>>(*a, tblocks);                              \
  } while (0)
#define RFGR_PICK(T)                                                  \
  do {                                                                \
    if (aligned) { if (mc) RFGR_LAUNCH(T, true, true); else RFGR_LAUNCH(T, true, false); }   \
    else { if (mc) RFGR_LAUNCH(T, false, true); else RFGR_LAUNCH(T, false, false); }         \
  } while (0)
  if (a->dtype == MRPHY_F64) RFGR_PICK(double); else RFGR_PICK(float);
#undef RFGR_PICK
#undef RFGR_LAUNCH
  timing_end(st);
  ++launch_count();
  CK(cudaGetLastError());
  return MRPHY_OK;
}

namespace {
struct RBPlan { int NC, W, S, per_split, tblocks; };
// S spin ranges per (batch entry, 256-step block): about 4 blocks per SM in total, at least 64 spins per range
int rb_plan(const mrphy_rfgr2beff_args* a, RBPlan* p) {
  if (!a || !DTYPE_OK(a) || a->N < 1 || a->N > 65535 || a->nM < 1 || a->nT < 1 || a->nC < 1) return fail(MRPHY_ERR_ARG, "bad sizes or dtype%s");
  const int nc = a->b1 ? a->nC : 1;
  if (nc > 16) return fail(MRPHY_ERR_ARG, "more than 16 transmit coils with a b1Map are not supported%s");
  p->NC = nc <= 1 ? 1 : nc <= 2 ? 2 : nc <= 4 ? 4 : nc <= 8 ? 8 : 16;
  p->W = 2 * p->NC + 3;
  p->tblocks = (a->nT + 255) / 256;
  int S = (4 * 148 + p->tblocks * a->N - 1) / (p->tblocks * a->N);
  const int smax = (a->nM + 63) / 64;
  S = S < 1 ? 1 : (S > smax ? smax : S);
  if (S > 65535) S = 65535;
  p->per_split = ((a->nM + S - 1) / S + 31) / 32 * 32;
  p->S = (a->nM + p->per_split - 1) / p->per_split;
  return MRPHY_OK;
}

template <typename T, int NC>
int launch_rb(const mrphy_rfgr2beff_args* a, const RBPlan& p, cudaStream_t st) {
  const bool al = a->nT % 4 == 0 && ((uintptr_t)a->gBeff & 15) == 0;
  auto kern = al ? rfgr2beff_bwd_kernel<T, NC, true> : rfgr2beff_bwd_kernel<T, NC, false>;
  const size_t smem = al ? RBCfg<T, true>::smem(p.W) : RBCfg<T, false>::smem(p.W);
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  timing_begin(st);
  kern<<<dim3(p.tblocks, p.S, a->N), 256, smem, st>>>(*a, p.per_split);
  timing_end(st);
  ++launch_count();
  CK(cudaGetLastError());
  dim3 fgrid((a->nT + 31) / 32, p.W, a->N), fblock(32, 32);
  grad_finalize_kernel<T><<<fgrid, fblock, 0, st>>>((const T*)a->partials, p.S, p.W, p.NC, a->nC, a->nT,
                                                    (a->flags & MRPHY_RF_COIL_DIM) ? 1 : 0, a->b1 ? 0 : 1, (T)1,
                                                    (T*)a->grf, (T*)a->ggr);
  ++launch_count();
  CK(cudaGetLastError());
  return MRPHY_OK;
}

template <typename T>
int dispatch_rb(const mrphy_rfgr2beff_args* a, const RBPlan& p, cudaStream_t st) {
  switch (p.NC) {
    case 1: return launch_rb<T, 1>(a, p, st);
    case 2: return launch_rb<T, 2>(a, p, st);
    case 4: return launch_rb<T, 4>(a, p, st);
    case 8: return launch_rb<T, 8>(a, p, st);
    default: return launch_rb<T, 16>(a, p, st);
  }
}
}  // namespace

extern "C" size_t mrphy_rfgr2beff_partial_elems(const mrphy_rfgr2beff_args* a) {
  RBPlan p;
  if (rb_plan(a, &p) != MRPHY_OK) return 0;
  return (size_t)a->N * p.S * p.W * (size_t)a->nT;
}

extern "C" int mrphy_rfgr2beff_bwd(const mrphy_rfgr2beff_args* a, void* cuda_stream) {
  BEGIN_CALL();
  RBPlan p;
  const int rc = rb_plan(a, &p);
  if (rc) return rc;
  if (!a->loc || !a->gBeff || !a->grf || !a->ggr || !a->partials) return fail(MRPHY_ERR_ARG, "loc, gBeff, grf, ggr, partials are required%s");
  cudaStream_t st = (cudaStream_t)cuda_stream;
  return a->dtype == MRPHY_F64 ? dispatch_rb<double>(a, p, st) : dispatch_rb<float>(a, p, st);
}

static int check_beff2ab(const mrphy_beff2ab_args* a, bool bwd) {
  if (!DTYPE_OK(a) || a->N < 1 || a->N > 65535 || a->nM < 1 || a->nT < 1) return fail(MRPHY_ERR_ARG, "bad sizes or dtype%s");
  if (!a->Beff || !a->A || !a->B || !a->E1.ptr || !a->E2.ptr || !a->gamma.ptr || !a->dt.ptr) return fail(MRPHY_ERR_ARG, "Beff, A, B, E1, E2, gamma, dt are required%s");
  if ((a->ckpt || bwd) && a->K < 1) return fail(MRPHY_ERR_ARG, "K must be >= 1%s");
  if (bwd && (!a->ckpt || !a->gA || !a->gB || !a->gBeff || !a->gP)) return fail(MRPHY_ERR_ARG, "ckpt, gA, gB, gBeff, gP are required%s");
  return MRPHY_OK;
}

namespace {
template <typename T>
int launch_spin_grads(const mrphy_rfgr2beff_args* a, cudaStream_t st) {
  const int nc = (a->flags & MRPHY_RF_COIL_DIM) ? a->nC : 1;
  dim3 grid((unsigned)((a->nM + 7) / 8), a->N);
  if (nc <= 1) rfgr2beff_spin_grads_kernel<T, 1><<<grid, 256, 0, st>>>(*a);
  else if (nc <= 2) rfgr2beff_spin_grads_kernel<T, 2><<<grid, 256, 0, st>>>(*a);
  else if (nc <= 4) rfgr2beff_spin_grads_kernel<T, 4><<<grid, 256, 0, st>>>(*a);
  else if (nc <= 8) rfgr2beff_spin_grads_kernel<T, 8><<<grid, 256, 0, st>>>(*a);
  else rfgr2beff_spin_grads_kernel<T, 16><<<grid, 256, 0, st>>>(*a);
  ++launch_count();
  CK(cudaGetLastError());
  return MRPHY_OK;
}
}  // namespace

extern "C" int mrphy_rfgr2beff_spin_grads(const mrphy_rfgr2beff_args* a, void* cuda_stream) {
  BEGIN_CALL();
  if (!a) return fail(MRPHY_ERR_ARG, "null args%s");
  if (!DTYPE_OK(a) || a->N < 1 || a->nM < 1 || a->nT < 1 || a->nC < 1 || a->N > 65535)
    return fail(MRPHY_ERR_ARG, "bad sizes or dtype%s");
  if (!a->gBeff || !a->rf || !a->gr) return fail(MRPHY_ERR_ARG, "gBeff, rf and gr are required%s");
  if (!a->gloc && !a->gsz && !a->gb1) return MRPHY_OK;
  if (a->nC > 16) return fail(MRPHY_ERR_ARG, "more than 16 transmit coils are not supported%s");
  cudaStream_t st = (cudaStream_t)cuda_stream;
  return a->dtype == MRPHY_F64 ? launch_spin_grads<double>(a, st) : launch_spin_grads<float>(a, st);
}

extern "C" size_t mrphy_beff2ab_ckpt_elems(const mrphy_beff2ab_args* a) {
  if (!a || a->K < 1 || a->nT < 1) return 0;
  const size_t n = (size_t)a->N * (size_t)((a->nT - 1) / a->K) * 12 * (size_t)a->nM;
  return n ? n : 1;
}

template <bool BWD>
static int launch_beff2ab(const mrphy_beff2ab_args* a, cudaStream_t st) {
  dim3 grid((a->nM + 127) / 128, a->N);
  const bool precise = (a->flags & MRPHY_TRIG_PRECISE) != 0;
  timing_begin(st);
  if (BWD) {
    if (a->dtype == MRPHY_F64) beff2ab_bwd_kernel<double, TRIG_FAST><<<grid, 128, 0, st>>>(*a);
    else if (precise) beff2ab_bwd_kernel<float, TRIG_PRECISE><<<grid, 128, 0, st>>>(*a);
    else beff2ab_bwd_kernel<float, TRIG_FAST><<<grid, 128, 0, st>>>(*a);
  } else {
    if (a->dtype == MRPHY_F64) beff2ab_kernel<double, TRIG_FAST><<<grid, 128, 0, st>>>(*a);
    else if (precise) beff2ab_kernel<float, TRIG_PRECISE><<<grid, 128, 0, st>>>(*a);
    else beff2ab_kernel<float, TRIG_FAST><<<grid, 128, 0, st>>>(*a);
  }
  timing_end(st);
  ++launch_count();
  CK(cudaGetLastError());
  return MRPHY_OK;
}

extern "C" int mrphy_beff2ab(const mrphy_beff2ab_args* a, void* cuda_stream) {
  BEGIN_CALL();
  const int rc = check_beff2ab(a, false);
  return rc ? rc : launch_beff2ab<false>(a, (cudaStream_t)cuda_stream);
}

extern "C" int mrphy_beff2ab_bwd(const mrphy_beff2ab_args* a, void* cuda_stream) {
  BEGIN_CALL();
  const int rc = check_beff2ab(a, true);
  return rc ? rc : launch_beff2ab<true>(a, (cudaStream_t)cuda_stream);
}

extern "C" int mrphy_beff2uphi(const mrphy_beff2uphi_args* a, void* cuda_stream) {
  BEGIN_CALL();
  if (!DTYPE_OK(a) || a->N < 1 || a->N > 65535 || a->nM < 1) return fail(MRPHY_ERR_ARG, "bad sizes or dtype%s");
  if (!a->beff || !a->g.ptr) return fail(MRPHY_ERR_ARG, "beff and g are required%s");
  if (!a->adjoint && (!a->U || !a->Phi)) return fail(MRPHY_ERR_ARG, "U and Phi are required%s");
  if (a->adjoint && !a->gbeff) return fail(MRPHY_ERR_ARG, "gbeff is required%s");
  cudaStream_t st = (cudaStream_t)cuda_stream;
  dim3 grid((a->nM + 255) / 256, a->N);
  if (a->dtype == MRPHY_F64) beff2uphi_kernel<double><<<grid, 256, 0, st>>>(*a);
  else beff2uphi_kernel<float><<<grid, 256, 0, st>>>(*a);
  ++launch_count();
  CK(cudaGetLastError());
  return MRPHY_OK;
}

extern "C" int mrphy_freeprec(const mrphy_freeprec_args* a, void* cuda_stream) {
  BEGIN_CALL();
  if (!DTYPE_OK(a) || a->N < 1 || a->N > 65535 || a->nM < 1) return fail(MRPHY_ERR_ARG, "bad sizes or dtype%s");
  if (!a->Mi || !a->Mo || !a->dur.ptr) return fail(MRPHY_ERR_ARG, "Mi, Mo, dur are required%s");
  if ((a->T1.ptr == nullptr) != (a->T2.ptr == nullptr)) return fail(MRPHY_ERR_ARG, "T1 and T2: both or neither%s");
  cudaStream_t st = (cudaStream_t)cuda_stream;
  dim3 grid((a->nM + 255) / 256, a->N);
  if (a->dtype == MRPHY_F64) freeprec_kernel<double><<<grid, 256, 0, st>>>(*a);
  else freeprec_kernel<float><<<grid, 256, 0, st>>>(*a);
  ++launch_count();
  CK(cudaGetLastError());
  return MRPHY_OK;
}
