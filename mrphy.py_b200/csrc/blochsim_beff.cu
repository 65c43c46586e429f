// Explicit-field Bloch simulation for sm_100a: the API-faithful replacement of sims.BlochSim
// (sims.py:24-269) for callers that pass a dense Beff (N,nM,nT,3).  HBM-bound: 12 B/spin.step
// read forward; 12 B read + 12 B written backward (fp32).  Each warp owns 32 spins and streams
// [32 spins] x [192-byte] tiles of their Beff rows through a ring in shared memory with cp.async;
// one thread then walks its own row.  The backward pass overwrites the tile in place with
// dL/dBeff and streams it back out the same way.  States are not stored: time-reversed
// reconstruction + checkpoints every K steps, as in the fused path.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <type_traits>

#include "../../include/mrphy_b200.h"
#include "abi_common.cuh"
#include "bloch_math.cuh"

namespace mrphy {

constexpr int EBLK = 128;
constexpr int EWARP = EBLK / 32;

template <typename T> struct EArgs {
  int N, nM, nT, K, nCk;
  const T* Mi; int64_t Mi_sn, Mi_sm;
  const T* B; int64_t B_sn, B_sm;
  mrphy_param T1, T2, gamma, dt;
  T* Mo; T* ckpt;
  const T* gMo; int64_t gMo_sn, gMo_sm;
  T* gMi; T* gB;
};

template <typename T, bool RELAX>
__device__ __forceinline__ void load_consts(const EArgs<T>& a, int n, int i, SpinConst<T, 1>& k, T& g) {
  const double gam = ld_param(a.gamma, n, i), dt = ld_param(a.dt, n, 0);
  const double t1 = RELAX ? ld_param(a.T1, n, i) : 1.0, t2 = RELAX ? ld_param(a.T2, n, i) : 1.0;
  make_consts<T, 1>(k, gam, dt, RELAX, t1, t2, 0.0, (T)0, (T)0, (T)0, nullptr, nullptr);
  g = (T)(6.283185307179586476925286766559 * gam * dt);   // sims.py:62
}

// ------------------------------------------------------------------------------------------
// Tile pipeline.  A tile row is 192 data bytes (16 fp32 steps / 8 fp64 steps) + 16 bytes pad = 208-byte pitch, so that
//  * the warp fills it with cp.async straight from HBM, double-buffered: tile k+1 is in flight while tile k is consumed,
//    no registers staged;
//  * each thread reads its own row with LDS.128 without bank conflicts (20*r mod 32 hits 8 distinct quads);
//  * the backward overwrites the row in place with dL/dBeff and the warp streams it out with coalesced stores.
// ALIGNED (every Beff row starts on 16 bytes: rows_aligned16) moves 16-byte chunks (LDGSTS.128, 128-bit stores); other
// rows move element by element into the same layout, which needs only the element alignment every tensor has.
constexpr int NST = 2;     // tiles in the per-warp ring (NST - 1 in flight while one is consumed)
constexpr int ROWB = 192, PITCHB = ROWB + 16;   // pitch 13 x 16 B: odd

template <int E>           // one copy of E bytes: 16 with .cg (L2 only), 4 or 8 with .ca (the only form for < 16 B)
__device__ __forceinline__ void cp_async(void* smem_dst, const void* gmem_src) {
  if constexpr (E == 16)
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src)
                 : "memory");
  else
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src),
                 "n"(E) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// unit of the warp-cooperative tile copies: a 16-byte chunk on aligned rows, one element otherwise
template <typename T, bool ALIGNED> struct TileCopy {
  using V = std::conditional_t<ALIGNED, float4, T>;
  static constexpr int LG = ALIGNED ? 4 : (sizeof(T) == 8 ? 3 : 2), E = 1 << LG;   // bytes per copy: 16, 8 or 4
  static constexpr int CHUNKS = ROWB / E;                                           // copies per full row
  static_assert(sizeof(V) == E, "copy unit");
};

// warp-cooperative async copy of rows [i0, i0+32) x bytes [t0*3*sizeof(T), +nbytes) into `tile`
template <typename T, bool ALIGNED, int ROWS = 32>
__device__ __forceinline__ void tile_load_async(const T* __restrict__ B, int64_t B_sm, int i0, int nM, int t0, int nbytes,
                                                unsigned char* tile, int lane) {
  using C = TileCopy<T, ALIGNED>;
  constexpr int E = C::E, CHUNKS = C::CHUNKS;
  const int nch = nbytes >> C::LG;         // chunks per row in this tile
  const unsigned char* base = reinterpret_cast<const unsigned char*>(B + (int64_t)t0 * 3);
  const int64_t rowb = B_sm * (int64_t)sizeof(T);
  // full tile of 16-byte chunks: compile-time divisor, 12 copies per lane (per 32 rows).  Element copies always take the
  // loop below: unrolled, their 24 or 48 copies per lane would hold as many addresses in registers.
  if (ALIGNED && nch == CHUNKS) {
#pragma unroll
    for (int k = 0; k < CHUNKS * ROWS / 32; ++k) {
      const int q = k * 32 + lane, r = q / CHUNKS, c = q - r * CHUNKS;
      cp_async<E>(tile + r * PITCHB + c * E, base + (int64_t)min(i0 + r, nM - 1) * rowb + c * E);
    }
    return;
  }
  for (int q = lane; q < ROWS * nch; q += 32) {
    const int r = q / nch, c = q - r * nch;
    cp_async<E>(tile + r * PITCHB + c * E, base + (int64_t)min(i0 + r, nM - 1) * rowb + c * E);
  }
}
template <typename T, bool ALIGNED, int ROWS = 32>
__device__ __forceinline__ void tile_store(T* __restrict__ G, int64_t G_sm, int i0, int nM, int t0, int nbytes,
                                           const unsigned char* tile, int lane) {
  using C = TileCopy<T, ALIGNED>;
  using V = typename C::V;
  constexpr int E = C::E, CHUNKS = C::CHUNKS;
  const int nch = nbytes >> C::LG;
  unsigned char* base = reinterpret_cast<unsigned char*>(G + (int64_t)t0 * 3);
  const int64_t rowb = G_sm * (int64_t)sizeof(T);
  if (ALIGNED && nch == CHUNKS) {
#pragma unroll
    for (int k = 0; k < CHUNKS * ROWS / 32; ++k) {
      const int q = k * 32 + lane, r = q / CHUNKS, c = q - r * CHUNKS;
      if (i0 + r < nM)
        *reinterpret_cast<V*>(base + (int64_t)(i0 + r) * rowb + c * E) = *reinterpret_cast<const V*>(tile + r * PITCHB + c * E);
    }
    return;
  }
  for (int q = lane; q < ROWS * nch; q += 32) {
    const int r = q / nch, c = q - r * nch;
    if (i0 + r < nM)
      *reinterpret_cast<V*>(base + (int64_t)(i0 + r) * rowb + c * E) = *reinterpret_cast<const V*>(tile + r * PITCHB + c * E);
  }
}

template <typename T, int POL, bool RELAX, bool BWD, bool ALIGNED>
__global__ void __launch_bounds__(EBLK) beff_v2_kernel(const EArgs<T> a, const int need_gmi, const int need_gb) {
  constexpr int TB = ROWB / (3 * (int)sizeof(T));      // steps per tile: 16 (fp32), 8 (fp64)
  constexpr int PITCH = PITCHB / (int)sizeof(T);       // row pitch in elements
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n = blockIdx.y;
  unsigned char* buf0 = smem_raw + (size_t)warp * NST * 32 * PITCHB;
  const int nM = a.nM, nT = a.nT, K = a.K;
  const int i0 = (blockIdx.x * EWARP + warp) * 32;
  if (i0 >= nM) return;
  const bool ok = i0 + lane < nM;
  const int i = ok ? i0 + lane : nM - 1;
  SpinConst<T, 1> k;
  T g;
  load_consts<T, RELAX>(a, n, i, k, g);
  T mx, my, mz, hx = 0, hy = 0, hz = 0;
  if (BWD) {
    const T* mp = a.Mo + ((size_t)n * nM + i) * 3;
    mx = mp[0]; my = mp[1]; mz = mp[2];
    const T* gp = a.gMo + (int64_t)n * a.gMo_sn + (int64_t)i * a.gMo_sm;
    hx = gp[0]; hy = gp[1]; hz = gp[2];
  } else {
    const T* mp = a.Mi + (int64_t)n * a.Mi_sn + (int64_t)i * a.Mi_sm;
    mx = mp[0]; my = mp[1]; mz = mp[2];
  }
  const T* Bn = a.B + (int64_t)n * a.B_sn;
  T* Gn = BWD ? a.gB + (size_t)n * nM * (size_t)nT * 3 : nullptr;
  const T ng = -g;
  // Checkpoints by a running counter instead of a test (and an integer division for the slot) at every step: `until` steps
  // are left before the next checkpoint, whose slot pointer moves by one stride each time.  A 4-step group that contains
  // no checkpoint (15 of 16 at K = 64) is a clean run of steps; the others take the per-step path.
  const size_t ck_stride = 3 * (size_t)nM;
  int until;                 // forward: steps until state after (slot+1)*K steps is stored; backward: steps until resync
  T* ckp;                    // slot the next checkpoint is written to / read from (this spin's x entry)
  if (!BWD) {
    until = K;
    ckp = a.ckpt + (size_t)n * a.nCk * ck_stride + i;
  } else {
    const int last = ((nT - 1) / K) * K;           // the backward resyncs when it has undone step `last`, `last - K`, ...
    until = nT - last;
    ckp = a.ckpt + ((size_t)n * a.nCk + (last / K - 1)) * ck_stride + i;     // only dereferenced when last > 0
  }
  const int ntiles = (nT + TB - 1) / TB;
  auto tile_t0 = [&](int q) { return (BWD ? ntiles - 1 - q : q) * TB; };     // q-th tile in processing order
  auto tile_len = [&](int q) { return min(TB, nT - tile_t0(q)); };
  // ring of NST tiles: NST - 1 loads in flight while one tile is consumed; every iteration commits exactly one group (an
  // empty one past the end), so "all but the newest NST - 1 groups" is always "tile q has landed"
#pragma unroll
  for (int p = 0; p < NST - 1; ++p) {
    if (p < ntiles) tile_load_async<T, ALIGNED>(Bn, a.B_sm, i0, nM, tile_t0(p), tile_len(p) * 3 * (int)sizeof(T), buf0 + p * 32 * PITCHB, lane);
    cp_async_commit();
  }
  for (int q = 0; q < ntiles; ++q) {
    unsigned char* cur = buf0 + (q % NST) * 32 * PITCHB;
    if (q + NST - 1 < ntiles)
      tile_load_async<T, ALIGNED>(Bn, a.B_sm, i0, nM, tile_t0(q + NST - 1), tile_len(q + NST - 1) * 3 * (int)sizeof(T),
                         buf0 + ((q + NST - 1) % NST) * 32 * PITCHB, lane);
    cp_async_commit();
    cp_async_wait<NST - 1>();
    __syncwarp();
    T* row = reinterpret_cast<T*>(cur) + lane * PITCH;
    const int t0 = tile_t0(q), len = tile_len(q);
    // 48 bytes = GS steps per group, moved with three conflict-free 128-bit accesses
    constexpr int GS = 16 / (int)sizeof(T);            // 4 (fp32) or 2 (fp64) steps
    constexpr int GV = 3 * GS;                         // values per group
    // Aligned rows hold a multiple of GS steps.  Otherwise the last group of the last tile in time can hold gl < GS steps
    // (it is the first group the backward processes): it runs its gl steps on the per-step path and leaves the rest of v,
    // stale data inside the row, untouched.  No zero padding: a zero-field step is not the identity under relaxation.
    auto group_len = [&](int j0) { return ALIGNED ? GS : min(GS, len - j0); };
    if (!BWD) {
      for (int j0 = 0; j0 < len; j0 += GS) {
        const int gl = group_len(j0);
        T v[GV];
        float4* v4 = reinterpret_cast<float4*>(v);
        const float4* src = reinterpret_cast<const float4*>(row + 3 * j0);
        v4[0] = src[0]; v4[1] = src[1]; v4[2] = src[2];
        if (until > GS && gl == GS) {
#pragma unroll
          for (int u = 0; u < GS; ++u)
            step_fwd<T, POL, RELAX>(g * v[3 * u], g * v[3 * u + 1], g * v[3 * u + 2], k.e1, k.e2, mx, my, mz);
          until -= GS;
        } else {
#pragma unroll
          for (int u = 0; u < GS; ++u) {
            if (u >= gl) break;
            step_fwd<T, POL, RELAX>(g * v[3 * u], g * v[3 * u + 1], g * v[3 * u + 2], k.e1, k.e2, mx, my, mz);
            if (--until == 0) {
              if (t0 + j0 + u + 1 < nT && ok) {
                ckp[0] = mx; ckp[(size_t)nM] = my; ckp[2 * (size_t)nM] = mz;
              }
              ckp += ck_stride;
              until = K;
            }
          }
        }
      }
    } else {
      for (int j0 = ALIGNED ? len - GS : (len - 1) / GS * GS; j0 >= 0; j0 -= GS) {
        const int gl = group_len(j0);
        T v[GV];
        float4* v4 = reinterpret_cast<float4*>(v);
        float4* src = reinterpret_cast<float4*>(row + 3 * j0);
        v4[0] = src[0]; v4[1] = src[1]; v4[2] = src[2];
        if (until > GS && gl == GS) {
#pragma unroll
          for (int u = GS - 1; u >= 0; --u) {
            T Fx, Fy, Fz;
            step_bwd<T, POL, RELAX, 1>(k, g * v[3 * u], g * v[3 * u + 1], g * v[3 * u + 2], mx, my, mz, hx, hy, hz,
                                       Fx, Fy, Fz);
            v[3 * u] = ng * Fx;       // dL/dBeff = -2*pi*gamma*dt * F   (sims.py:194, 234-259)
            v[3 * u + 1] = ng * Fy;
            v[3 * u + 2] = ng * Fz;
          }
          until -= GS;
        } else {
#pragma unroll
          for (int u = GS - 1; u >= 0; --u) {
            if (u >= gl) continue;
            T Fx, Fy, Fz;
            step_bwd<T, POL, RELAX, 1>(k, g * v[3 * u], g * v[3 * u + 1], g * v[3 * u + 2], mx, my, mz, hx, hy, hz,
                                       Fx, Fy, Fz);
            v[3 * u] = ng * Fx;
            v[3 * u + 1] = ng * Fy;
            v[3 * u + 2] = ng * Fz;
            if (--until == 0) {     // step t = t0 + j0 + u undone: the state is now the one after t steps
              if (t0 + j0 + u > 0) {
                mx = ckp[0]; my = ckp[(size_t)nM]; mz = ckp[2 * (size_t)nM];
              }
              ckp -= ck_stride;
              until = K;
            }
          }
        }
        src[0] = v4[0]; src[1] = v4[1]; src[2] = v4[2];
      }
      __syncwarp();
      if (need_gb) tile_store<T, ALIGNED>(Gn, (int64_t)nT * 3, i0, nM, t0, len * 3 * (int)sizeof(T), cur, lane);
    }
    __syncwarp();   // the buffer is refilled two iterations later, after every lane has left it
  }
  if (!BWD && ok) {
    T* op = a.Mo + ((size_t)n * nM + i) * 3;
    op[0] = mx; op[1] = my; op[2] = mz;
  }
  if (BWD && need_gmi && ok) {
    T* op = a.gMi + ((size_t)n * nM + i) * 3;
    op[0] = hx; op[1] = hy; op[2] = hz;
  }
}

}  // namespace mrphy

using namespace mrphy;

namespace {

int check_beff(const mrphy_beff_args* a, bool bwd) {
  if (!a) return fail(MRPHY_ERR_ARG, "null args%s");
  if (a->dtype != MRPHY_F32 && a->dtype != MRPHY_F64) return fail(MRPHY_ERR_ARG, "dtype must be MRPHY_F32 or MRPHY_F64%s");
  if (a->N < 1 || a->nM < 1 || a->nT < 1 || a->N > 65535) return fail(MRPHY_ERR_ARG, "need 1 <= N <= 65535, nM >= 1, nT >= 1%s");
  if (a->K < 1) return fail(MRPHY_ERR_ARG, "checkpoint interval K must be >= 1%s");
  if (!a->Beff || !a->gamma.ptr || !a->dt.ptr || !a->Mo || !a->ckpt) return fail(MRPHY_ERR_ARG, "Beff, gamma, dt, Mo, ckpt are required%s");
  if ((a->T1.ptr == nullptr) != (a->T2.ptr == nullptr)) return fail(MRPHY_ERR_ARG, "T1 and T2: both or neither (sims.py:68)%s");
  if (a->B_st != 3) return fail(MRPHY_ERR_ARG, "Beff must be contiguous over (nT, xyz)%s");
  if (!bwd && !a->Mi) return fail(MRPHY_ERR_ARG, "Mi is null%s");
  if (bwd && !a->gMo) return fail(MRPHY_ERR_ARG, "gMo is null%s");
  if (bwd && (a->flags & MRPHY_NEED_GMI) && !a->gMi) return fail(MRPHY_ERR_ARG, "gMi is null but MRPHY_NEED_GMI is set%s");
  if (bwd && (a->flags & MRPHY_NEED_GBEFF) && !a->gBeff) return fail(MRPHY_ERR_ARG, "gBeff is null but MRPHY_NEED_GBEFF is set%s");
  return MRPHY_OK;
}

template <typename T>
EArgs<T> make_eargs(const mrphy_beff_args* a) {
  EArgs<T> e;
  memset(&e, 0, sizeof(e));
  e.N = a->N; e.nM = a->nM; e.nT = a->nT; e.K = a->K; e.nCk = (a->nT - 1) / a->K;
  e.Mi = (const T*)a->Mi; e.Mi_sn = a->Mi_sn; e.Mi_sm = a->Mi_sm;
  e.B = (const T*)a->Beff; e.B_sn = a->B_sn; e.B_sm = a->B_sm;
  e.T1 = a->T1; e.T2 = a->T2; e.gamma = a->gamma; e.dt = a->dt;
  e.Mo = (T*)a->Mo; e.ckpt = (T*)a->ckpt;
  e.gMo = (const T*)a->gMo; e.gMo_sn = a->gMo_sn; e.gMo_sm = a->gMo_sm;
  e.gMi = (T*)a->gMi; e.gB = (T*)a->gBeff;
  return e;
}

template <typename T>
bool rows_aligned16(const mrphy_beff_args* a) {
  const size_t es = sizeof(T);
  return ((size_t)a->nT * 3 * es) % 16 == 0 && ((size_t)a->B_sm * es) % 16 == 0 && ((size_t)a->B_sn * es) % 16 == 0 &&
         ((uintptr_t)a->Beff) % 16 == 0 && (!a->gBeff || ((uintptr_t)a->gBeff) % 16 == 0);
}

template <typename T, int POL, bool RELAX>
int launch_e(bool bwd, const mrphy_beff_args* a, cudaStream_t st) {
  const bool al = rows_aligned16<T>(a);
  auto kern = bwd ? (al ? beff_v2_kernel<T, POL, RELAX, true, true> : beff_v2_kernel<T, POL, RELAX, true, false>)
                  : (al ? beff_v2_kernel<T, POL, RELAX, false, true> : beff_v2_kernel<T, POL, RELAX, false, false>);
  constexpr size_t smem = (size_t)EWARP * NST * 32 * PITCHB;
  const int gmi = bwd && (a->flags & MRPHY_NEED_GMI) ? 1 : 0, gb = bwd && (a->flags & MRPHY_NEED_GBEFF) ? 1 : 0;
  dim3 grid((a->nM + EBLK - 1) / EBLK, a->N);
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  timing_begin(st);
  kern<<<grid, EBLK, smem, st>>>(make_eargs<T>(a), gmi, gb);
  timing_end(st);
  ++launch_count();
  CK(cudaGetLastError());
  return MRPHY_OK;
}

template <typename T>
int dispatch_e(bool bwd, const mrphy_beff_args* a, cudaStream_t st) {
  const bool relax = a->T1.ptr != nullptr;
  const bool precise = (a->flags & MRPHY_TRIG_PRECISE) != 0 && sizeof(T) == 4;
  if (precise) return relax ? launch_e<T, TRIG_PRECISE, true>(bwd, a, st) : launch_e<T, TRIG_PRECISE, false>(bwd, a, st);
  return relax ? launch_e<T, TRIG_FAST, true>(bwd, a, st) : launch_e<T, TRIG_FAST, false>(bwd, a, st);
}

}  // namespace

extern "C" size_t mrphy_beff_ckpt_elems(const mrphy_beff_args* a) {
  if (!a || a->K < 1 || a->nT < 1) return 0;
  const size_t n = (size_t)a->N * (size_t)((a->nT - 1) / a->K) * 3 * (size_t)a->nM;
  return n ? n : 1;
}

extern "C" int mrphy_blochsim_beff_fwd(const mrphy_beff_args* a, void* cuda_stream) {
  launch_count() = 0;
  err_buf()[0] = 0;
  int rc = check_beff(a, false);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)cuda_stream;
  return a->dtype == MRPHY_F64 ? dispatch_e<double>(false, a, st) : dispatch_e<float>(false, a, st);
}

extern "C" int mrphy_blochsim_beff_bwd(const mrphy_beff_args* a, void* cuda_stream) {
  launch_count() = 0;
  err_buf()[0] = 0;
  int rc = check_beff(a, true);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)cuda_stream;
  return a->dtype == MRPHY_F64 ? dispatch_e<double>(true, a, st) : dispatch_e<float>(true, a, st);
}
