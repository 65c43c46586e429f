// Fused Bloch simulation for sm_100a: waveform -> Beff -> (u,phi) -> Rodrigues -> relaxation for
// all nT steps with the magnetisation in registers, and its adjoint with on-chip reduction of
// dL/drf, dL/dgr over spins.  Replaces beffective.rfgr2beff (beffective.py:107-168) +
// sims.BlochSim.forward/backward (sims.py:31-269) + the autograd of rfgr2beff.
//
// Kernels in this file
//   pack_waveform_kernel      rf (N,2,nT[,nC]), gr (N,3,nT) -> wave[N][chunk][W][TCP]  (W = 2*NC+3)
//   fused_fwd_kernel<T,..>    one spin, or two spins packed in an f2 (FFMA2), per thread; checkpoint every K steps
//                             REC (OPT_RECORD): also the state every `every` steps (Mt, rec_store)
//                             RD (OPT_READOUT): instead the receive signal of those states summed over the CTA's spins
//                             (ro_accum, ro_flush) into a per-CTA slot
//   fused_bwd_kernel<T,..>    time-reversed state reconstruction + adjoint + spin reduction (only the gradient rows
//                             asked for: ROWS); tiles owned through SM-aware virtual CTA ids (SCHED_*)
//                             SG: also the per-spin sums over time behind dL/dloc, dL/ddf, dL/db1Map (sg_fold)
//                             REC: dL/dMt joins the adjoint at the recorded steps (rec_load)
//                             RD: the adjoint of the signal joins there instead (ro_adjoint), and dL/drx per spin
//   fused_fwd_tc_kernel<..>   fp32, >= 4 coils: the transmit field on the tensor cores (below); REC as fused_fwd_kernel
//   grad_finalize_kernel<T>   deterministic sum of the per-CTA partials, reference layout out (grad_finalize.cuh)
//   readout_finalize_kernel<T> RD: deterministic sum of the per-CTA signal slots -> S
//
// Data layout in HBM (T = float | double):
//   wave      [N][nChunks][W][TCP]   one chunk = K steps (TCP = K rounded up to 4): a chunk is
//                                    ONE contiguous 16-byte-aligned block -> one 1-D TMA bulk copy
//   ckpt      [N][nChunks-1][3][nM]  state after (c+1)*K steps, SoA so warps store 128-B lines
//   Mt, gMt   [N][nR][3][nM]         REC: state after (r+1)*every steps (lab frame) and its gradient, SoA likewise
//   S, gS     [N][2][nR][nRx]        RD: the signal and its gradient; slots of the forward [N][P][nR][2 nRx]
//   partials  [N][P][W][nT]          gradient partial sums, one slot per (virtual) CTA id, P ids per batch entry;
//                                    behind them 264 + P ints of scheduling state of the backward (SCHED_*)
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/mrphy_b200.h"
#include "abi_common.cuh"
#define MRPHY_VOTE_MASK 0xffffffffu   /* every loop of the fused kernels runs with all lanes of the warp (padding lanes compute too) */
#ifndef MRPHY_TC_MIN_NC
#define MRPHY_TC_MIN_NC 4   /* fp32, this many coils or more: transmit field on the tensor cores (fused_*_tc_kernel) */
#endif
#include "bloch_math.cuh"
#include "ptx_helpers.cuh"
#include "tc_helpers.cuh"
#include "grad_finalize.cuh"

namespace mrphy {

// Max steps per staged waveform chunk (== max checkpoint interval).  fp32 single coil: 128 -- half the chunk transitions
// (barrier, mbarrier wait, checkpoint traffic) of 64: +0.6 % at C5, +0.8 % at C2, gradients move by 1e-6 relative (the
// time-reversed states are resynchronised half as often); the other kernels keep 64 (their staged rows are wider).
#ifndef MRPHY_TCMAX1
#define MRPHY_TCMAX1 128
#endif
constexpr int TCMAX = 64;
template <typename T, int NC> struct ChunkMax { static constexpr int v = (sizeof(T) == 4 && NC == 1) ? MRPHY_TCMAX1 : TCMAX; };

#ifdef MRPHY_CTA_TRACE
// measurement build only (profiles/cta_trace.py): per CTA of the backward kernel (SM id, start, end) in ns
__device__ unsigned long long g_cta_trace[8192][4];
__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ unsigned smid() {
  unsigned s;
  asm volatile("mov.u32 %0, %smid;" : "=r"(s));
  return s;
}
#endif

// value type of a thread: one spin (T) or two spins packed for FFMA2 (f2)
template <typename T, int PK> struct Pack { typedef T type; };
template <> struct Pack<float, 2> { typedef f2 type; };

// Staged waveform layout of one chunk.  Up to 11 rows (44 bytes per step): row-major [W][TCP], a thread reads 4 steps of a row
// with one broadcast 128-bit load.  More rows (8 / 16 coils, fp64 with >= 2 coils): step-major [TCP][WS], WS = W padded to 4, so
// that the W samples of ONE step are ceil(W/4) 128-bit loads instead of W scalar ones.
template <typename T, int W> struct WaveLayout {
  static constexpr bool STEPMAJOR = W * sizeof(T) > 44;
  static constexpr int WS = STEPMAJOR ? ((W + 3) & ~3) : W;
};
// the W samples of step j of the staged chunk `wb`
template <typename T, int W>
__device__ __forceinline__ void load_step(const T* wb, int TCP, int j, T (&sv)[W]) {
  if constexpr (WaveLayout<T, W>::STEPMAJOR) {
    constexpr int WS = WaveLayout<T, W>::WS;
    T tmp[WS];
    const float4* src = reinterpret_cast<const float4*>(wb + (size_t)j * WS);
    float4* dst = reinterpret_cast<float4*>(tmp);
#pragma unroll
    for (int e = 0; e < WS * (int)sizeof(T) / 16; ++e) dst[e] = src[e];
#pragma unroll
    for (int w = 0; w < W; ++w) sv[w] = tmp[w];
  } else {
#pragma unroll
    for (int w = 0; w < W; ++w) sv[w] = wb[w * TCP + j];
  }
}

// steps per gradient-reduction tile (a CTA barrier every TR steps): the per-warp transposition tile [W][TR][32] is
// kept <= 10 KB; 11 KB with 4 coils (TR 8 instead of 4, still 4 CTAs per SM) and 20 KB with 8 and 16 coils
// (fp32 TR 8 / 4; 2 CTAs per SM -- measured 1.3x / 1.5x faster than TR 4 / 2 at twice the occupancy)
#ifndef MRPHY_RED_BUDGET
#define MRPHY_RED_BUDGET 10240
#endif
#ifndef MRPHY_NC2_MINB
#define MRPHY_NC2_MINB 14        // packed 2-coil forward: 64-thread CTAs per SM asked of the compiler: 72 registers and a 56-byte
                                 // spill frame beat 80 / 86 registers without one (measured 0.521 vs 0.588 / 0.598 ms at C2)
#endif
#ifndef MRPHY_WRED_TR_BYTES
#define MRPHY_WRED_TR_BYTES 64   // multi-coil backward: steps per reduction tile x sizeof(T)
#endif
#ifndef MRPHY_MC_MINB
#define MRPHY_MC_MINB 1         // multi-coil backward: minimum resident CTAs per SM asked of the compiler (register cap)
#endif
#ifndef MRPHY_BWD_MINB
#define MRPHY_BWD_MINB 8     // spin-packed backward: 128 registers, 8 CTAs (16 warps) per SM -- measured best of 6..10
#endif
#ifndef MRPHY_BWD_BLKT
#define MRPHY_BWD_BLKT 128   // threads per CTA of the spin-packed backward: one warp on each SM sub-partition, so the four
                             // schedulers of an SM always carry the same load (64-thread CTAs: 7 per SM = 4,4,3,3 warps)
#endif
constexpr int pick_tr(int W, int elem) {
  int tr = 16;
  // W == 7: two coils, two spins per thread -- 16 steps (14 KB per warp, 3 CTAs per SM) measured 8 % faster than 8 (4 CTAs)
  const int budget = W >= 19 ? 2 * MRPHY_RED_BUDGET : (W == 11 ? MRPHY_RED_BUDGET + 1024 : (W == 7 ? MRPHY_RED_BUDGET + 4096 : MRPHY_RED_BUDGET));
  while (tr > 1 && W * tr * 32 * elem > budget) tr >>= 1;
  return tr;
}

// dynamic shared memory layout of the backward kernel
// Single coil: the per-warp transposition tile holds the W = 5 weighted gradient terms of every (spin, step).
// Multi-coil (WRED): it holds only F = -dL/db (3 values + pad per spin and step, one 128-bit store per step instead of
// 2 NC + 3 scalar ones) and the per-spin weights (g*b1 of every coil, g*loc) sit beside it; they are applied in the reduce
// phase, where a lane owns ONE time step and sums over its share of the warp's spins (warp_tile_reduce_weighted).
template <typename T, int NC, int BLKT, int PK = 1> struct BwdSmem {
  static constexpr int W = 2 * NC + 3;
  static constexpr int NW = BLKT / 32;
  static constexpr bool WRED = NC > 1 && PK == 1;   // (two coils, two spins per thread: the single-coil scheme with 7 rows)
  static constexpr int TR = WRED ? MRPHY_WRED_TR_BYTES / (int)sizeof(T) : pick_tr(W, (int)sizeof(T));   // WRED: 16 (fp32), 8 (fp64)
  static constexpr int WP = (W + 3) & ~3;                                          // weights per spin, padded to 128-bit loads
  static constexpr int E16 = (int)sizeof(T) / 4;                                   // one F entry in 16-byte units
  static constexpr int P16 = TR * E16 + 1;                                         // per-spin pitch of the F tile (odd: conflict-free)
  static constexpr size_t red_bytes = WRED ? (size_t)NW * 32 * (P16 * 16 + WP * sizeof(T)) : (size_t)NW * W * TR * 32 * sizeof(T);
  static constexpr size_t wbuf = 0;                                                // T[2][W*TCMAX]
  static constexpr int WS = WaveLayout<T, W>::WS;
  static constexpr int TCM = ChunkMax<T, NC>::v;
  static constexpr size_t red = (2 * WS * TCM * sizeof(T) + 127) / 128 * 128;      // T[NW][W][TR][32]  |  F tiles + weights
  static constexpr size_t cta = (red + red_bytes + 15) / 16 * 16;                  // T[2][NW][W][TR] (double-buffered)
  static constexpr size_t bar = (cta + (size_t)2 * NW * W * TR * sizeof(T) + 15) / 16 * 16;   // uint64_t[2]
  static constexpr size_t bytes = bar + 16;
};

template <typename T> struct KArgs {
  int N, nM, nT, K, TCP, nChunks, P;
  int chunk_elems;     // elements of T per staged waveform chunk
  const T* Mi; int64_t Mi_sn, Mi_sm;
  const T* loc; int64_t loc_sn, loc_sm;
  const T* b1; int64_t b1_sn, b1_sm; int nC;
  mrphy_param df, T1, T2, gamma, dt;
  T* Mo;
  T* ckpt;
  const T* wave;
  const T* gMo; int64_t gMo_sn, gMo_sm;
  T* gMi;
  T* partials;
  int* sched;          // SM-aware tile ownership of the backward (null: CTA b owns tiles b, b+P, ...), see SCHED_* below
  int n_sm, c_per_sm;
  int* done;           // finished-CTA counters of grad_finalize_design_kernel, one per batch entry (null: no design tail); zeroed here
};
// per-spin gradient outputs of the SG backward (gloc, gsz, gb1 of mrphy_fused_args; each may be null).  A kernel parameter of its own behind
// the others, so that the kernels without per-spin gradients keep their parameter offsets.
template <typename T> struct SgOut {
  T* gloc; T* gsz; T* gb1;
  bool any() const { return gloc || gsz || gb1; }
};
// readout of the RD kernels (nRx, rx, S, gS, grx, S_work of mrphy_fused_args): the signal
// S[n][xy][r][k] = sum_i (cx + i cy)[n][i][k] (Mx + i My)[n][i] of the state after (r+1)*every steps (lab frame).  The
// forward sums its tiles into its own slot of `part` [N][P][nR][2 nRx]
// (P = gridDim.x; x values, then y values; readout_finalize_kernel sums the slots in a fixed order); the backward adds the
// adjoint of S to the adjoint state at the recorded steps (ro_adjoint) and, with grx, forms dL/drx per spin.
template <typename T> struct RoOut {
  const T* rx; int64_t rx_sn, rx_sm;   // (N,nM,2,nRx), inner (2,nRx) contiguous, or null: c = 1
  int nRx, every, nR;
  int rt;                              // fwd: records per flush, RO_COLS / (2 nRx)
  T* part;                             // fwd: per-CTA partial sums
  const T* gS;                         // bwd: dL/dS (N,2,nR,nRx) contiguous
  T* grx;                              // bwd: dL/drx (N,nM,2,nRx) contiguous, or null
};
// recorded magnetisation of the REC kernels (every, nR, Mt, gMt of mrphy_fused_args): the forward writes Mt, the backward reads dL/dMt, both
// [N][nR][3][nM] (SoA like the checkpoints), entry r = the state after (r+1)*every steps in the lab frame.  A kernel
// parameter of its own behind the others, like SgOut.  The readout of the RD kernels rides behind it (`ro`): appended to
// the last kernel parameter, it moves no parameter of the kernels without readout.
template <typename T> struct RecOut {
  T* Mt; const T* gMt;
  int every, nR;
  RoOut<T> ro;
};
// The option of fused_fwd_kernel, fused_fwd_tc_kernel and fused_bwd_kernel (template parameter OPT): none, record (REC) or
// readout (RD); a call takes at most one of them.
constexpr int OPT_NONE = 0, OPT_RECORD = 1, OPT_READOUT = 2;
// Dynamic shared memory of the readout, behind what the kernel already uses (runtime-sized by nRx; V = Pack<T, PK>::type):
//   forward   w V[2 nRx][BLKT]  |  tiles T[NW][32 columns][32 lanes]  |  ctab T[2][NW][32]
//   backward  w V[2 nRx][BLKT]  |  acc V[2 nRx][BLKT] (dL/drx sums)   |  gs T[records per chunk][2 nRx] (dL/dS of the chunk)
// A column of a forward tile is one (record, x|y, coil) value of the 32 lanes of the warp: 32 / (2 nRx) records per flush.
constexpr int RO_COLS = 32;
inline size_t ro_fwd_smem(int nRx, int BLKT, int vsz, int tsz) {
  return (size_t)2 * nRx * BLKT * vsz + (size_t)(BLKT / 32) * RO_COLS * 32 * tsz + (size_t)2 * (BLKT / 32) * 32 * tsz;
}
inline size_t ro_bwd_smem(int nRx, int BLKT, int vsz, int tsz, int nrc) {
  return (size_t)4 * nRx * BLKT * vsz + (size_t)nrc * 2 * nRx * tsz;
}

// Scheduling workspace of the backward kernel (ints, zeroed before every launch; lives behind the partial sums).
// The hardware spreads the P = c * n_sm co-resident CTAs breadth-first over the SMs, but not in blockIdx order (measured,
// profiles/cta_trace.py): with tiles owned by blockIdx some SMs end up with one tile more than ceil(tiles / n_sm) and
// the kernel waits for them.  Instead a CTA asks which SM it is on and which arrival it is there (rank), and serves the
// VIRTUAL id rank * n_sm + smid: ids, their tiles and their partial-sum slot are static, so the result stays bitwise
// reproducible whichever CTA serves an id.  Ids are claimed with a CAS, and a CTA that is done (or found no free home
// id: an SM with more than c arrivals) sweeps for unclaimed ids, so every id is served exactly once whatever the
// placement -- no waiting on other CTAs anywhere.
constexpr int SCHED_SM_SLOTS = 256;                     // [0, 256): arrivals per SM
constexpr int SCHED_NCLAIMED = 256;                     // [256]: ids claimed so far
constexpr int SCHED_CLAIM = 264;                        // [264, 264 + P): claim flag per id
__device__ __forceinline__ unsigned my_smid() {
  unsigned s;
  asm volatile("mov.u32 %0, %%smid;" : "=r"(s));
  return s;
}

__device__ __forceinline__ void load4(const float* p, float (&v)[4]) {
  const float4 q = *reinterpret_cast<const float4*>(p);
  v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
}
__device__ __forceinline__ void load4(const double* p, double (&v)[4]) {
  const double2 a = *reinterpret_cast<const double2*>(p);
  const double2 b = *reinterpret_cast<const double2*>(p + 2);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

// lane access for scalar / packed values
template <int Q> __device__ __forceinline__ float getq(f2 a) { return Q == 0 ? a.v.x : a.v.y; }
template <int Q> __device__ __forceinline__ float getq(float a) { return a; }
template <int Q> __device__ __forceinline__ double getq(double a) { return a; }
__device__ __forceinline__ f2 mkv(float a, float b, f2*) { return f2(a, b); }
__device__ __forceinline__ float mkv(float a, float, float*) { return a; }
__device__ __forceinline__ double mkv(double a, double, double*) { return a; }

// per-spin prologue shared by forward and backward: constants of one spin, in scalar T
template <typename T, int NC, bool RELAX>
__device__ __forceinline__ void load_spin(const KArgs<T>& a, int n, int i, T lx, T ly, T lz, SpinConst<T, NC>& k) {
  T br[NC], bi[NC];
  if (a.b1) {
    const T* bp = a.b1 + (int64_t)n * a.b1_sn + (int64_t)i * a.b1_sm;
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      br[c] = c < a.nC ? bp[c] : (T)0;
      bi[c] = c < a.nC ? bp[a.nC + c] : (T)0;
    }
  }
  const double gam = ld_param(a.gamma, n, i);
  const double dt = ld_param(a.dt, n, 0);
  const double df = a.df.ptr ? ld_param(a.df, n, i) : 0.0;
  const double t1 = RELAX ? ld_param(a.T1, n, i) : 1.0;
  const double t2 = RELAX ? ld_param(a.T2, n, i) : 1.0;
  make_consts<T, NC>(k, gam, dt, RELAX, t1, t2, df, lx, ly, lz, a.b1 ? br : nullptr, a.b1 ? bi : nullptr);
}
template <typename T, typename V, int NC, int PK, bool RELAX>
__device__ __forceinline__ void load_consts_v(const KArgs<T>& a, int n, const int (&idx)[PK], V lx, V ly, V lz,
                                              SpinConst<V, NC>& k) {
  if constexpr (PK == 1) {
    load_spin<T, NC, RELAX>(a, n, idx[0], lx, ly, lz, k);
  } else {
    SpinConst<float, NC> k0, k1;
    load_spin<float, NC, RELAX>(a, n, idx[0], getq<0>(lx), getq<0>(ly), getq<0>(lz), k0);
    load_spin<float, NC, RELAX>(a, n, idx[1], getq<1>(lx), getq<1>(ly), getq<1>(lz), k1);
    k = pack2<NC>(k0, k1);
  }
}
// three consecutive T's of PK spins -> three V's
template <typename T, typename V, int PK>
__device__ __forceinline__ void load_vec3(const T* base, int64_t stride, const int (&idx)[PK], V& x, V& y, V& z) {
  const T* p0 = base + (int64_t)idx[0] * stride;
  const T* p1 = base + (int64_t)idx[PK - 1] * stride;
  x = mkv(p0[0], p1[0], (V*)nullptr);
  y = mkv(p0[1], p1[1], (V*)nullptr);
  z = mkv(p0[2], p1[2], (V*)nullptr);
}

// Per-spin 3-vectors (Mi, Mo, dL/dMo, loc) of a whole tile are one contiguous run of 12*TILE bytes when the spin stride
// is 3 elements: the CTA reads it ONCE with coalesced 128-bit loads into `scr`, then every thread picks its spins.
// Ragged last tiles, foreign strides and unaligned bases take the direct (L1-coalesced) path.  CTA-uniform branch.
template <typename T, typename V, int PK, int BLKT>
__device__ __forceinline__ void load_vec3_tile(const T* base, int64_t stride, int tile, int nM, const int (&idx)[PK],
                                               T* scr, V& x, V& y, V& z) {
  constexpr int TILE = BLKT * PK;
  const T* src = base + (int64_t)tile * TILE * 3;
  const bool coop = stride == 3 && (tile + 1) * TILE <= nM && (reinterpret_cast<uintptr_t>(src) & 15) == 0;
  if (coop) {
    constexpr int NVEC = TILE * 3 * (int)sizeof(T) / 16;
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* d4 = reinterpret_cast<float4*>(scr);
    for (int q = threadIdx.x; q < NVEC; q += BLKT) d4[q] = s4[q];
    __syncthreads();
    const int l0 = threadIdx.x, l1 = (PK - 1) * BLKT + threadIdx.x;
    x = mkv(scr[3 * l0], scr[3 * l1], (V*)nullptr);
    y = mkv(scr[3 * l0 + 1], scr[3 * l1 + 1], (V*)nullptr);
    z = mkv(scr[3 * l0 + 2], scr[3 * l1 + 2], (V*)nullptr);
    __syncthreads();
  } else {
    load_vec3<T, V, PK>(base, stride, idx, x, y, z);
  }
}

// REC forward: state r (lab frame) of PK spins -> Mt[n][r][xyz][spin], streaming stores as the checkpoints; padding
// lanes store nothing
template <typename T, typename V, int PK>
__device__ __forceinline__ void rec_store(const RecOut<T>& o, int nM, int n, int r, const int (&idx)[PK], const bool (&ok)[PK],
                                          V x, V y, V z) {
  T* p = o.Mt + ((size_t)n * o.nR + r) * 3 * (size_t)nM;
  if (ok[0]) {
    __stcs(p + idx[0], getq<0>(x));
    __stcs(p + (size_t)nM + idx[0], getq<0>(y));
    __stcs(p + 2 * (size_t)nM + idx[0], getq<0>(z));
  }
  if (PK == 2 && ok[PK - 1]) {
    __stcs(p + idx[PK - 1], getq<1>(x));
    __stcs(p + (size_t)nM + idx[PK - 1], getq<1>(y));
    __stcs(p + 2 * (size_t)nM + idx[PK - 1], getq<1>(z));
  }
}
// REC backward: dL/dMt[r] of PK spins, turned into the spin frame; zero in padding lanes (their idx is a real spin)
template <typename T, typename V, int NC, int PK>
__device__ __forceinline__ void rec_load(const RecOut<T>& o, int nM, int n, int r, const int (&idx)[PK], const bool (&ok)[PK],
                                         const SpinConst<V, NC>& k, V& x, V& y, V& z) {
  const T* p = o.gMt + ((size_t)n * o.nR + r) * 3 * (size_t)nM;
  T v[PK][3];
#pragma unroll
  for (int q = 0; q < PK; ++q) {
#pragma unroll
    for (int e = 0; e < 3; ++e) v[q][e] = ok[q] ? __ldcs(p + e * (size_t)nM + idx[q]) : (T)0;
  }
  x = mkv(v[0][0], v[PK - 1][0], (V*)nullptr);
  y = mkv(v[0][1], v[PK - 1][1], (V*)nullptr);
  z = mkv(v[0][2], v[PK - 1][2], (V*)nullptr);
  to_frame(k, x, y);
}

// RD: the receive weights of this thread's PK spins, w[c] + i w[nRx + c] = c_k e^{i arg b1} (the state is kept in the spin's own
// frame, single coil: folding the turn into the weight once per spin spares turning the state at every record; elsewhere
// fc = 1, fs = 0).  Zero in padding lanes.  Each thread reads back only its own entries: no barrier.
template <typename T, typename V, int NC, int PK, int BLKT>
__device__ __forceinline__ void ro_weights(const RoOut<T>& ro, int n, const int (&idx)[PK], const bool (&ok)[PK],
                                           const SpinConst<V, NC>& k, V* w) {
  const int nRx = ro.nRx;
  for (int c = 0; c < nRx; ++c) {
    T wr[PK], wi[PK];
#pragma unroll
    for (int q = 0; q < PK; ++q) {
      T cr = ok[q] ? (T)1 : (T)0, ci = (T)0;
      if (ro.rx && ok[q]) {
        const T* p = ro.rx + (int64_t)n * ro.rx_sn + (int64_t)idx[q] * ro.rx_sm;
        cr = p[c];
        ci = p[nRx + c];
      }
      const T fc = q == 0 ? getq<0>(k.fc) : getq<1>(k.fc), fs = q == 0 ? getq<0>(k.fs) : getq<1>(k.fs);
      wr[q] = fnma_(fs, ci, fc * cr);
      wi[q] = fma_(fs, cr, fc * ci);
    }
    w[c * BLKT + threadIdx.x] = mkv(wr[0], wr[PK - 1], (V*)nullptr);
    w[(nRx + c) * BLKT + threadIdx.x] = mkv(wi[0], wi[PK - 1], (V*)nullptr);
  }
}
// RD forward, at a recorded state: this thread's weighted (Sx, Sy) per receive coil (its PK spins added first) into the columns
// slot * 2 nRx + (c | nRx + c) of its warp's tile
template <typename T, typename V, int BLKT>
__device__ __forceinline__ void ro_accum(const RoOut<T>& ro, const V* w, T* tile, int slot, V mx, V my) {
  const int nRx = ro.nRx, lane = threadIdx.x & 31;
  T* col = tile + (size_t)slot * 2 * nRx * 32 + lane;
  for (int c = 0; c < nRx; ++c) {
    const V wr = w[c * BLKT + threadIdx.x], wi = w[(nRx + c) * BLKT + threadIdx.x];
    col[c * 32] = hsum(fnma_(wi, my, wr * mx));
    col[(nRx + c) * 32] = hsum(fma_(wi, mx, wr * my));
  }
}
// RD forward: the CTA sums the nb buffered records r0 .. r0 + nb - 1 of its tiles into its slot, in the manner of
// warp_tile_reduce: lane l of each warp adds up column l (rotated start: conflict-free), the warps meet in a fixed order
// through the double-buffered ctab, and thread j owns value j of the slot -- stores on the CTA's first tile, adds on later
// ones.  One writer per value, no atomics: bitwise reproducible.  Every thread of the CTA must call it (one barrier).
// nb = the buffered records (bits 0-15) | the parity of ctab (bit 16); it leaves with no records and the other parity.
template <typename T, int BLKT>
__device__ __forceinline__ void ro_flush(const RoOut<T>& ro, const T* tiles, T* ctab, int n, int rr, int& nb, bool first) {
  constexpr int NW = BLKT / 32;
  const int cnt = nb & 0xffff, par = nb >> 16, r0 = rr - cnt;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, ncol = cnt * 2 * ro.nRx;
  __syncwarp();
  const T* t = tiles + (size_t)warp * RO_COLS * 32 + (size_t)lane * 32;
  T sum = (T)0;
  if (lane < ncol) {
#pragma unroll 8
    for (int q = 0; q < 32; ++q) sum += t[(q + lane) & 31];
  }
  T* cb = ctab + (size_t)par * NW * 32;
  cb[warp * 32 + lane] = sum;
  __syncthreads();
  if (tid < ncol) {
    T s = cb[tid];
#pragma unroll
    for (int q = 1; q < NW; ++q) s += cb[q * 32 + tid];
    T* dst = ro.part + (((size_t)n * gridDim.x + blockIdx.x) * ro.nR + r0) * 2 * ro.nRx + tid;
    *dst = first ? s : *dst + s;
  }
  nb = (par ^ 1) << 16;
}
// RD backward, at the step that produced record r: h += the adjoint of S[r] (gs = dL/dS[n, :, r, :], staged), and with grx the
// per-spin sums acc += conj(m) dL/dS[r] (in the spin frame; ro_grx_store turns them to the lab frame)
template <typename T, typename V, int BLKT>
__device__ __forceinline__ void ro_adjoint(const RoOut<T>& ro, const V* w, V* acc, const T* gs, V mx, V my, V& hx, V& hy) {
  const int nRx = ro.nRx, tid = threadIdx.x;
  for (int c = 0; c < nRx; ++c) {
    const V gx = V(gs[c]), gy = V(gs[nRx + c]);
    const V wr = w[c * BLKT + tid], wi = w[(nRx + c) * BLKT + tid];
    hx = fma_(wr, gx, fma_(wi, gy, hx));
    hy = fma_(wr, gy, fnma_(wi, gx, hy));
    if (ro.grx) {
      acc[c * BLKT + tid] = fma_(mx, gx, fma_(my, gy, acc[c * BLKT + tid]));
      acc[(nRx + c) * BLKT + tid] = fma_(mx, gy, fnma_(my, gx, acc[(nRx + c) * BLKT + tid]));
    }
  }
}
// RD backward, end of a tile: dL/drx = e^{-i arg b1} acc of the thread's spins (dL/dc = sum_r conj(m_lab) dL/dS[r])
template <typename T, typename V, int NC, int PK, int BLKT>
__device__ __forceinline__ void ro_grx_store(const RoOut<T>& ro, int n, int nM, const int (&idx)[PK], const bool (&ok)[PK],
                                             const SpinConst<V, NC>& k, const V* acc) {
  const int nRx = ro.nRx;
#pragma unroll
  for (int q = 0; q < PK; ++q) {
    if (!ok[q]) continue;
    const T fc = q == 0 ? getq<0>(k.fc) : getq<1>(k.fc), fs = q == 0 ? getq<0>(k.fs) : getq<1>(k.fs);
    T* o = ro.grx + ((size_t)n * nM + idx[q]) * 2 * nRx;
    for (int c = 0; c < nRx; ++c) {
      const V ax = acc[c * BLKT + threadIdx.x], ay = acc[(nRx + c) * BLKT + threadIdx.x];
      const T x = q == 0 ? getq<0>(ax) : getq<1>(ax), y = q == 0 ? getq<0>(ay) : getq<1>(ay);
      o[c] = fma_(fs, y, fc * x);
      o[nRx + c] = fnma_(fs, x, fc * y);
    }
  }
}

// ------------------------------------------------------------------------------------------
// pack: one thread per element of wave[N][nChunks][W][TCP]
template <typename T>
__global__ void pack_waveform_kernel(const T* __restrict__ rf, int64_t rf_sn, int64_t rf_sx, int64_t rf_st, int64_t rf_sc,
                                     const T* __restrict__ gr, int64_t gr_sn, int64_t gr_sx, int64_t gr_st, int nC,
                                     int NC, int sum_coils, int nT, int K, int TCP, int nChunks, int WS, int stepmajor,
                                     int64_t total, T* __restrict__ wave) {
  const int W = 2 * NC + 3;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    // row-major chunk [WS = W][TCP]  |  step-major chunk [TCP][WS]
    const int j = stepmajor ? (int)((e / WS) % TCP) : (int)(e % TCP);
    const int w = stepmajor ? (int)(e % WS) : (int)((e / TCP) % WS);
    const int c = (int)((e / ((int64_t)TCP * WS)) % nChunks);
    const int n = (int)(e / ((int64_t)TCP * WS * nChunks));
    const int t = c * K + j;
    T v = (T)0;
    if (j < K && t < nT && w < W) {
      if (w < 2 * NC) {
        const int x = w / NC, coil = w % NC;
        const T* p = rf + n * rf_sn + x * rf_sx + t * rf_st;
        if (sum_coils) {   // no b1Map: beffective.py:147-151 sums rf over coils
          for (int q = 0; q < nC; ++q) v += p[q * rf_sc];
        } else if (coil < nC) {
          v = p[coil * rf_sc];
        }
      } else {
        v = gr[n * gr_sn + (w - 2 * NC) * gr_sx + t * gr_st];
      }
    }
    wave[e] = v;
  }
}

// ------------------------------------------------------------------------------------------
// forward.  PK spins per thread (PK == 2: packed f2 arithmetic), BLKT threads per CTA.
// REC: also the state after every `rec.every` steps (rec_store), tracked by a countdown (no per-step division).
// RD: instead the signal of the state after every `ro.every` steps, on the same countdown (ro_accum / ro_flush).
template <typename T, int POL, bool RELAX, int NC, int PK, int BLKT, int OPT = OPT_NONE>
__global__ void __launch_bounds__(BLKT, (PK == 2 ? (NC == 1 ? 14 : MRPHY_NC2_MINB) : 1)) fused_fwd_kernel(const KArgs<T> a, const RecOut<T> rec) {
  constexpr bool REC = OPT == OPT_RECORD, RD = OPT == OPT_READOUT;
  const RoOut<T>& ro = rec.ro;
  typedef typename Pack<T, PK>::type V;
  constexpr int W = 2 * NC + 3;
  constexpr int WS = WaveLayout<T, W>::WS;
  __shared__ __align__(128) T wbuf[2][WS * ChunkMax<T, NC>::v];
  __shared__ __align__(16) T scr[3 * BLKT * PK];
  __shared__ __align__(8) uint64_t full[2];
  extern __shared__ __align__(16) unsigned char ro_smem[];   // RD (see RoOut); addresses formed where used: no live registers
#define RO_W reinterpret_cast<V*>(ro_smem)
#define RO_TILES reinterpret_cast<T*>(ro_smem + (size_t)2 * ro.nRx * BLKT * sizeof(V))
#define RO_CTAB (RO_TILES + (BLKT / 32) * RO_COLS * 32)
  int nb = 0;   // RD: records buffered since the last flush | ctab parity (ro_flush)
  const int tid = threadIdx.x, n = blockIdx.y;
  const int TCP = a.TCP, K = a.K, nT = a.nT, nChunks = a.nChunks, nM = a.nM;
  const uint32_t chunk_bytes = (uint32_t)(WS * TCP * sizeof(T));
  const T* wave_n = a.wave + (size_t)n * nChunks * WS * TCP;
  const int tiles = (nM + BLKT * PK - 1) / (BLKT * PK);
  const int my_tiles = ((int)blockIdx.x < tiles) ? (tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const uint32_t total = (uint32_t)my_tiles * (uint32_t)nChunks;
  if (tid == 0) {
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    fence_barrier_init();
  }
  __syncthreads();
  if (tid == 0 && total > 0) {
    mbar_arrive_expect_tx(&full[0], chunk_bytes);
    bulk_g2s(wbuf[0], wave_n, chunk_bytes, &full[0]);
  }
  uint32_t it = 0;
  for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    SpinConst<V, NC> k;
    V mx, my, mz;
    int idx[PK];
    bool ok[PK];
#pragma unroll
    for (int q = 0; q < PK; ++q) {
      const int i = (tile * PK + q) * BLKT + tid;
      ok[q] = i < nM;
      idx[q] = ok[q] ? i : nM - 1;
    }
    {
      V lx, ly, lz;
      load_vec3_tile<T, V, PK, BLKT>(a.loc + (int64_t)n * a.loc_sn, a.loc_sm, tile, nM, idx, scr, lx, ly, lz);
      load_consts_v<T, V, NC, PK, RELAX>(a, n, idx, lx, ly, lz, k);
    }
    load_vec3_tile<T, V, PK, BLKT>(a.Mi + (int64_t)n * a.Mi_sn, a.Mi_sm, tile, nM, idx, scr, mx, my, mz);
    to_frame(k, mx, my);   // single coil: the spin's own transverse frame (bloch_math.cuh: make_consts); checkpoints stay in it
    int rc = RD ? ro.every : rec.every, rr = 0;   // REC, RD: steps to the next recorded state, its index
    if constexpr (RD) ro_weights<T, V, NC, PK, BLKT>(ro, n, idx, ok, k, RO_W);
    for (int c = 0; c < nChunks; ++c, ++it) {
      if (tid == 0 && it + 1 < total) {   // prefetch the next chunk (possibly chunk 0 of the next tile)
        const int cn = (c + 1 == nChunks) ? 0 : c + 1;
        const uint32_t sn = (it + 1) & 1;
        mbar_arrive_expect_tx(&full[sn], chunk_bytes);
        bulk_g2s(wbuf[sn], wave_n + (size_t)cn * WS * TCP, chunk_bytes, &full[sn]);
      }
      mbar_wait(&full[it & 1], (it >> 1) & 1);
      const T* wb = wbuf[it & 1];
      const int ns = min(K, nT - c * K);
      auto one_step = [&](const T (&s)[W]) {
        V rx[NC], ry[NC], bx, by, bz;
#pragma unroll
        for (int q = 0; q < NC; ++q) { rx[q] = V(s[q]); ry[q] = V(s[NC + q]); }
        field<V, NC>(k, rx, ry, V(s[2 * NC]), V(s[2 * NC + 1]), V(s[2 * NC + 2]), bx, by, bz);
        step_fwd<V, POL, RELAX>(bx, by, bz, k.e1, k.e2, mx, my, mz);
        if constexpr (REC) {
          if (--rc == 0) {   // recorded states leave the spin frame (a copy: the state stays in it)
            V x = mx, y = my;
            from_frame(k, x, y);
            rec_store<T, V, PK>(rec, nM, n, rr++, idx, ok, x, y, mz);
            rc = rec.every;
          }
        }
        if constexpr (RD) {
          if (--rc == 0) {   // (CTA-uniform: every thread steps the same count)
            ro_accum<T, V, BLKT>(ro, RO_W, RO_TILES + (size_t)(tid >> 5) * RO_COLS * 32, nb & 0xffff, mx, my);
            ++rr;
            if ((++nb & 0xffff) == ro.rt || rr == ro.nR) ro_flush<T, BLKT>(ro, RO_TILES, RO_CTAB, n, rr, nb, tile == (int)blockIdx.x);
            rc = ro.every;
          }
        }
      };
      int j = 0;
      // 4 steps per iteration with 128-bit broadcast loads, while the staged samples fit ~40 registers
      constexpr bool VEC4 = !WaveLayout<T, W>::STEPMAJOR;
      for (; VEC4 && j + 4 <= ns; j += 4) {
        T wv[W][4];
#pragma unroll
        for (int w = 0; w < W; ++w) load4(wb + w * TCP + j, wv[w]);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          T s[W];
#pragma unroll
          for (int w = 0; w < W; ++w) s[w] = wv[w][u];
          one_step(s);
        }
      }
      for (; j < ns; ++j) {
        T s[W];
        load_step<T, W>(wb, TCP, j, s);
        one_step(s);
      }
      if (c + 1 < nChunks) {   // checkpoint: state after (c+1)*K steps
        T* cp = a.ckpt + ((size_t)n * (nChunks - 1) + c) * 3 * (size_t)nM;
        // streaming (evict-first) stores and, in the backward, loads: 12.7 GB of checkpoints at C5 pass through the 126-MB L2
        // exactly once and must not push the L2-resident partial sums out (ncu: 1.8 GB of write-backs per launch otherwise)
        if (ok[0]) {
          __stcs(cp + idx[0], getq<0>(mx));
          __stcs(cp + (size_t)nM + idx[0], getq<0>(my));
          __stcs(cp + 2 * (size_t)nM + idx[0], getq<0>(mz));
        }
        if (PK == 2 && ok[PK - 1]) {
          __stcs(cp + idx[PK - 1], getq<1>(mx));
          __stcs(cp + (size_t)nM + idx[PK - 1], getq<1>(my));
          __stcs(cp + 2 * (size_t)nM + idx[PK - 1], getq<1>(mz));
        }
      }
      __syncthreads();   // everyone is done with wbuf[it&1] before it is refilled
    }
    from_frame(k, mx, my);
#undef RO_W
#undef RO_TILES
#undef RO_CTAB
    if (ok[0]) {
      T* op = a.Mo + ((size_t)n * nM + idx[0]) * 3;
      op[0] = getq<0>(mx); op[1] = getq<0>(my); op[2] = getq<0>(mz);
    }
    if (PK == 2 && ok[PK - 1]) {
      T* op = a.Mo + ((size_t)n * nM + idx[PK - 1]) * 3;
      op[0] = getq<1>(mx); op[1] = getq<1>(my); op[2] = getq<1>(mz);
    }
  }
}

// S[n][xy][r][k] = sum over the P slots of part[n][p][r][xy * nRx + k] in slot order (bitwise reproducible).  Block (32, 8):
// 32 consecutive values of a batch entry's slot, the 8 rows take every 8th slot, then meet in a fixed order.
template <typename T>
__global__ void readout_finalize_kernel(const T* __restrict__ part, int P, int nR, int nRx, T* __restrict__ S) {
  __shared__ T red[8][32];
  const int n = blockIdx.y, cols = nR * 2 * nRx, col = blockIdx.x * 32 + threadIdx.x;
  T s = (T)0;
  if (col < cols)
    for (int p = threadIdx.y; p < P; p += 8) s += part[((size_t)n * P + p) * cols + col];
  red[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && col < cols) {
#pragma unroll
    for (int q = 1; q < 8; ++q) s += red[q][threadIdx.x];
    const int r = col / (2 * nRx), j = col % (2 * nRx), xy = j / nRx, kk = j % nRx;
    S[(((size_t)n * 2 + xy) * nR + r) * nRx + kk] = s;
  }
}

// Column sums of one warp's transposition tile red[W][TR][32]: every lane owns one row r and adds up the TR source
// lanes of its group, then the 32/TR groups meet through shuffles; one lane per row publishes out[w][r].
// fp32, TR == 16: lane l takes row l/2 and the half (l&1) of its 32 source lanes with four 128-bit loads whose
// chunk order is rotated by the row -- the 8 lanes of a quarter-warp then touch 8 distinct 16-byte bank groups
// (conflict-free).  Otherwise scalar loads with a rotated start (conflict-free).
template <typename T, int W, int TR, int W0 = 0, int W1 = W>
__device__ __forceinline__ void warp_tile_reduce(const T (*tile)[TR][32], int lane, T (*out)[TR]) {
  if constexpr (sizeof(T) == 4 && TR == 16) {
    const int r = lane >> 1, half = (lane & 1) << 4;
#pragma unroll
    for (int w = W0; w < W1; ++w) {
      const float4* row = reinterpret_cast<const float4*>(&tile[w][r][half]);
      T sum = (T)0;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 v = row[(q + r) & 3];
        sum += (v.x + v.y) + (v.z + v.w);
      }
      sum += __shfl_xor_sync(0xffffffffu, sum, 1);
      if (!(lane & 1)) out[w][r] = sum;
    }
  } else {
    const int r = lane & (TR - 1), grp = lane & ~(TR - 1);
#pragma unroll
    for (int w = W0; w < W1; ++w) {
      T sum = (T)0;
#pragma unroll
      for (int q = 0; q < TR; ++q) sum += tile[w][r][grp + ((q + lane) & (TR - 1))];
#pragma unroll
      for (int o = TR; o < 32; o <<= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      if (lane < TR) out[w][r] = sum;
    }
  }
}

// Multi-coil column sums: `ft` is the warp's F tile [32 spins][P16 x 16 B] (entry r of spin s = Fx, Fy, Fz, pad of step r),
// `wt` the per-spin weights [32][WP] = (g Re b1_c)_c, (g Im b1_c)_c, g loc.  Lane l owns step r = l % TR and the spins
// [grp*SP, (grp+1)*SP), grp = l / TR: per spin one 128-bit load of F (consecutive lanes = consecutive entries), broadcast
// 128-bit loads of the weights, 4 NC + 3 FMAs into W register accumulators; the 32/TR groups meet through shuffles.
// No second pass over shared memory, no per-step chain rule in the time loop.
template <typename T, int NC, int TR, int W0, int W1>
__device__ __forceinline__ void warp_tile_reduce_weighted(const unsigned char* ft, const T* wt, int lane, T (*out)[TR]) {
  constexpr int W = 2 * NC + 3, WP = (W + 3) & ~3, E16 = (int)sizeof(T) / 4, P16 = TR * E16 + 1, SP = TR;   // 32 / (32 / TR)
  constexpr bool WANT_RF = W0 == 0, WANT_GR = W1 == W;
  const int r = lane % TR, grp = lane / TR;
  T acc[W];
#pragma unroll
  for (int w = 0; w < W; ++w) acc[w] = (T)0;
#pragma unroll 2
  for (int q = 0; q < SP; ++q) {
    const int sp = grp * SP + q;
    T f[4];
    {
      const float4* src = reinterpret_cast<const float4*>(ft + ((size_t)sp * P16 + (size_t)r * E16) * 16);
      float4* dst = reinterpret_cast<float4*>(f);
#pragma unroll
      for (int e = 0; e < E16; ++e) dst[e] = src[e];
    }
    T wv[WP];
    {
      const float4* src = reinterpret_cast<const float4*>(wt + (size_t)sp * WP);
      float4* dst = reinterpret_cast<float4*>(wv);
#pragma unroll
      for (int e = 0; e < WP * (int)sizeof(T) / 16; ++e) dst[e] = src[e];
    }
    if constexpr (WANT_RF) {
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        acc[c] = fma_(wv[c], f[0], fma_(wv[NC + c], f[1], acc[c]));
        acc[NC + c] = fma_(wv[c], f[1], fnma_(wv[NC + c], f[0], acc[NC + c]));
      }
    }
    if constexpr (WANT_GR) {
      acc[2 * NC] = fma_(wv[2 * NC], f[2], acc[2 * NC]);
      acc[2 * NC + 1] = fma_(wv[2 * NC + 1], f[2], acc[2 * NC + 1]);
      acc[2 * NC + 2] = fma_(wv[2 * NC + 2], f[2], acc[2 * NC + 2]);
    }
  }
#pragma unroll
  for (int w = W0; w < W1; ++w) {
    T sum = acc[w];
#pragma unroll
    for (int o = TR; o < 32; o <<= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane < TR) out[w][r] = sum;
  }
}

// Per-spin gradients of the SG backward, in the reference's terms (mrphy_rfgr2beff_spin_grads) with G = dL/dBeff = -g F,
// g = 2 pi gamma dt:  gloc = sum_t gr(t) G_z,  gsz = sum_t G_z,  gb1_c = sum_t conj(rx_c + i ry_c) (G_x + i G_y).
// A thread sums F over the steps of one staged chunk in registers, acc = [sum gr F_z (3) | sum F_z | Re_c (NC) | Im_c (NC)],
// and folds that chunk sum into the outputs at the chunk's end -- a two-level sum over time that adds nothing per step.  The
// outputs belong to the thread that owns the spin: a plain read-modify-write.  The chunk processed first (time runs
// backwards) stores; the last one (c == 0) also scales by -g and, single coil, turns the frame sums back to the lab frame
// (the spin's own frame is the lab frame turned by arg b1: G_lab = e^{i arg b1} G_frame, bloch_math.cuh: make_consts).
template <typename T, typename V, int NC, int PK>
__device__ __forceinline__ void sg_fold(const KArgs<T>& a, const SgOut<T>& o, int n, const int (&idx)[PK], const bool (&ok)[PK], bool first,
                                        bool last, const SpinConst<V, NC>& k, const V (&acc)[4 + 2 * NC]) {
  constexpr int NA = 4 + 2 * NC;
#pragma unroll
  for (int q = 0; q < PK; ++q) {
    if (!ok[q]) continue;
    const size_t s = (size_t)n * a.nM + idx[q];
    T v[NA];
#pragma unroll
    for (int w = 0; w < NA; ++w) v[w] = q == 0 ? getq<0>(acc[w]) : getq<1>(acc[w]);
    T* const pl = o.gloc ? o.gloc + s * 3 : nullptr;
    T* const pz = o.gsz ? o.gsz + s : nullptr;
    T* const pb = o.gb1 ? o.gb1 + s * 2 * a.nC : nullptr;
    if (!first) {
      if (pl) { v[0] += pl[0]; v[1] += pl[1]; v[2] += pl[2]; }
      if (pz) v[3] += pz[0];
      if (pb) {
#pragma unroll
        for (int c = 0; c < NC; ++c)
          if (c < a.nC) { v[4 + c] += pb[c]; v[4 + NC + c] += pb[a.nC + c]; }
      }
    }
    if (last) {
      const T ng = (T)(-6.283185307179586476925286766559 * ld_param(a.gamma, n, idx[q]) * ld_param(a.dt, n, 0));
#pragma unroll
      for (int w = 0; w < NA; ++w) v[w] *= ng;
      if (NC == 1) {   // frame -> lab: (re + i im) * (fc + i fs)
        const T fc = q == 0 ? getq<0>(k.fc) : getq<1>(k.fc), fs = q == 0 ? getq<0>(k.fs) : getq<1>(k.fs);
        const T re = v[4], im = v[5];
        v[4] = fnma_(fs, im, fc * re);
        v[5] = fma_(fs, re, fc * im);
      }
    }
    if (pl) { pl[0] = v[0]; pl[1] = v[1]; pl[2] = v[2]; }
    if (pz) pz[0] = v[3];
    if (pb) {
#pragma unroll
      for (int c = 0; c < NC; ++c)
        if (c < a.nC) { pb[c] = v[4 + c]; pb[a.nC + c] = v[4 + NC + c]; }
    }
  }
}

// ------------------------------------------------------------------------------------------
// backward
// ROWS: which gradients the caller wants -- bit 0 dL/drf (rows [0, 2 NC)), bit 1 dL/dgr (rows [2 NC, W)); the other rows
// of the spin reduction are neither formed nor reduced (an RF-only design skips 3 of its 5 rows).
// SG: also the per-spin gradients (sg_fold).  ROWS == 0 (SG only, a fixed pulse): no transposition tile, no partial sums.
// REC: the loss also depends on the recorded states: dL/dMt[r] joins the adjoint before the adjoint of the step that
// produced state r, so that everything downstream (F, the spin reduction, sg_fold, dL/dMi) sees the total dL/dm.
// RD: the adjoint of the readout joins instead, at the same steps (ro_adjoint), and with ro.grx the kernel also forms dL/drx.
template <typename T, int POL, bool RELAX, int NC, int PK, int BLKT, int ROWS = 3, bool SG = false, int OPT = OPT_NONE>
__global__ void __launch_bounds__(BLKT, (PK == 2 ? MRPHY_BWD_MINB * 64 / BLKT : (sizeof(T) == 8 && NC == 1 ? 4 : (sizeof(T) == 4 && NC > 1 ? MRPHY_MC_MINB : 1)))) fused_bwd_kernel(const KArgs<T> a, const int need_gmi, const SgOut<T> sgo, const RecOut<T> rec) {
  constexpr bool REC = OPT == OPT_RECORD, RD = OPT == OPT_READOUT;
  const RoOut<T>& ro = rec.ro;
  typedef typename Pack<T, PK>::type V;
  using L = BwdSmem<T, NC, BLKT, PK>;
  constexpr int W = L::W, TR = L::TR, NW = L::NW;
  constexpr bool WANT_RF = (ROWS & 1) != 0, WANT_GR = (ROWS & 2) != 0;
  constexpr int W0 = WANT_RF ? 0 : 2 * NC, W1 = WANT_GR ? W : 2 * NC;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int WS = L::WS;
  T(*wbuf)[WS * L::TCM] = reinterpret_cast<T(*)[WS * L::TCM]>(smem_raw + L::wbuf);
  T(*red)[W][TR][32] = reinterpret_cast<T(*)[W][TR][32]>(smem_raw + L::red);   // per-warp transposition tile (single coil)
  constexpr bool WRED = L::WRED;
  unsigned char* const ft = smem_raw + L::red + (size_t)(threadIdx.x >> 5) * 32 * L::P16 * 16;            // WRED: this warp's F tile
  T* const wt = reinterpret_cast<T*>(smem_raw + L::red + (size_t)NW * 32 * L::P16 * 16) + (size_t)(threadIdx.x >> 5) * 32 * L::WP;
  T(*cta)[W][TR] = reinterpret_cast<T(*)[W][TR]>(smem_raw + L::cta);          // per-warp tile sums
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + L::bar);
  // RD (see RoOut): the weights, the dL/drx sums and the staged dL/dS behind the kernel's own shared memory
#define RO_W reinterpret_cast<V*>(smem_raw + L::bytes)
#define RO_ACC (RO_W + (size_t)2 * ro.nRx * BLKT)
#define RO_GS reinterpret_cast<T*>(RO_ACC + (size_t)2 * ro.nRx * BLKT)
  __shared__ __align__(16) T scr[3 * BLKT * PK];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, n = blockIdx.y;
  const int TCP = a.TCP, K = a.K, nT = a.nT, nChunks = a.nChunks, nM = a.nM;
  const uint32_t chunk_bytes = (uint32_t)(WS * TCP * sizeof(T));
  const T* wave_n = a.wave + (size_t)n * nChunks * WS * TCP;
  const int tiles = (nM + BLKT * PK - 1) / (BLKT * PK);
#define NCTA ((int)gridDim.x)   /* constant-bank operand, not a register */
  __shared__ int s_vid, s_sweep;
  if (tid == 0) {
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    fence_barrier_init();
  }
  if (a.done && blockIdx.x == 0 && tid == 0) a.done[n] = 0;   // for the epilogue that follows in stream order
  // which virtual id does this CTA serve first (see SCHED_*)
  int vid = blockIdx.x;
  if (a.sched && tid == 0) {
    int* const sched = a.sched;
    s_sweep = 0;
    const int s = (int)my_smid();
    int v0 = -1;
    if (s < a.n_sm && s < SCHED_SM_SLOTS) {
      const int rank = atomicAdd(&sched[s], 1);
      const int cand = rank * a.n_sm + s;
      if (rank < a.c_per_sm && cand < NCTA && atomicCAS(&sched[SCHED_CLAIM + cand], 0, 1) == 0) {
        v0 = cand;
        atomicAdd(&sched[SCHED_NCLAIMED], 1);
      }
    }
    s_vid = v0;
  }
  __syncthreads();
  if (a.sched) vid = s_vid;
#ifdef MRPHY_CTA_TRACE
  if (tid == 0 && blockIdx.x < 8192 && n == 0) { g_cta_trace[blockIdx.x][0] = smid(); g_cta_trace[blockIdx.x][1] = gtime(); g_cta_trace[blockIdx.x][3] = (unsigned long long)(long long)vid; }
#endif
  uint32_t it = 0, red_par = 0;
  for (;;) {
   if (vid >= 0) {
    const int my_tiles = (vid < tiles) ? (tiles - vid + NCTA - 1) / NCTA : 0;
    const uint32_t total = it + (uint32_t)my_tiles * (uint32_t)nChunks;   // `it` once this id's last chunk is consumed
    T* part = a.partials + ((size_t)n * a.P + vid) * W * (size_t)nT;
    if (my_tiles == 0) {   // an id without work still owns a partial slot: zero it
      if constexpr (ROWS != 0)
        for (int e = tid; e < W * nT; e += BLKT) part[e] = (T)0;
    } else if (tid == 0) {
      mbar_arrive_expect_tx(&full[it & 1], chunk_bytes);
      bulk_g2s(wbuf[it & 1], wave_n + (size_t)(nChunks - 1) * WS * TCP, chunk_bytes, &full[it & 1]);
    }
  bool first = true;
  for (int tile = vid; tile < tiles; tile += NCTA, first = false) {
    SpinConst<V, NC> k;
    V mx, my, mz, hx, hy, hz;
    int idx[PK];
    bool ok[PK];
#pragma unroll
    for (int q = 0; q < PK; ++q) {
      const int i = (tile * PK + q) * BLKT + tid;
      ok[q] = i < nM;
      idx[q] = ok[q] ? i : nM - 1;
    }
    {
      V lx, ly, lz;
      load_vec3_tile<T, V, PK, BLKT>(a.loc + (int64_t)n * a.loc_sn, a.loc_sm, tile, nM, idx, scr, lx, ly, lz);
      load_consts_v<T, V, NC, PK, RELAX>(a, n, idx, lx, ly, lz, k);
    }
    load_vec3_tile<T, V, PK, BLKT>(a.Mo + (size_t)n * nM * 3, 3, tile, nM, idx, scr, mx, my, mz);
    load_vec3_tile<T, V, PK, BLKT>(a.gMo + (int64_t)n * a.gMo_sn, a.gMo_sm, tile, nM, idx, scr, hx, hy, hz);
    to_frame(k, mx, my);   // Mo and dL/dMo enter the spin's transverse frame, dL/dMi leaves it (single coil)
    to_frame(k, hx, hy);
    if constexpr (WRED && ROWS != 0) {   // this spin's weights for the reduce phase (the previous tile's last reduce ended with a CTA barrier)
      T* wrow = wt + (size_t)lane * L::WP;
#pragma unroll
      for (int q = 0; q < NC; ++q) { wrow[q] = lane0(k.cbr[q]); wrow[NC + q] = lane0(k.cbi[q]); }
      wrow[2 * NC] = lane0(k.glx); wrow[2 * NC + 1] = lane0(k.gly); wrow[2 * NC + 2] = lane0(k.glz);
#pragma unroll
      for (int q = W; q < L::WP; ++q) wrow[q] = (T)0;
      __syncwarp();
    }
    {   // padding lanes carry a zero adjoint: they add nothing to the spin sums
      const T z0 = ok[0] ? (T)1 : (T)0, z1 = ok[PK - 1] ? (T)1 : (T)0;
      const V zm = mkv(z0, z1, (V*)nullptr);
      hx = hx * zm; hy = hy * zm; hz = hz * zm;
    }
    // REC: steps (backwards from the end) before the last recorded state, its index, and its dL/dMt loaded one record ahead
    int rc = 0, rr = 0;
    V gx, gy, gz;
    if constexpr (REC) {
      rc = nT - rec.nR * rec.every;
      rr = rec.nR - 1;
      rec_load<T, V, NC, PK>(rec, nM, n, rr, idx, ok, k, gx, gy, gz);
    }
    if constexpr (RD) {
      rc = nT - ro.nR * ro.every;
      rr = ro.nR - 1;
      ro_weights<T, V, NC, PK, BLKT>(ro, n, idx, ok, k, RO_W);
      if (ro.grx)
        for (int c = 0; c < 2 * ro.nRx; ++c) RO_ACC[c * BLKT + tid] = V(0.0f);
    }
    for (int c = nChunks - 1; c >= 0; --c, ++it) {
      [[maybe_unused]] int ro_lo;   // RD: the first record this chunk produced; dL/dS of its records staged in RO_GS
      if constexpr (RD) {
        const int t0 = c * K, t1 = t0 + min(K, nT - c * K);   // records r with (r+1) * every - 1 in [t0, t1)
        ro_lo = (t0 + ro.every) / ro.every - 1;
        const int hi = min(ro.nR, t1 / ro.every), cols = 2 * ro.nRx;
        for (int e = tid; e < (hi - ro_lo) * cols; e += BLKT) {
          const int j = e / cols, v = e % cols;
          RO_GS[e] = ro.gS[(((size_t)n * 2 + v / ro.nRx) * ro.nR + ro_lo + j) * ro.nRx + v % ro.nRx];
        }
        __syncthreads();   // (the previous chunk's last reads of RO_GS precede its last barrier)
      }
      if (tid == 0 && it + 1 < total) {
        const int cn = (c == 0) ? nChunks - 1 : c - 1;
        const uint32_t sn = (it + 1) & 1;
        mbar_arrive_expect_tx(&full[sn], chunk_bytes);
        bulk_g2s(wbuf[sn], wave_n + (size_t)cn * WS * TCP, chunk_bytes, &full[sn]);
      }
      // prefetch the checkpoint this chunk ends on (state after c*K steps) while we compute
      V kx = mx, ky = my, kz = mz;
      if (c > 0) {
        const T* cp = a.ckpt + ((size_t)n * (nChunks - 1) + (c - 1)) * 3 * (size_t)nM;
        kx = mkv(__ldcs(cp + idx[0]), __ldcs(cp + idx[PK - 1]), (V*)nullptr);
        ky = mkv(__ldcs(cp + (size_t)nM + idx[0]), __ldcs(cp + (size_t)nM + idx[PK - 1]), (V*)nullptr);
        kz = mkv(__ldcs(cp + 2 * (size_t)nM + idx[0]), __ldcs(cp + 2 * (size_t)nM + idx[PK - 1]), (V*)nullptr);
      }
      mbar_wait(&full[it & 1], (it >> 1) & 1);
      const T* wb = wbuf[it & 1];
      const int ns = min(K, nT - c * K);
      V sacc[SG ? 4 + 2 * NC : 1];   // SG: this chunk's per-spin sums (sg_fold)
      if constexpr (SG) {
#pragma unroll
        for (int w = 0; w < 4 + 2 * NC; ++w) sacc[w] = V(0.0f);
      }
      // one adjoint step; the W per-thread gradient contributions go to row `row` of the warp's tile
      auto one_step = [&](const T (&s)[W], int row) {
        if constexpr (REC) {
          if (rc == 0) {   // this step produced recorded state rr: h += dL/dMt[rr], then fetch the next one back in time
            hx = hx + gx; hy = hy + gy; hz = hz + gz;
            if (--rr >= 0) rec_load<T, V, NC, PK>(rec, nM, n, rr, idx, ok, k, gx, gy, gz);
            rc = rec.every;
          }
          --rc;
        }
        if constexpr (RD) {
          if (rc == 0) {   // this step produced record rr: h += the adjoint of S[rr]
            ro_adjoint<T, V, BLKT>(ro, RO_W, RO_ACC, RO_GS + (size_t)(rr - ro_lo) * 2 * ro.nRx, mx, my, hx, hy);
            --rr;
            rc = ro.every;
          }
          --rc;
        }
        V rx[NC], ry[NC], bx, by, bz, Fx, Fy, Fz;
#pragma unroll
        for (int q = 0; q < NC; ++q) { rx[q] = V(s[q]); ry[q] = V(s[NC + q]); }
        field<V, NC>(k, rx, ry, V(s[2 * NC]), V(s[2 * NC + 1]), V(s[2 * NC + 2]), bx, by, bz);
        step_bwd<V, POL, RELAX, NC>(k, bx, by, bz, mx, my, mz, hx, hy, hz, Fx, Fy, Fz);
        if constexpr (SG) {
          sacc[0] = fma_(V(s[2 * NC]), Fz, sacc[0]);
          sacc[1] = fma_(V(s[2 * NC + 1]), Fz, sacc[1]);
          sacc[2] = fma_(V(s[2 * NC + 2]), Fz, sacc[2]);
          sacc[3] = sacc[3] + Fz;
#pragma unroll
          for (int q = 0; q < NC; ++q) {
            sacc[4 + q] = fma_(rx[q], Fx, fma_(ry[q], Fy, sacc[4 + q]));
            sacc[4 + NC + q] = fma_(rx[q], Fy, fnma_(ry[q], Fx, sacc[4 + NC + q]));
          }
        }
        if constexpr (ROWS == 0) return;
        if constexpr (WRED) {   // multi-coil: only F goes to the tile; the weights are applied in the reduce phase
          T fv[4] = {lane0(Fx), lane0(Fy), lane0(Fz), (T)0};
          float4* dst = reinterpret_cast<float4*>(ft + ((size_t)lane * L::P16 + (size_t)row * L::E16) * 16);
          const float4* src = reinterpret_cast<const float4*>(fv);
#pragma unroll
          for (int e = 0; e < L::E16; ++e) dst[e] = src[e];
          return;
        }
        if constexpr (WANT_RF) {
#pragma unroll
          for (int q = 0; q < NC; ++q) {
            V gx_, gy_;
            rf_chain<V, NC>(k, q, Fx, Fy, gx_, gy_);
            red[warp][q][row][lane] = hsum(gx_);
            red[warp][NC + q][row][lane] = hsum(gy_);
          }
        }
        if constexpr (WANT_GR) {
          red[warp][2 * NC][row][lane] = hsum(k.glx * Fz);
          red[warp][2 * NC + 1][row][lane] = hsum(k.gly * Fz);
          red[warp][2 * NC + 2][row][lane] = hsum(k.glz * Fz);
        }
      };
      for (int j1 = ns; j1 > 0;) {
        const int j0 = ((j1 - 1) / TR) * TR;   // tile [j0, j1), at most TR steps
        constexpr bool VEC4 = !WaveLayout<T, W>::STEPMAJOR && TR % 4 == 0;
        if (VEC4 && j1 - j0 == TR) {
#pragma unroll 1
          for (int jj = TR - 4; jj >= 0; jj -= 4) {
            T wv[W][4];
#pragma unroll
            for (int w = 0; w < W; ++w) load4(wb + w * TCP + j0 + jj, wv[w]);
#pragma unroll
            for (int u = 3; u >= 0; --u) {
              T s[W];
#pragma unroll
              for (int w = 0; w < W; ++w) s[w] = wv[w][u];
              one_step(s, jj + u);
            }
          }
        } else {
          for (int j = j1 - 1; j >= j0; --j) {
            T s[W];
            load_step<T, W>(wb, TCP, j, s);
            one_step(s, j - j0);
          }
        }
        if constexpr (ROWS != 0) {
        __syncwarp();
        T(*ctab)[W][TR] = cta + (size_t)(red_par & 1) * NW;   // this tile's half of the double buffer
        if constexpr (WRED) warp_tile_reduce_weighted<T, NC, TR, W0, W1>(ft, wt, lane, ctab[warp]);
        else warp_tile_reduce<T, W, TR, W0, W1>(red[warp], lane, ctab[warp]);
        __syncthreads();   // the only CTA barrier per tile: `cta` alternates, `red` is re-written after it
        for (int e = tid; e < (W1 - W0) * TR; e += BLKT) {   // fixed-order combine of the warps
          const int w = W0 + e / TR, r = e % TR;
          if (j0 + r < j1) {
            T sum = ctab[0][w][r];
#pragma unroll
            for (int q = 1; q < NW; ++q) sum += ctab[q][w][r];
            T* dst = part + (size_t)w * nT + (c * K + j0 + r);
            // the slot belongs to this CTA alone, so a fire-and-forget RED keeps the result bitwise
            // reproducible and takes the L2 round trip of a read-modify-write off the critical path
            if (first) *dst = sum; else atomicAdd(dst, sum);
          }
        }
        ++red_par;
        }
        j1 = j0;
      }
      if constexpr (SG) sg_fold<T, V, NC, PK>(a, sgo, n, idx, ok, c == nChunks - 1, c == 0, k, sacc);
      if constexpr (ROWS == 0) __syncthreads();   // (else the reduce's barrier) everyone is done with wbuf[it&1] before it is refilled
      if (c > 0) {   // resynchronise the reconstructed state with the forward checkpoint
        mx = kx; my = ky; mz = kz;
      }
    }
    if (need_gmi) {
      from_frame(k, hx, hy);
      if (ok[0]) {
        T* op = a.gMi + ((size_t)n * nM + idx[0]) * 3;
        op[0] = getq<0>(hx); op[1] = getq<0>(hy); op[2] = getq<0>(hz);
      }
      if (PK == 2 && ok[PK - 1]) {
        T* op = a.gMi + ((size_t)n * nM + idx[PK - 1]) * 3;
        op[0] = getq<1>(hx); op[1] = getq<1>(hy); op[2] = getq<1>(hz);
      }
    }
    if constexpr (RD) {
      if (ro.grx) ro_grx_store<T, V, NC, PK, BLKT>(ro, n, nM, idx, ok, k, RO_ACC);
    }
  }
   }   // vid >= 0
   if (!a.sched) break;
   // done with this id: is any id still unclaimed (an SM that received fewer CTAs than planned)?  Normally one load.
   __syncthreads();
   if (tid == 0) {
     int* const sched = a.sched;
     int f = -1, sweep = s_sweep;
     if (*(volatile int*)&sched[SCHED_NCLAIMED] < NCTA) {
       for (; sweep < NCTA; ++sweep) {
         if (*(volatile int*)&sched[SCHED_CLAIM + sweep] == 0 && atomicCAS(&sched[SCHED_CLAIM + sweep], 0, 1) == 0) {
           f = sweep++;
           atomicAdd(&sched[SCHED_NCLAIMED], 1);
           break;
         }
       }
     }
     s_sweep = sweep;
     s_vid = f;
   }
   __syncthreads();
   vid = s_vid;
   if (vid < 0) break;
  }
#undef NCTA
#undef RO_W
#undef RO_ACC
#undef RO_GS
#ifdef MRPHY_CTA_TRACE
  if (tid == 0 && blockIdx.x < 8192 && n == 0) g_cta_trace[blockIdx.x][2] = gtime();
#endif
}


// ==========================================================================================
// Multi-coil (pTx) path on the tensor cores, fp32, NC >= 4 coils.
//
// The transmit field  Bx + i By [spin][step] = sum_c g b1[spin][c] rf[c][step]  is the one contraction on this path: per
// spin tile (128 spins = one CTA = the 128 TMEM lanes) and staged chunk (<= 64 steps) it is ONE product
//     D[128 spins][2 steps] = A[128][2 NC] * B[2 steps][2 NC]^T        A[s] = (g Re b1_c, g Im b1_c)_c
//                                                                       B[(j,x)] = (rx_c, -ry_c)_c   B[(j,y)] = (ry_c, rx_c)_c
// issued by one thread as tcgen05.mma (kind::tf32), accumulated in TMEM, and read back by the thread that owns the spin
// (thread t of warp w <-> TMEM lane 32 w + t) with tcgen05.ld -- 4 NC FMAs and 2 NC shared-memory operands per spin and
// step become one 64-bit TMEM read.  fp32 accuracy: every operand is split into two TF32-representable parts
// (hi = rn_tf32(x), mid = rn_tf32(x - hi)); the products mid*hi + hi*mid + hi*hi are exact in the tensor core and leave
// 2^-22 relative -- measured as accurate as the fp32 FMA chain it replaces (profiles/ubench/tc_field.cu: 7.5e-8 vs 7.4e-8).
// The pack kernel writes B (both parts) in the canonical K-major operand layout (tc_helpers.cuh), so a chunk still arrives
// with one TMA bulk copy; A is written once per tile by the threads.
constexpr int TC_TCMAX = 32;   // steps per staged chunk (= checkpoint interval) of the tensor-core kernels
template <int NC> struct TcLayout {
  static constexpr int KC = NC / 2;       // 16-byte K-chunks per operand row (K = 2 NC values)
  static constexpr int KSTEPS = NC / 4;   // tcgen05.mma instructions along K (8 values each)
  static constexpr int PER_STEP = 16 * KC + 3;                 // floats per step of a staged chunk: 2 parts x 2 rows x 2 NC + gr
  static constexpr int CHUNK_MAX = TC_TCMAX * PER_STEP;        // floats
  static constexpr int A_FLOATS = 2 * KC * 128 * 4;            // one tile's A, both parts
  static constexpr int TILE_COLS = 2 * TC_TCMAX;               // TMEM columns of one tile's field for one chunk: (Bx, By) per step
};
// PK spin tiles (128 spins each) per CTA: thread t owns spin t of every tile.  PK = 1: one spin per thread (scalar step), two
// TMEM buffers so that the product of chunk c+1 runs while chunk c is stepped.  PK = 2: two spins per thread as one f2 (FFMA2:
// half the issue slots -- the scalar loop is issue-bound, ncu: 78 % of the slots, 61 % of the FMA pipe), one TMEM buffer (the
// product of a chunk is waited for; four resident CTAs cover for it).  Either way 128 TMEM columns per CTA: 4 CTAs per SM.
template <int NC, int PK> struct TcCfg {
  static constexpr int NBUF = PK == 1 ? 2 : 1;                                   // TMEM buffers
  static constexpr int NST = (PK == 1 && NC <= 8) ? 3 : 2;                       // staged chunks
  static constexpr int BUF_COLS = PK * TcLayout<NC>::TILE_COLS;
  static constexpr int TMEM_COLS = NBUF * BUF_COLS;                              // 128
  // dynamic shared memory, in bytes from a 128-byte aligned base
  static constexpr size_t wbuf = 0;                                                                   // float[NST][CHUNK_MAX]
  static constexpr size_t sa = ((size_t)NST * TcLayout<NC>::CHUNK_MAX * 4 + 127) / 128 * 128;         // float[PK][2][KC][128][4]
  static constexpr size_t scr = sa + (size_t)PK * TcLayout<NC>::A_FLOATS * 4;                         // float[3 * 128 * PK]
  static constexpr size_t bars = scr + (size_t)3 * 128 * PK * 4;                     // full[NST], mma[2], tmem slot: 64 B
  static constexpr size_t bytes = bars + 64;
};

// pack for the tensor-core path: one thread per (n, chunk, step j < TCP, coil q < NC)
template <int NC>
__global__ void pack_waveform_tc_kernel(const float* __restrict__ rf, int64_t rf_sn, int64_t rf_sx, int64_t rf_st, int64_t rf_sc,
                                        const float* __restrict__ gr, int64_t gr_sn, int64_t gr_sx, int64_t gr_st, int nC,
                                        int nT, int K, int TCP, int nChunks, int64_t total, float* __restrict__ wave) {
  using L = TcLayout<NC>;
  const int rows = 2 * TCP;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int q = (int)(e % NC);
    const int j = (int)((e / NC) % TCP);
    const int c = (int)((e / ((int64_t)NC * TCP)) % nChunks);
    const int n = (int)(e / ((int64_t)NC * TCP * nChunks));
    const int t = c * K + j;
    const bool live = j < K && t < nT;
    float rx = 0.f, ry = 0.f;
    if (live && q < nC) {
      const float* p = rf + n * rf_sn + t * rf_st + q * rf_sc;
      rx = p[0];
      ry = p[rf_sx];
    }
    float* chunk = wave + ((size_t)n * nChunks + c) * (size_t)(TCP * L::PER_STEP);
    const float xh = tc::tf32_rn(rx), xm = tc::tf32_rn(rx - xh), yh = tc::tf32_rn(ry), ym = tc::tf32_rn(ry - yh);
    const int kc = q >> 1, pos = (q & 1) * 2;
    float* b_hi = chunk + ((size_t)(0 * L::KC + kc) * rows) * 4 + pos;
    float* b_mid = chunk + ((size_t)(1 * L::KC + kc) * rows) * 4 + pos;
    *reinterpret_cast<float2*>(b_hi + (size_t)(2 * j) * 4) = make_float2(xh, -yh);       // row (j, x)
    *reinterpret_cast<float2*>(b_hi + (size_t)(2 * j + 1) * 4) = make_float2(yh, xh);    // row (j, y)
    *reinterpret_cast<float2*>(b_mid + (size_t)(2 * j) * 4) = make_float2(xm, -ym);
    *reinterpret_cast<float2*>(b_mid + (size_t)(2 * j + 1) * 4) = make_float2(ym, xm);
    if (q < 3) chunk[(size_t)2 * L::KC * rows * 4 + (size_t)q * TCP + j] = live ? gr[n * gr_sn + q * gr_sx + t * gr_st] : 0.f;
  }
}

// Per-spin prologue of the tensor-core kernel: the scalar constants (no b1: SpinConst<float, 1>) and this thread's row of A
// = (g Re b1_c, g Im b1_c)_c in both TF32 parts.  The coils are walked two
// at a time so that the 2 NC sensitivities never sit in registers together.  A CTA barrier must follow before the first
// tcgen05.mma.
template <int NC, bool RELAX>
__device__ __forceinline__ void tc_load_spin(const KArgs<float>& a, int n, int i, float lx, float ly, float lz,
                                             SpinConst<float, 1>& k, float* sa, int tid) {
  using L = TcLayout<NC>;
  const double gam = ld_param(a.gamma, n, i);
  const double dt = ld_param(a.dt, n, 0);
  const double df = a.df.ptr ? ld_param(a.df, n, i) : 0.0;
  const double t1 = RELAX ? ld_param(a.T1, n, i) : 1.0;
  const double t2 = RELAX ? ld_param(a.T2, n, i) : 1.0;
  make_consts<float, 1>(k, gam, dt, RELAX, t1, t2, df, lx, ly, lz, nullptr, nullptr);
  const double g = 6.283185307179586476925286766559 * gam * dt;
  const float* bp = a.b1 + (int64_t)n * a.b1_sn + (int64_t)i * a.b1_sm;   // [re (nC) | im (nC)]
#pragma unroll 2
  for (int kc = 0; kc < L::KC; ++kc) {
    float v[4], h[4], m[4];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int c = 2 * kc + e;
      v[2 * e] = c < a.nC ? (float)(g * (double)bp[c]) : 0.f;              // one rounding per constant, as make_consts
      v[2 * e + 1] = c < a.nC ? (float)(g * (double)bp[a.nC + c]) : 0.f;
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) { h[e] = tc::tf32_rn(v[e]); m[e] = tc::tf32_rn(v[e] - h[e]); }
    *reinterpret_cast<float4*>(sa + ((size_t)(0 * L::KC + kc) * 128 + tid) * 4) = make_float4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<float4*>(sa + ((size_t)(1 * L::KC + kc) * 128 + tid) * 4) = make_float4(m[0], m[1], m[2], m[3]);
  }
  fence_proxy_async_smem();   // generic-proxy stores -> visible to the tensor core's (async-proxy) reads
}
// the products of one staged chunk, by ONE thread: per tile D = A_mid B_hi^T + A_hi B_mid^T + A_hi B_hi^T, then commit to `bar`
template <int NC, int PK>
__device__ __forceinline__ void tc_issue(const float* sa, const float* wb, int rows, uint32_t tmem, uint64_t* bar) {
  using L = TcLayout<NC>;
  const uint32_t idesc = tc::idesc_tf32(128, rows);
  const int pa[3] = {1, 0, 0}, pb[3] = {0, 1, 0};
  tc::fence_after_sync();
#pragma unroll
  for (int t = 0; t < PK; ++t) {
    bool acc = false;
#pragma unroll
    for (int q = 0; q < 3; ++q) {
#pragma unroll
      for (int ks = 0; ks < L::KSTEPS; ++ks) {
        tc::mma_tf32(tmem + t * L::TILE_COLS, tc::kmajor_desc(sa + (size_t)t * L::A_FLOATS + ((size_t)(pa[q] * L::KC + 2 * ks) * 128) * 4, 128),
                     tc::kmajor_desc(wb + ((size_t)(pb[q] * L::KC + 2 * ks) * rows) * 4, rows), idesc, acc);
        acc = true;
      }
    }
  }
  tc::commit(bar);
}

// Per chunk iteration `it` of a CTA (its tiles x chunks in order) thread 0 works ahead of the stepping threads, so that neither
// the copy nor (with two TMEM buffers) the tensor-core latency is exposed.  NST staged chunks, NBUF TMEM buffers:
//   TC_CHUNK_BEGIN   TMA(it + NST - 1) into the stage the steps of it - 1 have just left.  NBUF = 2, NST = 3: product(it + 1)
//                    into the other TMEM buffer (its operands landed an iteration ago); a tile's FIRST chunk also issues its
//                    own product here (A changes with the tile: products never run ahead of a tile).  NBUF = 1: every chunk
//                    issues its own product here.  Then everybody waits for the product of chunk `it`.
//   TC_PRODUCT_AHEAD NBUF = 2, NST = 2 (16 coils: a stage is 17 KB): product(it + 1) after 16 steps, when its operands have
//                    landed (a copy takes ~1-2 us, 8 steps ~1 us).
// full[s]: k-th use has parity k & 1; mma_bar[b] likewise.
#define TC_CHUNK_BEGIN(CHUNK_OF, FIRST_OF_TILE, HAS_NEXT_IN_TILE)                                                          \
  if (tid == 0) {                                                                                                          \
    if (it + (NST - 1) < total) {                                                                                          \
      const uint32_t sq = (it + (NST - 1)) % NST;                                                                          \
      mbar_arrive_expect_tx(&full[sq], chunk_bytes);                                                                       \
      bulk_g2s(wbuf[sq], wave_n + (size_t)(CHUNK_OF(it + (NST - 1))) * a.chunk_elems, chunk_bytes, &full[sq]);              \
    }                                                                                                                      \
    if ((FIRST_OF_TILE) || NBUF == 1) {                                                                                    \
      mbar_wait(&full[it % NST], (it / NST) & 1);                                                                          \
      tc_issue<NC, PK>(sa, wbuf[it % NST], rows, tmem + (it % NBUF) * C::BUF_COLS, &mma_bar[it % NBUF]);                    \
    }                                                                                                                      \
    if (NBUF == 2 && NST == 3 && (HAS_NEXT_IN_TILE)) {                                                                     \
      mbar_wait(&full[(it + 1) % NST], ((it + 1) / NST) & 1);                                                              \
      tc_issue<NC, PK>(sa, wbuf[(it + 1) % NST], rows, tmem + ((it + 1) % NBUF) * C::BUF_COLS, &mma_bar[(it + 1) % NBUF]);  \
    }                                                                                                                      \
  }                                                                                                                        \
  mbar_wait(&full[it % NST], (it / NST) & 1);                                                                              \
  mbar_wait(&mma_bar[it % NBUF], (it / NBUF) & 1);                                                                         \
  tc::fence_after_sync();
#define TC_PRODUCT_AHEAD(HAS_NEXT_IN_TILE)                                                                                 \
  if (NBUF == 2 && NST == 2 && tid == 0 && (HAS_NEXT_IN_TILE)) {                                                           \
    mbar_wait(&full[(it + 1) % NST], ((it + 1) / NST) & 1);                                                                \
    tc_issue<NC, PK>(sa, wbuf[(it + 1) % NST], rows, tmem + ((it + 1) % NBUF) * C::BUF_COLS, &mma_bar[(it + 1) % NBUF]);    \
  }

// REC, RD as in fused_fwd_kernel (this kernel has no spin frame: the state is in the lab frame throughout); the readout's
// shared memory follows C::bytes.
template <int POL, bool RELAX, int NC, int PK, int OPT = OPT_NONE>
__global__ void __launch_bounds__(128, (NC <= 8 ? 4 : (PK == 1 ? 3 : 2))) fused_fwd_tc_kernel(const KArgs<float> a, const RecOut<float> rec) {
  constexpr bool REC = OPT == OPT_RECORD, RD = OPT == OPT_READOUT;
  const RoOut<float>& ro = rec.ro;
  using L = TcLayout<NC>;
  using C = TcCfg<NC, PK>;
  typedef float T;
  typedef typename Pack<float, PK>::type V;
  constexpr int BLKT = 128, NST = C::NST, NBUF = C::NBUF;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float(*wbuf)[L::CHUNK_MAX] = reinterpret_cast<float(*)[L::CHUNK_MAX]>(smem_raw + C::wbuf);
  float* const sa = reinterpret_cast<float*>(smem_raw + C::sa);
  float* const scr = reinterpret_cast<float*>(smem_raw + C::scr);
  uint64_t* const full = reinterpret_cast<uint64_t*>(smem_raw + C::bars);
  uint64_t* const mma_bar = full + NST;
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(full + NST + 2);
  // RD (see RoOut), behind C::bytes; addresses formed where used
#define RO_W reinterpret_cast<V*>(smem_raw + C::bytes)
#define RO_TILES reinterpret_cast<float*>(smem_raw + C::bytes + (size_t)2 * ro.nRx * BLKT * sizeof(V))
#define RO_CTAB (RO_TILES + (BLKT / 32) * RO_COLS * 32)
  int nb = 0;   // RD: records buffered since the last flush | ctab parity (ro_flush)
  const int tid = threadIdx.x, warp = tid >> 5, n = blockIdx.y;
  const int TCP = a.TCP, K = a.K, nT = a.nT, nChunks = a.nChunks, nM = a.nM, rows = 2 * TCP;
  const uint32_t chunk_bytes = (uint32_t)(a.chunk_elems * sizeof(float));
  const float* wave_n = a.wave + (size_t)n * nChunks * a.chunk_elems;
  const int tiles = (nM + BLKT * PK - 1) / (BLKT * PK);   // CTA tiles of PK x 128 consecutive spins
  const int my_tiles = ((int)blockIdx.x < tiles) ? (tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const uint32_t total = (uint32_t)my_tiles * (uint32_t)nChunks;
  if (tid == 0) {
#pragma unroll
    for (int q = 0; q < NST; ++q) mbar_init(&full[q], 1);
    mbar_init(&mma_bar[0], 1);
    mbar_init(&mma_bar[1], 1);
    fence_barrier_init();
  }
  if (warp == 0) tc::tmem_alloc<C::TMEM_COLS>(tmem_slot);
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = *tmem_slot, tlane = tmem + ((uint32_t)(warp * 32) << 16);
#define FWD_CHUNK_OF(i) ((i) % (uint32_t)nChunks)
  if (tid == 0) {
    for (uint32_t q = 0; q + 1 < (uint32_t)NST && q < total; ++q) {
      mbar_arrive_expect_tx(&full[q], chunk_bytes);
      bulk_g2s(wbuf[q], wave_n + (size_t)FWD_CHUNK_OF(q) * a.chunk_elems, chunk_bytes, &full[q]);
    }
  }
  uint32_t it = 0;
  for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    SpinConst<V, 1> k;
    V mx, my, mz;
    int idx[PK];
    bool ok[PK];
#pragma unroll
    for (int q = 0; q < PK; ++q) {
      const int i = (tile * PK + q) * BLKT + tid;
      ok[q] = i < nM;
      idx[q] = ok[q] ? i : nM - 1;
    }
    {   // (the previous tile's products have completed: every chunk waits on its mma_bar, so A may be rewritten)
      V lx, ly, lz;
      load_vec3_tile<T, V, PK, BLKT>(a.loc + (int64_t)n * a.loc_sn, a.loc_sm, tile, nM, idx, scr, lx, ly, lz);
      if constexpr (PK == 1) {
        tc_load_spin<NC, RELAX>(a, n, idx[0], lx, ly, lz, k, sa, tid);
      } else {
        SpinConst<float, 1> k0, k1;
        tc_load_spin<NC, RELAX>(a, n, idx[0], getq<0>(lx), getq<0>(ly), getq<0>(lz), k0, sa, tid);
        tc_load_spin<NC, RELAX>(a, n, idx[1], getq<1>(lx), getq<1>(ly), getq<1>(lz), k1, sa + L::A_FLOATS, tid);
        k = pack2<1>(k0, k1);
      }
    }
    load_vec3_tile<T, V, PK, BLKT>(a.Mi + (int64_t)n * a.Mi_sn, a.Mi_sm, tile, nM, idx, scr, mx, my, mz);
    tc::fence_before_sync();
    __syncthreads();
    const V glx = k.glx, gly = k.gly, glz = k.glz, gbz0 = k.gbz0, e1 = k.e1, e2 = k.e2;
    int rc = RD ? ro.every : rec.every, rr = 0;   // REC, RD: steps to the next recorded state, its index
    if constexpr (RD) ro_weights<T, V, 1, PK, BLKT>(ro, n, idx, ok, k, RO_W);
    for (int c = 0; c < nChunks; ++c, ++it) {
      TC_CHUNK_BEGIN(FWD_CHUNK_OF, c == 0, c + 1 < nChunks)
      const float* gw = wbuf[it % NST] + (size_t)2 * L::KC * rows * 4;   // gr rows [3][TCP]
      const int ns = min(K, nT - c * K);
      const uint32_t tcol = tlane + (it % NBUF) * C::BUF_COLS;
      // 8 steps from 16 TMEM columns per tile: (Bx, By) of steps j0 .. j0 + 7
      auto steps8 = [&](const float (&b)[PK][16], int j0) {
        float g[3][8];
#pragma unroll
        for (int w = 0; w < 3; ++w) {
          load4(gw + w * TCP + j0, *reinterpret_cast<float(*)[4]>(&g[w][0]));
          load4(gw + w * TCP + j0 + 4, *reinterpret_cast<float(*)[4]>(&g[w][4]));
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (j0 + u < ns) {
            const V bz = fma_(glx, V(g[0][u]), fma_(gly, V(g[1][u]), fma_(glz, V(g[2][u]), gbz0)));
            const V bx = mkv(b[0][2 * u], b[PK - 1][2 * u], (V*)nullptr), by = mkv(b[0][2 * u + 1], b[PK - 1][2 * u + 1], (V*)nullptr);
            step_fwd<V, POL, RELAX>(bx, by, bz, e1, e2, mx, my, mz);
            if constexpr (REC) {
              if (--rc == 0) {
                rec_store<T, V, PK>(rec, nM, n, rr++, idx, ok, mx, my, mz);
                rc = rec.every;
              }
            }
            if constexpr (RD) {
              if (--rc == 0) {
                ro_accum<T, V, BLKT>(ro, RO_W, RO_TILES + (size_t)warp * RO_COLS * 32, nb & 0xffff, mx, my);
                ++rr;
                if ((++nb & 0xffff) == ro.rt || rr == ro.nR) ro_flush<T, BLKT>(ro, RO_TILES, RO_CTAB, n, rr, nb, tile == (int)blockIdx.x);
                rc = ro.every;
              }
            }
          }
        }
      };
      auto issue = [&](float (&b)[PK][16], int g) {
#pragma unroll
        for (int q = 0; q < PK; ++q) tc::tmem_ld16_issue(tcol + q * L::TILE_COLS + 16 * g, b[q]);
      };
      auto wait = [&](float (&b)[PK][16]) {
        tc::tmem_ld_wait(b[0]);
        if constexpr (PK == 2) tc::tmem_ld_wait(b[1]);
      };
      float b0[PK][16], b1[PK][16];
      issue(b0, 0);
#pragma unroll 1
      for (int g = 0; g < TC_TCMAX / 8; g += 2) {   // the read of the next 8 steps is in flight while these 8 are computed
        if (8 * g < ns) {
          wait(b0);
          if (8 * (g + 1) < ns) issue(b1, g + 1);
          steps8(b0, 8 * g);
          if (ns <= 8) { TC_PRODUCT_AHEAD(c + 1 < nChunks) }
        }
        if (8 * (g + 1) < ns) {
          wait(b1);
          if (g + 2 < TC_TCMAX / 8 && 8 * (g + 2) < ns) issue(b0, g + 2);
          steps8(b1, 8 * (g + 1));
          if (g == 0) { TC_PRODUCT_AHEAD(c + 1 < nChunks) }
        }
      }
      if (c + 1 < nChunks) {   // checkpoint: state after (c+1)*K steps (streaming stores, see fused_fwd_kernel)
        T* cp = a.ckpt + ((size_t)n * (nChunks - 1) + c) * 3 * (size_t)nM;
        if (ok[0]) {
          __stcs(cp + idx[0], getq<0>(mx));
          __stcs(cp + (size_t)nM + idx[0], getq<0>(my));
          __stcs(cp + 2 * (size_t)nM + idx[0], getq<0>(mz));
        }
        if (PK == 2 && ok[PK - 1]) {
          __stcs(cp + idx[PK - 1], getq<1>(mx));
          __stcs(cp + (size_t)nM + idx[PK - 1], getq<1>(my));
          __stcs(cp + 2 * (size_t)nM + idx[PK - 1], getq<1>(mz));
        }
      }
      tc::fence_before_sync();
      __syncthreads();   // everyone is done with this chunk's stage and TMEM buffer
      tc::fence_after_sync();
    }
    if (ok[0]) {
      T* op = a.Mo + ((size_t)n * nM + idx[0]) * 3;
      op[0] = getq<0>(mx); op[1] = getq<0>(my); op[2] = getq<0>(mz);
    }
    if (PK == 2 && ok[PK - 1]) {
      T* op = a.Mo + ((size_t)n * nM + idx[PK - 1]) * 3;
      op[0] = getq<1>(mx); op[1] = getq<1>(my); op[2] = getq<1>(mz);
    }
  }
#undef FWD_CHUNK_OF
#undef RO_W
#undef RO_TILES
#undef RO_CTAB
  __syncthreads();
  if (warp == 0) tc::tmem_free<C::TMEM_COLS>(tmem);
}

#undef TC_CHUNK_BEGIN
#undef TC_PRODUCT_AHEAD

}  // namespace mrphy

// =============================================================================================
// C ABI
using namespace mrphy;

static thread_local char g_err[512] = "";
static thread_local int g_launches = 0;
// bench-only, process-wide on purpose: backward runs on the autograd engine's thread
static int g_timing = 0;
static cudaEvent_t g_ev0 = nullptr, g_ev1 = nullptr;
static int g_ev_valid = 0;
namespace mrphy {
char* err_buf() { return g_err; }
int& launch_count() { return g_launches; }
void timing_begin(cudaStream_t st) {
  if (!g_timing) return;
  if (!g_ev0 && (cudaEventCreate(&g_ev0) != cudaSuccess || cudaEventCreate(&g_ev1) != cudaSuccess)) {
    cudaGetLastError();
    g_ev0 = g_ev1 = nullptr;
    return;
  }
  g_ev_valid = 0;
  cudaEventRecord(g_ev0, st);
}
void timing_end(cudaStream_t st) {
  if (!g_timing || !g_ev0) return;
  cudaEventRecord(g_ev1, st);
  g_ev_valid = 1;
}
}  // namespace mrphy

extern "C" int mrphy_kernel_timing(int enable) {
  g_timing = enable ? 1 : 0;
  g_ev_valid = 0;
  return MRPHY_OK;
}
extern "C" float mrphy_last_kernel_ms(void) {
  if (!g_ev_valid) return -1.0f;
  float ms = -1.0f;
  if (cudaEventSynchronize(g_ev1) != cudaSuccess || cudaEventElapsedTime(&ms, g_ev0, g_ev1) != cudaSuccess) {
    cudaGetLastError();
    return -1.0f;
  }
  return ms;
}

#ifdef MRPHY_CTA_TRACE
extern "C" int mrphy_debug_cta_trace(unsigned long long* host_out, int n_ctas) {
  return cudaMemcpyFromSymbol(host_out, mrphy::g_cta_trace, sizeof(unsigned long long) * 4 * (size_t)n_ctas) == cudaSuccess ? 0 : -2;
}
#endif
extern "C" int mrphy_abi_version(void) { return MRPHY_ABI_VERSION; }
extern "C" const char* mrphy_last_error(void) { return g_err; }
extern "C" int mrphy_last_launch_count(void) { return g_launches; }

extern "C" int mrphy_device_sm_count(int device) {
  int v = 0;
  if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) {
    fail(MRPHY_ERR_CUDA, "cudaDeviceGetAttribute failed%s");
    cudaGetLastError();
    return MRPHY_ERR_CUDA;
  }
  return v;
}

namespace {

struct Plan {
  int NC;        // coils held in registers (1,2,4,8)
  int PK;        // spins per thread (2 = packed f2 arithmetic, fp32 single-coil only)
  int BLKT;      // threads per CTA
  int K, TCP, nChunks, W;
  int WS, stepmajor;   // staged waveform layout (WaveLayout): row-major [W][TCP] or step-major [TCP][WS]
  int sum_coils; // no b1Map
  int tiles;     // spin tiles per batch entry (BLKT*PK spins each)
  int Pmax;      // upper bound on CTAs per batch entry (sizes the partial-sum workspace)
  int rows;      // gradients wanted by the backward: bit 0 dL/drf, bit 1 dL/dgr (MRPHY_SKIP_GRF / _GGR clear them)
  int chunk_elems;   // elements per staged waveform chunk (WS * TCP)
  int tc;        // fp32 forward with >= 4 coils on the tensor cores (fused_fwd_tc_kernel); its staged chunks (TcLayout) have
  int tc_TCP, tc_chunk_elems;   // tc_TCP (multiple of 8) steps and tc_chunk_elems elements; the backward re-packs for itself
};

int sm_count_cached() {
  // per device ordinal: a process may drive GPUs of different size, and the first call may come from any of them
  static int sms[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cudaGetLastError();
    return 148;   // B200; only used for grid sizing
  }
  if (dev < 0 || dev >= 64) dev = 0;
  if (sms[dev] <= 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) {
      cudaGetLastError();
      v = 148;
    }
    sms[dev] = v;
  }
  return sms[dev];
}

int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  if (!e) return dflt;
  const int v = atoi(e);
  return v > 0 ? v : dflt;
}

int make_plan(const mrphy_fused_args* a, Plan* p, bool need_device) {
  if (!a) return fail(MRPHY_ERR_ARG, "null args%s");
  if (a->dtype != MRPHY_F32 && a->dtype != MRPHY_F64) return fail(MRPHY_ERR_ARG, "dtype must be MRPHY_F32 or MRPHY_F64%s");
  if (a->N < 1 || a->nM < 1 || a->nT < 1 || a->nC < 1 || a->N > 65535) return fail(MRPHY_ERR_ARG, "need 1 <= N <= 65535 and nM, nT, nC >= 1%s");
  p->sum_coils = a->b1 == nullptr;
  const int nc = p->sum_coils ? 1 : a->nC;
  if (nc > 16) return fail(MRPHY_ERR_ARG, "more than 16 transmit coils with a b1Map are not supported%s");
  p->NC = nc <= 1 ? 1 : nc <= 2 ? 2 : nc <= 4 ? 4 : nc <= 8 ? 8 : 16;
  if (a->K < 1 || a->K > ((a->dtype == MRPHY_F32 && p->NC == 1) ? MRPHY_TCMAX1 : TCMAX))
    return fail(MRPHY_ERR_ARG, "checkpoint interval K must be in [1, 64] (fp32 with one transmit channel: [1, 128])%s");
  p->W = 2 * p->NC + 3;
  p->stepmajor = (size_t)p->W * (a->dtype == MRPHY_F64 ? 8 : 4) > 44;
  p->WS = p->stepmajor ? ((p->W + 3) & ~3) : p->W;
  p->K = a->K;
  p->TCP = (a->K + 3) & ~3;
  p->nChunks = (a->nT + a->K - 1) / a->K;
  p->chunk_elems = p->WS * p->TCP;
  // fp32 with >= 4 coils: the transmit field as a TF32 tensor-core product (MRPHY_B200_TC=0: the FMA kernels)
  const char* tc_env = getenv("MRPHY_B200_TC");
  p->tc = a->dtype == MRPHY_F32 && p->NC >= MRPHY_TC_MIN_NC && a->K <= 32 && !(tc_env && tc_env[0] == '0');   // TC_TCMAX
  p->tc_TCP = (a->K + 7) & ~7;
  p->tc_chunk_elems = p->tc ? p->tc_TCP * (16 * (p->NC / 2) + 3) : 0;   // TcLayout<NC>::PER_STEP
  // fp32 single coil: two spins per thread, packed FFMA2 arithmetic.  fp64 and multi-coil: one spin per thread (scalar
  // kernels); a build with -DMRPHY_FP32_SCALAR also carries the fp32 single-coil scalar kernels (MRPHY_B200_PACK=1)
#ifdef MRPHY_FP32_SCALAR
  const int want = env_int("MRPHY_B200_PACK", 2);
#else
  const int want = 2;
#endif
  p->PK = (a->dtype == MRPHY_F32 && p->NC == 1 && want == 2) ? 2 : 1;
  p->BLKT = p->PK == 2 ? 64 : 128;
  p->tiles = (a->nM + p->BLKT * (p->PK == 2 ? 2 : 1) - 1) / (p->BLKT * (p->PK == 2 ? 2 : 1));
  const int sms = need_device ? sm_count_cached() : 148;
  const int cap = env_int("MRPHY_B200_MAX_CTAS", sms * 32);   // 32 CTAs/SM is the hardware limit
  int P = p->tiles;
  if ((int64_t)P * a->N > cap) P = cap / a->N > 0 ? cap / a->N : 1;
  p->Pmax = P;
  p->rows = ((a->flags & MRPHY_SKIP_GRF) ? 0 : 1) | ((a->flags & MRPHY_SKIP_GGR) ? 0 : 2);
  return MRPHY_OK;
}

// CTAs per batch entry: all CTAs co-resident (one wave), c CTAs per SM chosen so that the tiles split
// evenly -- minimise passes(c) * c over c in [occ/2, occ]; e.g. 64^3 spins on 148 SMs: c = 7, 2 passes.
int pick_ctas(const Plan& p, int N, int occ, bool sm_aware = false, int warps_per_cta = 4) {
  const int sms = sm_count_cached();
  occ = occ < 1 ? 1 : occ;
  const int forced = env_int("MRPHY_B200_CTAS_PER_SM", 0);
  // With SM-aware tile ownership (backward, one batch entry) every SM serves ceil or floor(tiles / sms) tiles whatever
  // c is, so take all the resident slots the tiles can fill.
  if (sm_aware && N == 1 && !forced && p.tiles >= 2 * sms) {
    const int c = p.tiles / sms < occ ? p.tiles / sms : occ;
    if (sms * c <= p.Pmax) return sms * c;     // never more ids than the partial-sum workspace was sized for (MRPHY_B200_MAX_CTAS)
  }
  int best_P = 1, best_cost = 1 << 30;
  for (int c = occ; c >= (occ + 1) / 2; --c) {
    if (forced) c = forced < occ ? forced : occ;
    // the four schedulers of an SM must carry the same number of warps (the kernels are throughput-bound per scheduler:
    // 11 two-warp CTAs = 6,6,5,5 warps cost 9 % at C4): skip CTA counts that do not fill them evenly
    if (!forced && (c * warps_per_cta) % 4 != 0 && c > 1 && occ > 2) continue;
    int P = (int)((int64_t)sms * c / N);
    if (P < 1) P = 1;
    if (P > p.Pmax) P = p.Pmax;
    const int passes = (p.tiles + P - 1) / P;
    const int cost = passes * c;
    if (cost < best_cost) { best_cost = cost; best_P = P; }
    if (forced) break;
  }
  return best_P;
}

}  // namespace

extern "C" size_t mrphy_fused_ckpt_elems(const mrphy_fused_args* a) {
  Plan p;
  if (make_plan(a, &p, false) != MRPHY_OK) return 0;
  const size_t n = (size_t)a->N * (size_t)(p.nChunks - 1) * 3 * (size_t)a->nM;
  return n ? n : 1;
}
extern "C" size_t mrphy_fused_wave_elems(const mrphy_fused_args* a) {
  Plan p;
  if (make_plan(a, &p, false) != MRPHY_OK) return 0;
  return (size_t)a->N * p.nChunks * (p.tc_chunk_elems > p.chunk_elems ? p.tc_chunk_elems : p.chunk_elems);
}
extern "C" size_t mrphy_fused_partial_elems(const mrphy_fused_args* a) {
  Plan p;
  if (make_plan(a, &p, true) != MRPHY_OK) return 0;
  // + the scheduling ints + one finished-CTA counter per batch entry (design tail of the gradient epilogue)
  return (size_t)a->N * p.Pmax * p.W * (size_t)a->nT + (size_t)(SCHED_CLAIM + p.Pmax) + (size_t)a->N;
}

extern "C" size_t mrphy_fused_readout_elems(const mrphy_fused_args* a) {
  Plan p;
  if (make_plan(a, &p, true) != MRPHY_OK) return 0;
  if (a->nRx < 1 || a->nRx > 16 || a->nR < 1) return 0;
  return (size_t)a->N * p.Pmax * (size_t)a->nR * 2 * a->nRx;
}

namespace {

template <typename T>
int check_common(const mrphy_fused_args* a, bool bwd) {
  if (!a->Mi && !bwd) return fail(MRPHY_ERR_ARG, "Mi is null%s");
  if (!a->rf || !a->gr || !a->loc) return fail(MRPHY_ERR_ARG, "rf, gr and loc are required%s");
  if (!a->gamma.ptr || !a->dt.ptr) return fail(MRPHY_ERR_ARG, "gamma and dt are required%s");
  if ((a->T1.ptr == nullptr) != (a->T2.ptr == nullptr)) return fail(MRPHY_ERR_ARG, "T1 and T2: both or neither (sims.py:68)%s");
  if (!a->Mo || !a->ckpt || !a->wave) return fail(MRPHY_ERR_ARG, "Mo, ckpt and wave buffers are required%s");
  if (bwd && (!a->gMo || !a->partials)) return fail(MRPHY_ERR_ARG, "gMo and partials are required%s");
  if (bwd && ((!a->grf && !(a->flags & MRPHY_SKIP_GRF)) || (!a->ggr && !(a->flags & MRPHY_SKIP_GGR))))
    return fail(MRPHY_ERR_ARG, "grf / ggr are required unless MRPHY_SKIP_GRF / MRPHY_SKIP_GGR is set%s");
  if (bwd && (a->flags & MRPHY_NEED_GMI) && !a->gMi) return fail(MRPHY_ERR_ARG, "gMi is null but MRPHY_NEED_GMI is set%s");
  return MRPHY_OK;
}

template <typename T>
KArgs<T> make_kargs(const mrphy_fused_args* a, const Plan& p) {
  KArgs<T> k;
  memset(&k, 0, sizeof(k));
  k.N = a->N; k.nM = a->nM; k.nT = a->nT; k.K = p.K; k.TCP = p.TCP; k.nChunks = p.nChunks; k.P = p.Pmax;
  k.chunk_elems = p.chunk_elems;
  k.Mi = (const T*)a->Mi; k.Mi_sn = a->Mi_sn; k.Mi_sm = a->Mi_sm;
  k.loc = (const T*)a->loc; k.loc_sn = a->loc_sn; k.loc_sm = a->loc_sm;
  k.b1 = (const T*)a->b1; k.b1_sn = a->b1_sn; k.b1_sm = a->b1_sm; k.nC = a->nC;
  k.df = a->df; k.T1 = a->T1; k.T2 = a->T2; k.gamma = a->gamma; k.dt = a->dt;
  k.Mo = (T*)a->Mo; k.ckpt = (T*)a->ckpt; k.wave = (const T*)a->wave;
  k.gMo = (const T*)a->gMo; k.gMo_sn = a->gMo_sn; k.gMo_sm = a->gMo_sm;
  k.gMi = (T*)a->gMi; k.partials = (T*)a->partials;
  k.sched = nullptr; k.n_sm = 0; k.c_per_sm = 0; k.done = nullptr;
  return k;
}

template <int NC>
int launch_pack_tc(const mrphy_fused_args* a, const Plan& p, cudaStream_t st) {
  const int64_t total = (int64_t)a->N * p.nChunks * p.tc_TCP * NC;
  const int grid = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
  const int64_t rf_sc = (a->flags & MRPHY_RF_COIL_DIM) ? a->rf_sc : 0;
  pack_waveform_tc_kernel<NC><<<grid, 256, 0, st>>>((const float*)a->rf, a->rf_sn, a->rf_sx, a->rf_st, rf_sc, (const float*)a->gr,
                                                    a->gr_sn, a->gr_sx, a->gr_st, a->nC, a->nT, p.K, p.tc_TCP, p.nChunks, total,
                                                    (float*)a->wave);
  ++g_launches;
  CK(cudaGetLastError());
  return MRPHY_OK;
}

template <typename T>
int launch_pack(const mrphy_fused_args* a, const Plan& p, cudaStream_t st, bool tc_layout = false) {
  if (tc_layout) {
    if (p.NC == 4) return launch_pack_tc<4>(a, p, st);
    if (p.NC == 8) return launch_pack_tc<8>(a, p, st);
    return launch_pack_tc<16>(a, p, st);
  }
  const int64_t total = (int64_t)a->N * p.nChunks * p.WS * p.TCP;
  const int grid = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
  const int64_t rf_sc = (a->flags & MRPHY_RF_COIL_DIM) ? a->rf_sc : 0;
  pack_waveform_kernel<T><<<grid, 256, 0, st>>>((const T*)a->rf, a->rf_sn, a->rf_sx, a->rf_st, rf_sc, (const T*)a->gr,
                                                a->gr_sn, a->gr_sx, a->gr_st, a->nC, p.NC, p.sum_coils, a->nT, p.K,
                                                p.TCP, p.nChunks, p.WS, p.stepmajor, total, (T*)a->wave);
  ++g_launches;
  CK(cudaGetLastError());
  return MRPHY_OK;
}

// P (CTAs per batch entry) actually launched by the last backward kernel; the finalize kernel needs it
thread_local int g_last_P = 0;
// ... by the last forward kernel: the readout's finalize sums that many slots
thread_local int g_last_fwd_P = 0;
// records a staged chunk of K steps can produce (the backward's dL/dS staging)
inline int ro_chunk_records(int K, int every) { return (K + every - 1) / every; }

template <typename T, int POL, bool RELAX, int NC, int PK, int BLKT, int OPT>
int launch_fwd_s(KArgs<T> k, const Plan& p, cudaStream_t st, const RecOut<T>& rec) {
  constexpr bool REC = OPT == OPT_RECORD;
  const size_t smem =
      OPT == OPT_READOUT ? ro_fwd_smem(rec.ro.nRx, BLKT, (int)sizeof(typename Pack<T, PK>::type), (int)sizeof(T)) : 0;
  auto kern = fused_fwd_kernel<T, POL, RELAX, NC, PK, BLKT, OPT>;
  if (smem) CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, BLKT, smem));
  k.P = pick_ctas(p, k.N, occ, false, BLKT / 32);
  g_last_fwd_P = k.P;
  dim3 grid(k.P, k.N);
  if (OPT && getenv("MRPHY_B200_DEBUG"))
    fprintf(stderr, "[mrphy_b200] fused_fwd<%s,NC=%d,PK=%d,BLK=%d,%s,%s=1> grid=(%d,%d) tiles=%d occ=%d K=%d every=%d\n",
            sizeof(T) == 4 ? "f32" : "f64", NC, PK, BLKT, POL == TRIG_PRECISE ? "precise" : "fast", REC ? "REC" : "RD", k.P, k.N,
            p.tiles, occ, p.K, REC ? rec.every : rec.ro.every);
  timing_begin(st);
  kern<<<grid, BLKT, smem, st>>>(k, rec);
  timing_end(st);
  ++g_launches;
  CK(cudaGetLastError());
  return MRPHY_OK;
}
template <typename T, int POL, bool RELAX, int NC, int PK, int BLKT, int ROWS, bool SG, int OPT>
int launch_bwd_s(KArgs<T> k, const Plan& p, int need_gmi, cudaStream_t st, const SgOut<T>& sg, const RecOut<T>& rec) {
  constexpr bool REC = OPT == OPT_RECORD;
  const size_t smem = BwdSmem<T, NC, BLKT, PK>::bytes +
                      (OPT == OPT_READOUT ? ro_bwd_smem(rec.ro.nRx, BLKT, (int)sizeof(typename Pack<T, PK>::type), (int)sizeof(T),
                                                        ro_chunk_records(p.K, rec.ro.every)) : 0);
  auto kern = fused_bwd_kernel<T, POL, RELAX, NC, PK, BLKT, ROWS, SG, OPT>;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));   // static + dynamic may exceed 48 KB
  int occ = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, BLKT, smem));
  Plan q = p;   // the backward may use larger CTAs than the forward the plan was sized for: fewer, larger tiles
  q.tiles = (k.nM + BLKT * PK - 1) / (BLKT * PK);
  if (q.Pmax > q.tiles) q.Pmax = q.tiles;
  const bool sm_aware = env_int("MRPHY_B200_SCHED", 1) != 2;
  k.P = pick_ctas(q, k.N, occ, sm_aware, BLKT / 32);
  if (k.P < 1 || k.P > p.Pmax) return fail(MRPHY_ERR_ARG, "internal: backward grid exceeds the partial-sum workspace%s");
  g_last_P = k.P;
  dim3 grid(k.P, k.N);
  // SM-aware tile ownership when the grid is exactly c CTAs on each SM of one batch entry (see SCHED_*)
  const int sms = sm_count_cached();
  if (k.N == 1 && k.P % sms == 0 && k.P > sms && sms <= SCHED_SM_SLOTS && sm_aware) {
    k.sched = reinterpret_cast<int*>(k.partials + (size_t)k.N * p.Pmax * p.W * (size_t)k.nT);
    k.n_sm = sms;
    k.c_per_sm = k.P / sms;
    CK(cudaMemsetAsync(k.sched, 0, sizeof(int) * (size_t)(SCHED_CLAIM + k.P), st));
  }
  if (getenv("MRPHY_B200_DEBUG"))
    fprintf(stderr, "[mrphy_b200] fused_bwd<%s,NC=%d,PK=%d,BLK=%d,%s,ROWS=%d,SG=%d%s> grid=(%d,%d) tiles=%d occ=%d smem=%zu K=%d\n",
            sizeof(T) == 4 ? "f32" : "f64", NC, PK, BLKT, POL == TRIG_PRECISE ? "precise" : "fast", ROWS, (int)SG,
            REC ? ",REC=1" : (OPT == OPT_READOUT ? ",RD=1" : ""), k.P, k.N, q.tiles, occ, smem, p.K);
  timing_begin(st);
  kern<<<grid, BLKT, smem, st>>>(k, need_gmi, sg, rec);
  timing_end(st);
  ++g_launches;
  CK(cudaGetLastError());
  return MRPHY_OK;
}

// Resident CTAs per SM of a tensor-core kernel.  cudaOccupancyMaxActiveBlocksPerMultiprocessor answers 1 for kernels that
// allocate TMEM (measured), although CTAs do share an SM as long as their TMEM columns fit: count registers, shared memory
// and the 512 TMEM columns by hand.
template <typename Kern>
int tc_occupancy(Kern kern, size_t dyn_smem, int tmem_cols) {
  cudaFuncAttributes fa;
  if (cudaFuncGetAttributes(&fa, kern) != cudaSuccess) {
    cudaGetLastError();
    return 1;
  }
  const int regs_per_cta = ((fa.numRegs + 7) / 8 * 8) * 128;
  int occ = regs_per_cta > 0 ? 65536 / regs_per_cta : 1;
  const size_t per_cta = dyn_smem + fa.sharedSizeBytes + 1024;   // 1 KB reserved per CTA
  const int by_smem = (int)((size_t)228 * 1024 / per_cta);
  if (by_smem < occ) occ = by_smem;
  if (512 / tmem_cols < occ) occ = 512 / tmem_cols;
  const int forced = env_int("MRPHY_B200_TC_OCC", 0);
  if (forced) occ = forced;
  return occ < 1 ? 1 : occ;
}

// tensor-core multi-coil kernels (fp32): at most 4 CTAs per SM, each owns 128 of the 512 TMEM columns
template <int POL, bool RELAX, int NC, int PK, int OPT>
int launch_fwd_tc_pk(KArgs<float> k, const Plan& p, cudaStream_t st, const RecOut<float>& rec) {
  using C = TcCfg<NC, PK>;
  constexpr bool REC = OPT == OPT_RECORD;
  const size_t smem =
      C::bytes + (OPT == OPT_READOUT ? ro_fwd_smem(rec.ro.nRx, 128, (int)sizeof(typename Pack<float, PK>::type), 4) : 0);
  auto kern = fused_fwd_tc_kernel<POL, RELAX, NC, PK, OPT>;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k.TCP = p.tc_TCP;
  k.chunk_elems = p.tc_chunk_elems;
  const int occ = tc_occupancy(kern, smem, C::TMEM_COLS);
  const int tiles = (k.nM + 128 * PK - 1) / (128 * PK);
  k.P = (int)((int64_t)sm_count_cached() * occ / k.N);   // every resident slot (pick_ctas trades slots for even passes)
  if (k.P < 1) k.P = 1;
  if (k.P > tiles) k.P = tiles;
  if (OPT == OPT_READOUT && k.P > p.Pmax) k.P = p.Pmax;   // one readout slot per CTA: mrphy_fused_readout_elems sized Pmax of them
  g_last_fwd_P = k.P;
  dim3 grid(k.P, k.N);
  if (getenv("MRPHY_B200_DEBUG"))
    fprintf(stderr, "[mrphy_b200] fused_fwd_tc<NC=%d,PK=%d%s> grid=(%d,%d) tiles=%d occ=%d smem=%zu K=%d\n", NC, PK,
            REC ? ",REC=1" : (OPT == OPT_READOUT ? ",RD=1" : ""), k.P, k.N, tiles, occ, smem, p.K);
  timing_begin(st);
  kern<<<grid, 128, smem, st>>>(k, rec);
  timing_end(st);
  ++g_launches;
  CK(cudaGetLastError());
  return MRPHY_OK;
}
template <int POL, bool RELAX, int NC, int OPT>
int launch_fwd_tc(const KArgs<float>& k, const Plan& p, cudaStream_t st, const RecOut<float>& rec) {
  // two spin tiles per CTA (packed f2 step): measured 3 % (4, 8 coils) to 17 % (16 coils) faster than one tile with two TMEM
  // buffers; a build with -DMRPHY_TC_SCALAR also carries the one-tile kernels (MRPHY_B200_TC_PACK=1) for measurements
#ifdef MRPHY_TC_SCALAR
  if (env_int("MRPHY_B200_TC_PACK", 2) == 1) return launch_fwd_tc_pk<POL, RELAX, NC, 1, OPT>(k, p, st, rec);
#endif
  return launch_fwd_tc_pk<POL, RELAX, NC, 2, OPT>(k, p, st, rec);
}
// One launch of the kernels with spins in registers: the forward, or the backward with its ROWS / SG.  With per-spin gradients
// the backward takes the ROWS == 0 kernel when no waveform gradient is wanted, else all rows (the finalize reads only the
// wanted ones); without, the spin-packed kernels also come with dL/drf-only and dL/dgr-only rows.
template <typename T, int POL, bool RELAX, int NC, int PK, int OPT>
int launch(bool bwd, const KArgs<T>& k, const Plan& p, int need_gmi, cudaStream_t st, const SgOut<T>& sg, const RecOut<T>& rec) {
  if (!bwd) return launch_fwd_s<T, POL, RELAX, NC, PK, PK == 2 ? 64 : 128, OPT>(k, p, st, rec);
  constexpr int B = PK == 2 ? MRPHY_BWD_BLKT : 128;
  if (sg.any())
    return p.rows == 0 ? launch_bwd_s<T, POL, RELAX, NC, PK, B, 0, true, OPT>(k, p, need_gmi, st, sg, rec)
                       : launch_bwd_s<T, POL, RELAX, NC, PK, B, 3, true, OPT>(k, p, need_gmi, st, sg, rec);
  if constexpr (PK == 2) {
    if (p.rows == 1) return launch_bwd_s<T, POL, RELAX, NC, PK, B, 1, false, OPT>(k, p, need_gmi, st, sg, rec);   // dL/drf only
    if (p.rows == 2) return launch_bwd_s<T, POL, RELAX, NC, PK, B, 2, false, OPT>(k, p, need_gmi, st, sg, rec);   // dL/dgr only
  }
  return launch_bwd_s<T, POL, RELAX, NC, PK, B, 3, false, OPT>(k, p, need_gmi, st, sg, rec);
}

template <typename T, int POL, bool RELAX, int OPT>
int dispatch_nc(bool bwd, const KArgs<T>& k, const Plan& p, int need_gmi, cudaStream_t st, const SgOut<T>& sg,
                const RecOut<T>& rec) {
  if constexpr (sizeof(T) == 4) {
    if (p.PK == 2) return launch<T, POL, RELAX, 1, 2, OPT>(bwd, k, p, need_gmi, st, sg, rec);
  }
#ifdef MRPHY_ONLY_PK2   /* tuning builds (profiles/operand_model.py): compile the default fp32 kernels only */
  return fail(MRPHY_ERR_ARG, "built with MRPHY_ONLY_PK2%s");
#else
  if constexpr (sizeof(T) == 4) {
    // 2 coils: two spins per thread (FFMA2) like the single-coil kernels; same tiles of 128 spins, same staging
    if (p.NC == 2 && env_int("MRPHY_B200_NC2_PACK", 2) == 2 && (!bwd || env_int("MRPHY_B200_NC2_PACK_BWD", 2) == 2))
      return launch<T, POL, RELAX, 2, 2, OPT>(bwd, k, p, need_gmi, st, sg, rec);
    if (p.tc && !bwd) {   // forward with >= 4 coils: transmit field on the tensor cores
      if (p.NC == 4) return launch_fwd_tc<POL, RELAX, 4, OPT>(k, p, st, rec);
      if (p.NC == 8) return launch_fwd_tc<POL, RELAX, 8, OPT>(k, p, st, rec);
      return launch_fwd_tc<POL, RELAX, 16, OPT>(k, p, st, rec);
    }
  }
  switch (p.NC) {
    case 1:
#ifndef MRPHY_FP32_SCALAR
      if constexpr (sizeof(T) == 4) return fail(MRPHY_ERR_ARG, "internal: fp32 single-coil scalar kernels not built%s");
      else
#endif
      return launch<T, POL, RELAX, 1, 1, OPT>(bwd, k, p, need_gmi, st, sg, rec);
    case 2: return launch<T, POL, RELAX, 2, 1, OPT>(bwd, k, p, need_gmi, st, sg, rec);
    case 4: return launch<T, POL, RELAX, 4, 1, OPT>(bwd, k, p, need_gmi, st, sg, rec);
    case 8: return launch<T, POL, RELAX, 8, 1, OPT>(bwd, k, p, need_gmi, st, sg, rec);
    case 16: return launch<T, POL, RELAX, 16, 1, OPT>(bwd, k, p, need_gmi, st, sg, rec);
  }
  return fail(MRPHY_ERR_ARG, "internal: bad NC%s");
#endif
}

template <typename T, int POL>
int dispatch_pol(bool bwd, const KArgs<T>& k, const Plan& p, bool relax, int opt, int need_gmi, cudaStream_t st,
                 const SgOut<T>& sg, const RecOut<T>& rec) {
  if (opt == OPT_READOUT)
    return relax ? dispatch_nc<T, POL, true, OPT_READOUT>(bwd, k, p, need_gmi, st, sg, rec)
                 : dispatch_nc<T, POL, false, OPT_READOUT>(bwd, k, p, need_gmi, st, sg, rec);
  if (opt == OPT_RECORD)
    return relax ? dispatch_nc<T, POL, true, OPT_RECORD>(bwd, k, p, need_gmi, st, sg, rec)
                 : dispatch_nc<T, POL, false, OPT_RECORD>(bwd, k, p, need_gmi, st, sg, rec);
  return relax ? dispatch_nc<T, POL, true, OPT_NONE>(bwd, k, p, need_gmi, st, sg, rec)
               : dispatch_nc<T, POL, false, OPT_NONE>(bwd, k, p, need_gmi, st, sg, rec);
}

// an option is on when any of its fields is set (check_record / check_readout then want all of them consistent); the
// readout shares every / nR with the record
bool recording(const mrphy_fused_args* a) { return a->every || a->nR || a->Mt || a->gMt; }
bool reading_out(const mrphy_fused_args* a) { return a->nRx || a->rx || a->S || a->gS || a->grx || a->S_work; }

template <typename T>
int dispatch(bool bwd, const mrphy_fused_args* a, const Plan& p, cudaStream_t st, int* done) {
  KArgs<T> k = make_kargs<T>(a, p);
  k.done = done;
  const SgOut<T> sg{(T*)a->gloc, (T*)a->gsz, (T*)a->gb1};
  const int opt = reading_out(a) ? OPT_READOUT : recording(a) ? OPT_RECORD : OPT_NONE;
  RecOut<T> rec{};
  if (opt == OPT_RECORD) rec = RecOut<T>{(T*)a->Mt, (const T*)a->gMt, a->every, a->nR, RoOut<T>{}};
  if (opt == OPT_READOUT)
    rec.ro = RoOut<T>{(const T*)a->rx, a->rx_sn, a->rx_sm, a->nRx, a->every, a->nR, RO_COLS / (2 * a->nRx), (T*)a->S_work,
                      (const T*)a->gS, (T*)a->grx};
  const bool relax = a->T1.ptr != nullptr;
  const int need_gmi = (a->flags & MRPHY_NEED_GMI) ? 1 : 0;
  // fp64 has one trigonometry (TRIG_FAST names it), so only fp32 instantiates both
  if constexpr (sizeof(T) == 4) {
    if ((a->flags & MRPHY_TRIG_PRECISE) && !(bwd && (a->flags & MRPHY_TRIG_FAST_BWD)))
      return dispatch_pol<T, TRIG_PRECISE>(bwd, k, p, relax, opt, need_gmi, st, sg, rec);
  }
  return dispatch_pol<T, TRIG_FAST>(bwd, k, p, relax, opt, need_gmi, st, sg, rec);
}

// the record stride and its buffer (Mt for the forward, gMt for the backward)
int check_record(const mrphy_fused_args* a, bool bwd) {
  if (a->every < 1 || a->every > a->nT || a->nR != a->nT / a->every)
    return fail(MRPHY_ERR_ARG, "record: need 1 <= every <= nT and nR == nT / every%s");
  if (bwd ? !a->gMt : !a->Mt) return fail(MRPHY_ERR_ARG, bwd ? "record: gMt is null%s" : "record: Mt is null%s");
  return MRPHY_OK;
}

// the readout: its stride (a->every, a->nR), coils and buffers; exclusive with record and the design tail
int check_readout(const mrphy_fused_args* a, bool bwd) {
  if (a->Mt || a->gMt) return fail(MRPHY_ERR_ARG, "readout: does not combine with record (Mt / gMt)%s");
  if (a->design) return fail(MRPHY_ERR_ARG, "readout: does not combine with the design tail%s");
  if (a->every < 1 || a->every > a->nT || a->nR != a->nT / a->every)
    return fail(MRPHY_ERR_ARG, "readout: need 1 <= every <= nT and nR == nT / every%s");
  if (a->nRx < 1 || a->nRx > 16) return fail(MRPHY_ERR_ARG, "readout: need 1 <= nRx <= 16 receive coils%s");
  if (bwd ? !a->gS : (!a->S || !a->S_work)) return fail(MRPHY_ERR_ARG, bwd ? "readout: gS is null%s" : "readout: S or work is null%s");
  return MRPHY_OK;
}

template <typename T>
int run_fwd(const mrphy_fused_args* a, cudaStream_t st) {
  Plan p;
  int rc = make_plan(a, &p, true);
  if (rc) return rc;
  if ((rc = check_common<T>(a, false))) return rc;
  const bool ro = reading_out(a);
  if (ro && (rc = check_readout(a, false))) return rc;
  if (!ro && recording(a) && (rc = check_record(a, false))) return rc;
  if ((rc = launch_pack<T>(a, p, st, p.tc != 0))) return rc;
  if ((rc = dispatch<T>(false, a, p, st, nullptr))) return rc;
  if (!ro) return MRPHY_OK;
  dim3 grid((a->nR * 2 * a->nRx + 31) / 32, a->N), block(32, 8);
  readout_finalize_kernel<T><<<grid, block, 0, st>>>((const T*)a->S_work, g_last_fwd_P, a->nR, a->nRx, (T*)a->S);
  ++g_launches;
  CK(cudaGetLastError());
  return MRPHY_OK;
}

// the re-parametrisation the design tail can take: adjoint of an rf half and/or a gradient half that ends in a gradient
int check_design(const mrphy_fused_args* a, const mrphy_reparam_args* d) {
  if (d->dtype != a->dtype || d->N != a->N || d->nT != a->nT || !d->adjoint)
    return fail(MRPHY_ERR_ARG, "design: dtype, N, nT must match the simulation and adjoint must be set%s");
  if (d->rf_kind < 0 || d->rf_kind > 2 || d->gr_kind < 0 || d->gr_kind > 2 || (d->rf_kind == 0 && d->gr_kind == 0))
    return fail(MRPHY_ERR_ARG, "design: rf_kind 0..2, gr_kind 0..2 (ts -> s is not a gradient), not both 0%s");
  if (d->rf_kind) {
    if (a->flags & MRPHY_SKIP_GRF) return fail(MRPHY_ERR_ARG, "design: the rf half needs dL/drf (MRPHY_SKIP_GRF is set)%s");
    if (d->nC != ((a->flags & MRPHY_RF_COIL_DIM) ? a->nC : 1)) return fail(MRPHY_ERR_ARG, "design: nC differs from rf's coil dimension%s");
    if (!d->rho || !d->theta || !d->rfmax || !d->grho || !d->gtheta) return fail(MRPHY_ERR_ARG, "design: rho, theta, rfmax, grho, gtheta are required%s");
  }
  if (d->gr_kind) {
    if (a->flags & MRPHY_SKIP_GGR) return fail(MRPHY_ERR_ARG, "design: the gradient half needs dL/dgr (MRPHY_SKIP_GGR is set)%s");
    if (!d->ts || !d->gts || (d->gr_kind == 1 && !d->smax) || !d->dt.ptr) return fail(MRPHY_ERR_ARG, "design: ts, gts, dt (and smax for ts -> g) are required%s");
  }
  return MRPHY_OK;
}

template <typename T>
int run_bwd(const mrphy_fused_args* a, int wave_is_packed, cudaStream_t st) {
  Plan p;
  int rc = make_plan(a, &p, true);
  if (rc) return rc;
  if ((rc = check_common<T>(a, true))) return rc;
  const bool ro = reading_out(a);
  if (ro && (rc = check_readout(a, true))) return rc;
  const mrphy_reparam_args* d = a->design;
  const bool rec = !ro && recording(a), sg = a->gloc || a->gsz || a->gb1;
  if (d && (rec || sg)) return fail(MRPHY_ERR_ARG, "design: does not combine with record or per-spin gradients%s");
  if (d && (rc = check_design(a, d))) return rc;
  if (rec && (rc = check_record(a, true))) return rc;
  if (a->gb1 && !a->b1) return fail(MRPHY_ERR_ARG, "spin gradients: gb1 needs b1%s");
  // (after a tensor-core forward `wave` holds that kernel's operand tiles: the backward stages its own layout over them)
  if ((!wave_is_packed || p.tc) && (rc = launch_pack<T>(a, p, st))) return rc;
  // finished-CTA counters of the design tail: behind the scheduling ints, zeroed by the backward kernel itself
  int* const done = d ? reinterpret_cast<int*>((T*)a->partials + (size_t)a->N * p.Pmax * p.W * (size_t)a->nT) + SCHED_CLAIM + p.Pmax : nullptr;
  if ((rc = dispatch<T>(true, a, p, st, done))) return rc;
  if (sg && p.rows == 0) return MRPHY_OK;   // per-spin gradients only: nothing to finalize
  dim3 grid((a->nT + 31) / 32, p.W, a->N), block(32, 32);
  const int coil_dim = (a->flags & MRPHY_RF_COIL_DIM) ? 1 : 0;
  const int w_lo = (p.rows & 1) ? 0 : 2 * p.NC, w_hi = (p.rows & 2) ? p.W : 2 * p.NC;
  T* tail = nullptr;   // MRPHY_ZERO_GRAD_TAIL: the 4 spare elements behind the last gradient of the caller's flat buffer
  if (a->flags & MRPHY_ZERO_GRAD_TAIL)
    tail = (p.rows & 2) ? (T*)a->ggr + (size_t)a->N * 3 * a->nT
                        : (p.rows & 1) ? (T*)a->grf + (size_t)a->N * 2 * a->nT * (coil_dim ? a->nC : 1) : nullptr;
  if (d)
    grad_finalize_design_kernel<T><<<grid, block, 0, st>>>((const T*)a->partials, g_last_P, p.W, p.NC, a->nC, a->nT, coil_dim,
                                                           p.sum_coils, (T)-1, (T*)a->grf, (T*)a->ggr, w_lo, w_hi, *d, done,
                                                           tail);
  else
    grad_finalize_kernel<T><<<grid, block, 0, st>>>((const T*)a->partials, g_last_P, p.W, p.NC, a->nC, a->nT, coil_dim,
                                                    p.sum_coils, (T)-1, (T*)a->grf, (T*)a->ggr, w_lo, w_hi, tail);
  ++g_launches;
  CK(cudaGetLastError());
  return MRPHY_OK;
}

}  // namespace

extern "C" int mrphy_blochsim_fused_fwd(const mrphy_fused_args* a, void* cuda_stream) {
  g_launches = 0;
  g_err[0] = 0;
  if (!a) return fail(MRPHY_ERR_ARG, "null args%s");
  cudaStream_t st = (cudaStream_t)cuda_stream;
  return a->dtype == MRPHY_F64 ? run_fwd<double>(a, st) : run_fwd<float>(a, st);
}

extern "C" int mrphy_blochsim_fused_bwd(const mrphy_fused_args* a, int wave_is_packed, void* cuda_stream) {
  g_launches = 0;
  g_err[0] = 0;
  if (!a) return fail(MRPHY_ERR_ARG, "null args%s");
  cudaStream_t st = (cudaStream_t)cuda_stream;
  return a->dtype == MRPHY_F64 ? run_bwd<double>(a, wave_is_packed, st) : run_bwd<float>(a, wave_is_packed, st);
}
