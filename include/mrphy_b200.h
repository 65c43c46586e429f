/* mrphy_b200.h -- C ABI of libmrphy_b200.so (hand-written CUDA for sm_100a).
 *
 * The drop-in boundary of the Bloch-simulation hot path of MRphy.py (reference v0.2.0).  The
 * reference is pure Python/PyTorch and has no FFI; what a maintainer would bind is exactly the
 * operator pair below, called from `mrphy/sims.py` (`BlochSim.forward/backward`, sims.py:31-269)
 * and from `mrphy/mobjs.py` (`SpinArray.applypulse`, mobjs.py:394-450).  INTEGRATION.md shows the
 * ctypes stub.  No torch types cross this boundary: plain device pointers, element strides and
 * sizes.  The library never allocates or frees device memory; every buffer (outputs, checkpoints,
 * workspaces) is owned by the caller.  All entry points are re-entrant, launch asynchronously
 * on the given CUDA stream and return 0 or a negative mrphy_status; mrphy_last_error() gives the
 * thread-local message.
 *
 * Shapes follow the reference (mrphy/__init__.py:20-47): N batch, nM spins per batch (compact),
 * nT time steps, nC transmit coils.  `dtype` is MRPHY_F32 or MRPHY_F64 and selects the arithmetic
 * type T of the kernel: Mi/Mo, rf, gr, loc, b1Map, gradients and workspaces are arrays of T.
 * The per-spin / per-batch physical constants (gamma, dt, T1, T2, df) may independently be fp32
 * or fp64 (`*_f64` flags), so the float64 0-dim defaults of the reference (mrphy/__init__.py:58-65)
 * are consumed without a cast.  Strides are in ELEMENTS; a stride of 0 broadcasts (the reference
 * stores T1_/T2_/gamma_ as stride-0 expands, mobjs.py:389).
 */
#ifndef MRPHY_B200_H
#define MRPHY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MRPHY_ABI_VERSION 8

enum mrphy_dtype { MRPHY_F32 = 0, MRPHY_F64 = 1 };

enum mrphy_status {
  MRPHY_OK = 0,
  MRPHY_ERR_ARG = -1,      /* inconsistent sizes / null pointers / unsupported option   */
  MRPHY_ERR_CUDA = -2,     /* a CUDA runtime call or kernel launch failed               */
  MRPHY_ERR_WORKSPACE = -3 /* caller-provided workspace too small                       */
};

enum mrphy_flags {
  MRPHY_TRIG_PRECISE = 1 << 0, /* fp32 only: rotation coefficients on the FMA pipe (half-angle polynomials in |b|^2 up to 2 pi, Newton
                                  rsqrt + Cody-Waite reduced polynomial sincos beyond) instead of MUFU.SIN/COS/RSQ */
  MRPHY_NEED_GMI = 1 << 1,     /* backward: also write dL/dMi                                   */
  MRPHY_RF_COIL_DIM = 1 << 2,  /* rf (and its gradient) carry the trailing nCoils dimension     */
  MRPHY_NEED_GBEFF = 1 << 3,   /* explicit-field backward: also write dL/dBeff                  */
  MRPHY_TRIG_FAST_BWD = 1 << 4, /* with MRPHY_TRIG_PRECISE: the BACKWARD kernel uses MUFU trigonometry (M unchanged) */
  MRPHY_SKIP_GRF = 1 << 5,     /* fused backward: dL/drf is not wanted (grf may be NULL); its rows of the spin   */
  MRPHY_SKIP_GGR = 1 << 6,     /* reduction are not computed.  Likewise dL/dgr (ggr may be NULL).               */
  MRPHY_ZERO_GRAD_TAIL = 1 << 7 /* fused backward: grf, ggr are consecutive parts of ONE buffer [grf | ggr | 4 spare elements]
                                  (what a sharded run all-reduces in place); the epilogue zeroes the 4 spare elements    */
};

/* A strided per-spin scalar: element (n, i) lives at ptr[n*sn + i*sm]; f64 selects the type. */
typedef struct mrphy_param {
  const void* ptr; /* device pointer or NULL when the quantity is absent */
  int64_t sn, sm;
  int32_t f64;
  int32_t _pad;
} mrphy_param;

/* Arguments of the fused path  rf,gr,loc,df,b1Map -> Beff -> (u,phi) -> rotate -> relax  for all
 * nT steps, replacing  beffective.rfgr2beff (beffective.py:107-168) + sims.BlochSim.forward
 * (sims.py:31-132)  and, for the backward entry point, sims.BlochSim.backward (sims.py:134-269)
 * + the autograd of rfgr2beff (sum over spins -> rf.grad, gr.grad).                            */
typedef struct mrphy_fused_args {
  int32_t dtype;  /* mrphy_dtype */
  int32_t flags;  /* mrphy_flags */
  int32_t N, nM, nT;
  int32_t nC;     /* coils of rf; with b1 == NULL the coils are summed (beffective.py:147-151) */
  int32_t K;      /* checkpoint interval in steps: 1..64; fp32 with one transmit channel (nC == 1 or
                     b1 == NULL): 1..128.  fp32, >= 3 coils, K <= 32: the forward runs its tensor-core kernel */
  int32_t _pad;

  const void* Mi; int64_t Mi_sn, Mi_sm;   /* (N,nM,3), inner stride 1                          */
  const void* rf; int64_t rf_sn, rf_sx, rf_st, rf_sc; /* (N,2,nT[,nC])                         */
  const void* gr; int64_t gr_sn, gr_sx, gr_st;        /* (N,3,nT)                              */
  const void* loc; int64_t loc_sn, loc_sm;            /* (N,nM,3), inner stride 1              */
  const void* b1; int64_t b1_sn, b1_sm;   /* (N,nM,2,nC) inner (2,nC) contiguous, or NULL      */
  mrphy_param df;                         /* (N,nM) Hz, or ptr NULL                            */
  mrphy_param T1, T2;                     /* (N,nM) s; both NULL = no relaxation (sims.py:68)  */
  mrphy_param gamma;                      /* (N,nM) Hz/G                                       */
  mrphy_param dt;                         /* (N,) s  (sm ignored)                              */

  void* Mo;        /* fwd: out (N,nM,3) contiguous.  bwd: in, the forward output               */
  void* ckpt;      /* fwd: out, bwd: in.  mrphy_fused_ckpt_elems() elements of T               */
  void* wave;      /* scratch, mrphy_fused_wave_elems() elements of T (packed waveform)        */

  /* backward only */
  const void* gMo; int64_t gMo_sn, gMo_sm; /* dL/dMo (N,nM,3), inner stride 1                  */
  void* gMi;       /* out (N,nM,3) contiguous when MRPHY_NEED_GMI                              */
  void* grf;       /* out (N,2,nT[,nC]) contiguous                                             */
  void* ggr;       /* out (N,3,nT) contiguous                                                  */
  void* partials;  /* scratch, mrphy_fused_partial_elems() elements of T                       */

  /* options, off when zero / NULL (see the entry points below) */
  int32_t every, nR;   /* record: 1 <= every <= nT, nR == nT / every                                 */
  void* Mt;            /* record, fwd: out [N][nR][3][nM] contiguous                                 */
  const void* gMt;     /* record, bwd: in, dL/dMt in the same layout                                 */
  void* gloc;          /* per-spin gradients, bwd: out (N,nM,3) contiguous, or NULL                  */
  void* gsz;           /* per-spin gradients, bwd: out (N,nM) contiguous, or NULL                    */
  void* gb1;           /* per-spin gradients, bwd: out (N,nM,2,nC) contiguous, or NULL (needs b1)    */
  const struct mrphy_reparam_args* design;   /* design tail, bwd: the re-parametrisation, or NULL  */
  int32_t nRx, _pad2;  /* readout: receive coils, 1..16                                              */
  const void* rx; int64_t rx_sn, rx_sm; /* readout: (N,nM,2,nRx) receive map, inner (2,nRx) contiguous, or NULL (c = 1) */
  void* S;             /* readout, fwd: out (N,2,nR,nRx) contiguous                                  */
  const void* gS;      /* readout, bwd: in, dL/dS like S                                             */
  void* grx;           /* readout, bwd: out dL/drx (N,nM,2,nRx) contiguous, or NULL                  */
  void* S_work;        /* readout, fwd: scratch, mrphy_fused_readout_elems() elements of T           */
} mrphy_fused_args;

int mrphy_abi_version(void);
const char* mrphy_last_error(void);

/* Device facts the host side needs for sizing (queried once per device, cached). */
int mrphy_device_sm_count(int device);

/* Workspace sizes, in ELEMENTS of T.  They depend only on dtype, N, nM, nT, nC, K, b1 != NULL (the readout's S_work also
 * on nR and nRx: 0 unless 1 <= nRx <= 16 and nR >= 1). */
size_t mrphy_fused_ckpt_elems(const mrphy_fused_args* a);
size_t mrphy_fused_wave_elems(const mrphy_fused_args* a);
size_t mrphy_fused_partial_elems(const mrphy_fused_args* a);
size_t mrphy_fused_readout_elems(const mrphy_fused_args* a);

/* Forward: writes Mo and ckpt.  Launches: pack_waveform, blochsim_fused_fwd.  Two options, off when their fields are zero:
 *
 * Record (a->every != 0): the magnetisation during the pulse.  The forward also writes the state after every `every` steps,
 *   Mt[n][r][xyz][i] = M of spin i after (r+1)*every steps, r = 0 .. nR-1, nR = nT / every   (lab frame, like Mo)
 * -- what the forward returns as Mo for the pulse cut to its first (r+1)*every samples.  Needs a->Mt.  Up to 16 transmit
 * coils, like every fused call.  No workspace beyond the existing ones.
 *
 * Readout (any of a->nRx, a->rx, a->S, a->gS, a->grx, a->S_work set): the receive signal of the magnetisation every
 * `a->every` steps, summed over the spins inside the forward kernel,
 *   S[n][xy][r][k] (Sx + i Sy) = sum_i (cx + i cy)[n][i][k] * (Mx + i My)[n][i] after (r+1)*every steps,  r < nR = nT / every
 * (lab frame, the state record would return; no conjugation, no scale).  rx == NULL: c = 1.  a->every / a->nR give the stride
 * as for record.  Needs a->S and a->S_work; a readout_finalize launch follows.  S is bitwise reproducible: each CTA sums its
 * tiles into its own slot of S_work, the finalize sums the slots in a fixed order.  Excludes record and the design tail. */
int mrphy_blochsim_fused_fwd(const mrphy_fused_args* a, void* cuda_stream);
/* Backward: reads Mo, ckpt, gMo; writes grf, ggr (and gMi).  Launches: pack_waveform (unless
 * `wave` still holds the packed waveform of the matching forward: pass wave_is_packed != 0),
 * blochsim_fused_bwd, grad_reduce_finalize.  Four options, each off when its fields are zero / NULL:
 *
 * Record (a->every != 0): the backward of a recording forward with the same every / nR.  It takes dL/dMt (a->gMt, in
 * the layout of Mt) on top of dL/dMo; a->gMo is required (zeros when the loss ignores Mo).
 *
 * Per-spin gradients (any of a->gloc, a->gsz, a->gb1 non-NULL): what the autograd of rfgr2beff gives upstream for loc,
 * df, b1Map and gamma (beffective.py:137-167), without the dense field or dL/dBeff.  Each output is the sum over time
 * that mrphy_rfgr2beff_spin_grads forms from dL/dBeff, with the same meaning and layout:
 *   gloc (N,nM,3)     = sum_t gr[:,t] * gBz[t]                              (dL/dloc)
 *   gsz  (N,nM)       = sum_t gBz[t]                                        (dL/ddf = gsz/gamma, dL/dgamma = -gsz*df/gamma^2)
 *   gb1  (N,nM,2,nC)  = sum_t (rx_c gBx + ry_c gBy,  rx_c gBy - ry_c gBx)    (dL/db1Map; requires a->b1)
 * contiguous, any of them NULL = not wanted.  gMi, grf and ggr are bitwise those of a call without per-spin gradients.
 * With MRPHY_SKIP_GRF | MRPHY_SKIP_GGR (a fixed pulse) the backward forms no spin reduction and skips the finalize
 * launch.  Combines with record.
 *
 * Design tail (a->design non-NULL): the adjoint of the re-parametrisation fused into the gradient epilogue (SURVEY 8f-2):
 * what autograd does upstream in two stages -- BlochSim.backward (sims.py:187-269) -> dL/drf, dL/dgr, then the backward
 * of utils.t-rho-theta2rf / l-rho-theta2rf / ts2s / s2g (utils.py:114-131, 239-256, 293-330) -> dL/drho, dL/dtheta,
 * dL/dts.  `design` describes the chain that produced a->rf and/or a->gr: adjoint != 0, dtype / N / nT as in `a`,
 * nC = trailing coil dimension of rf; rf_kind 0..2 and gr_kind 0..2 as in mrphy_design_waveform (0: that waveform is
 * not re-parametrised); design->grf / ->ggr are ignored -- the tail reads a->grf / a->ggr, which are written as usual.
 * Same launches: the last CTA of the epilogue to finish for a batch entry evaluates that entry's adjoint and writes
 * design->grho, ->gtheta, ->gts.  Combines with neither record, per-spin gradients nor readout (MRPHY_ERR_ARG).
 *
 * Readout (the forward's fields): the backward of a readout forward.  It takes dL/dS (a->gS) on top of dL/dMo (zeros when
 * the loss ignores M) and, with a->grx, writes dL/dcx = sum_r (gSx Mx + gSy My), dL/dcy = sum_r (gSy Mx - gSx My).  Combines
 * with per-spin gradients.  MRPHY_ERR_ARG before any launch for: a->Mt / a->gMt or a->design set, nRx outside 1..16, a null
 * S / S_work (fwd) or gS (bwd), every / nR inconsistent.  No workspace beyond mrphy_fused_partial_elems().            */
int mrphy_blochsim_fused_bwd(const mrphy_fused_args* a, int wave_is_packed, void* cuda_stream);

/* Arguments of the explicit-field path: the API-faithful replacement of sims.BlochSim
 * (sims.py:24-269) for callers that hand in a dense Beff (N,nM,nT,3), e.g. tests/test_sims.py:88
 * upstream.  Backward returns dL/dMi and the dense dL/dBeff like the reference.                  */
typedef struct mrphy_beff_args {
  int32_t dtype;  /* mrphy_dtype */
  int32_t flags;  /* MRPHY_TRIG_PRECISE | MRPHY_NEED_GMI | MRPHY_NEED_GBEFF */
  int32_t N, nM, nT;
  int32_t K;      /* checkpoint interval (>= 1) */
  const void* Mi; int64_t Mi_sn, Mi_sm;          /* (N,nM,3), inner stride 1 */
  const void* Beff; int64_t B_sn, B_sm, B_st;    /* (N,nM,nT,3), inner stride 1 */
  mrphy_param T1, T2, gamma, dt;
  void* Mo;        /* fwd out / bwd in, (N,nM,3) contiguous */
  void* ckpt;      /* fwd out / bwd in, mrphy_beff_ckpt_elems() elements of T */
  const void* gMo; int64_t gMo_sn, gMo_sm;
  void* gMi;       /* bwd out (N,nM,3) contiguous when MRPHY_NEED_GMI */
  void* gBeff;     /* bwd out (N,nM,nT,3) contiguous when MRPHY_NEED_GBEFF */
} mrphy_beff_args;

size_t mrphy_beff_ckpt_elems(const mrphy_beff_args* a);
int mrphy_blochsim_beff_fwd(const mrphy_beff_args* a, void* cuda_stream);
int mrphy_blochsim_beff_bwd(const mrphy_beff_args* a, void* cuda_stream);

/* Standalone field synthesis, replacing beffective.rfgr2beff (beffective.py:107-168) for callers that
 * want the dense field: Beff (N,nM,nT,3) contiguous out.  HBM-bound: 12 B/spin.step written (fp32). */
typedef struct mrphy_rfgr2beff_args {
  int32_t dtype, flags;  /* MRPHY_RF_COIL_DIM */
  int32_t N, nM, nT, nC;
  const void* rf; int64_t rf_sn, rf_sx, rf_st, rf_sc;
  const void* gr; int64_t gr_sn, gr_sx, gr_st;
  const void* loc; int64_t loc_sn, loc_sm;            /* inner stride 1 */
  const void* b1; int64_t b1_sn, b1_sm;               /* (N,nM,2,nC) inner contiguous, or NULL */
  mrphy_param df, gamma;                              /* df.ptr NULL = no off-resonance */
  void* Beff;
  const void* gBeff;                                  /* adjoint in: dL/dBeff (N,nM,nT,3) contiguous */
  void* grf; void* ggr;                               /* adjoint out: dL/drf like rf (contiguous), dL/dgr (N,3,nT) */
  void* partials;                                     /* adjoint workspace, mrphy_rfgr2beff_partial_elems() */
  void* gloc; void* gsz; void* gb1;                   /* per-spin adjoint out (mrphy_rfgr2beff_spin_grads), each may be NULL */
} mrphy_rfgr2beff_args;
int mrphy_rfgr2beff(const mrphy_rfgr2beff_args* a, void* cuda_stream);
/* The spin sums of the autograd of rfgr2beff (upstream: bmm / expand / sum backward): dL/drf_c = sum_i conj(b1_c)*gBxy,
 * dL/dgr = sum_i loc*gBz -- one pass over dL/dBeff (12 B/spin.step read, fp32), two-stage and bitwise reproducible. */
size_t mrphy_rfgr2beff_partial_elems(const mrphy_rfgr2beff_args* a);
int mrphy_rfgr2beff_bwd(const mrphy_rfgr2beff_args* a, void* cuda_stream);
/* The per-spin half of that autograd -- sums over TIME instead of over spins -- in the same single pass over dL/dBeff:
 *   gloc (N,nM,3)     = sum_t gr[:,t] * gBz[t]                        (dL/dloc)
 *   gsz  (N,nM)       = sum_t gBz[t]                                  (dL/ddf = gsz/gamma, dL/dgamma = -gsz*df/gamma^2: caller)
 *   gb1  (N,nM,2,nC)  = sum_t (rx_c gBx + ry_c gBy,  rx_c gBy - ry_c gBx)   (dL/db1Map; nC = 1 when rf has no coil dim)
 * contiguous outputs, any of them NULL = not wanted.  One warp per spin, lanes along time (384-byte coalesced reads).  */
int mrphy_rfgr2beff_spin_grads(const mrphy_rfgr2beff_args* a, void* cuda_stream);

/* Hargreaves A/B propagation, replacing beffective.beff2ab (beffective.py:40-104) and its autograd:
 * A (N,nM,3,3), B (N,nM,3) contiguous out; E1, E2 are the per-step relaxation FACTORS as upstream.
 * With `ckpt` non-NULL the forward also stores the 12 entries of [A|B] every K steps
 * (mrphy_beff2ab_ckpt_elems() elements) for mrphy_beff2ab_bwd, which takes dL/dA, dL/dB and writes
 * dL/dBeff (N,nM,nT,3) and, per spin, gP (N,nM,3) = [dL/dE1, dL/dE2, dL/d(2*pi*gamma*dt)] for the caller to
 * reduce onto the broadcast shapes of E1, E2, gamma, dt.  K == 1 never divides by E1/E2 (valid for E = 0). */
typedef struct mrphy_beff2ab_args {
  int32_t dtype, flags;
  int32_t N, nM, nT, K;                               /* K: checkpoint interval (used when ckpt != NULL) */
  const void* Beff; int64_t B_sn, B_sm;               /* (N,nM,nT,3), (nT,3) contiguous */
  mrphy_param E1, E2, gamma, dt;
  void* A; void* B;                                   /* fwd out / bwd in */
  void* ckpt;                                         /* fwd out (optional) / bwd in */
  const void* gA; const void* gB;                     /* bwd in, contiguous like A, B */
  void* gBeff; void* gP;                              /* bwd out, contiguous */
} mrphy_beff2ab_args;
size_t mrphy_beff2ab_ckpt_elems(const mrphy_beff2ab_args* a);
int mrphy_beff2ab(const mrphy_beff2ab_args* a, void* cuda_stream);
int mrphy_beff2ab_bwd(const mrphy_beff2ab_args* a, void* cuda_stream);

/* Rotation axis / angle of a field, replacing beffective.beff2u-phi (beffective.py:14-37) and its autograd:
 * U = beff / max(|beff|, 1e-12) (N,nM,3), Phi = -|beff| * g (N,nM), g = the caller's 2*pi*gamma*dt.
 * adjoint != 0: from gU, gPhi write gbeff (N,nM,3) and, when gg != NULL, the per-spin dL/dg (N,nM). */
typedef struct mrphy_beff2uphi_args {
  int32_t dtype, adjoint;
  int32_t N, nM;
  const void* beff; int64_t b_sn, b_sm;               /* (N,nM,3) inner stride 1 */
  mrphy_param g;
  void* U; void* Phi;                                 /* forward out, contiguous */
  const void* gU; const void* gPhi;                   /* adjoint in, contiguous (either may be NULL = zero) */
  void* gbeff; void* gg;                              /* adjoint out, contiguous */
} mrphy_beff2uphi_args;
int mrphy_beff2uphi(const mrphy_beff2uphi_args* a, void* cuda_stream);

/* Free precession, replacing sims.FreePrec.forward / .backward (sims.py:325-421): rotate about z by
 * -2*pi*df*dur then relax over dur (adjoint != 0: the transposed map applied to dL/dMo).            */
typedef struct mrphy_freeprec_args {
  int32_t dtype, adjoint;
  int32_t N, nM;
  const void* Mi; int64_t Mi_sn, Mi_sm;               /* (N,nM,3) inner stride 1 */
  mrphy_param dur, T1, T2, df;                        /* T1/T2 both NULL = no relaxation; df NULL = no precession */
  void* Mo;                                           /* (N,nM,3) contiguous */
} mrphy_freeprec_args;
int mrphy_freeprec(const mrphy_freeprec_args* a, void* cuda_stream);

/* Waveform re-parametrisation of the design loop (SURVEY 8f-2), replacing the elementwise chains of
 * utils.t-rho-theta2rf / l-rho-theta2rf (utils.py:114-131, 311-330), utils.ts2s (utils.py:293-308) and utils.s2g
 * (utils.py:239-256) and their autograd -- what the optimiser differentiates through on either side of applypulse:
 *   rf[n,:,t,c] = A(rho[n,0,t,c]) * rfmax[n,c] * (cos theta, sin theta),  A = atan(.)*2/pi (rf_kind 1) | sigmoid (rf_kind 2)
 *   s[n,x,t]    = atan(ts[n,x,t])*2/pi * smax[n,x]                        (gr_kind 1 and 3; gr_kind 2 takes s as `ts`)
 *   g[n,x,t]    = dt[n] * sum_{t' <= t} s[n,x,t']                          (gr_kind 1 and 2; gr_kind 3 returns s)
 * ONE launch does both halves (either may be absent: kind 0).  adjoint != 0: from grf, ggr write grho, gtheta, gts
 * (the reversed running sum for the gradient half).  Everything is contiguous in the reference layouts.          */
typedef struct mrphy_reparam_args {
  int32_t dtype, adjoint;
  int32_t N, nT, nC;                    /* nC: trailing coil dimension of rho/theta/rf (1 when absent)            */
  int32_t rf_kind;                      /* 0 none, 1 t-rho (atan), 2 l-rho (sigmoid)                              */
  int32_t gr_kind;                      /* 0 none, 1 ts -> g, 2 s -> g, 3 ts -> s                                 */
  int32_t _pad;
  const void* rho; const void* theta;   /* (N,1,nT,nC)                                                            */
  const void* rfmax; int64_t rfmax_sn, rfmax_sc;   /* element (n,c) at rfmax[n*sn + c*sc] (strides 0 broadcast)    */
  const void* ts;                       /* (N,3,nT)                                                               */
  const void* smax; int64_t smax_sn, smax_sx;      /* element (n,x) at smax[n*sn + x*sx]                           */
  mrphy_param dt;                       /* (N,) s                                                                 */
  void* rf; void* gr;                   /* forward out: (N,2,nT,nC), (N,3,nT)                                     */
  const void* grf; const void* ggr;     /* adjoint in, like rf, gr                                                */
  void* grho; void* gtheta; void* gts;  /* adjoint out, like rho, theta, ts                                       */
} mrphy_reparam_args;
int mrphy_design_waveform(const mrphy_reparam_args* a, void* cuda_stream);

/* Amplitude limits of the design loop (SURVEY 8f-2), replacing utils.rfclamp (utils.py:217-236) and utils.sclamp
 * (utils.py:278-293) and their autograd, one launch each way:
 *   kind 1  rf (N,2,nT,nC):  out = rf * min((rfmax[n,c] - eps) / |rf|, 1),  |rf| over the xy axis
 *   kind 2  s  (N,3,nT):     out = min(max(s, -smax[n,x]), smax[n,x])
 * adjoint != 0: from g = dL/dout write gx = dL/dx -- inside the limit g; kind 1 outside: (lim/|rf|) (g - (g.rf) rf/|rf|^2)
 * (the radial part is cut); kind 2 outside: 0, exactly on the limit g/2 (torch's maximum/minimum tie rule).        */
typedef struct mrphy_clamp_args {
  int32_t dtype, adjoint;
  int32_t kind, N, nT, nC;              /* nC: trailing coil dimension of rf (1 when absent; kind 2: 1)                 */
  const void* x;                        /* rf (N,2,nT,nC) | s (N,3,nT), contiguous                                      */
  const void* lim; int64_t lim_sn, lim_sc;   /* rfmax: element (n,c) at lim[n*sn + c*sc]; smax: (n,x) likewise           */
  double eps;                           /* kind 1 only                                                                  */
  const void* g;                        /* adjoint in, like x                                                           */
  void* out;                            /* forward: clamped x; adjoint: dL/dx                                           */
} mrphy_clamp_args;
int mrphy_clamp_waveform(const mrphy_clamp_args* a, void* cuda_stream);

/* Mask gather of the spin axis (mobjs.SpinArray.extract / .embed, mobjs.py:512-553) as ONE pass over the output:
 *   out[n, j, :] = idx[j] >= 0 ? in[n, idx[j], :] : NaN        j in [0, nOut), `inner` trailing elements per spin
 * extract: idx = row-major positions of the mask's True entries (nOut = nM, nIn = prod(Nd));
 * embed:   idx = the inverse map, -1 outside the mask (nOut = prod(Nd), nIn = nM) -- NaN padding as mobjs.py:525.
 * in (N,nIn,inner) and out (N,nOut,inner) contiguous.                                                             */
typedef struct mrphy_mask_args {
  int32_t dtype, N;
  int32_t fill_zero, _pad;          /* != 0: rows with idx < 0 are 0 instead of NaN (the transposed map of the other direction) */
  int64_t nOut, nIn, inner;
  const int64_t* idx;
  const void* in;
  void* out;
} mrphy_mask_args;
int mrphy_mask_copy(const mrphy_mask_args* a, void* cuda_stream);

/* sizeof() of the argument structs as this library was compiled, for bindings to check their mirror of the layout:
 * which = 0 mrphy_param, 1 mrphy_fused_args, 2 mrphy_beff_args, 3 mrphy_rfgr2beff_args, 4 mrphy_beff2ab_args,
 * 5 mrphy_beff2uphi_args, 6 mrphy_freeprec_args, 7 mrphy_reparam_args, 8 mrphy_mask_args, 9 mrphy_clamp_args;
 * 0 for any other value. */
size_t mrphy_sizeof_args(int which);

/* Number of kernel launches the last forward / backward call on this thread issued. */
int mrphy_last_launch_count(void);

/* Per-kernel timing for bench.py's roofline leg.  With timing enabled, each entry point brackets its
 * MAIN kernel (fused_fwd / fused_bwd / beff_fwd / beff_bwd -- not pack/finalize) with CUDA events on
 * the launching stream; mrphy_last_kernel_ms() synchronises on the stop event and returns the
 * duration in milliseconds of the last such kernel launched by this process (< 0 if none).  Process-
 * wide and not thread-safe: a measurement aid for single-stream benchmarks only.                 */
int mrphy_kernel_timing(int enable);
float mrphy_last_kernel_ms(void);

#ifdef __cplusplus
}
#endif
#endif /* MRPHY_B200_H */
