// lcpb200.cu -- C ABI (include/lcpb200.h), launch planning, host-buffer pipeline.
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>
#include <algorithm>
#include <new>
#include <string>
#include <vector>

#include "../../include/lcpb200.h"
#include "lcp_assemble.cuh"
#include "lcp_launch.h"
#include "lcp_cond_launch.h"
#include "lcp_band_launch.h"
#include "lcp_contacts.cuh"
#include "lcp_joints.cuh"

using namespace lcpb200;
using cnd::CPlan;

static thread_local std::string g_err;
static int fail(const std::string& s) { g_err = s; return 1; }
#define CK(call)                                                                                 \
  do {                                                                                           \
    cudaError_t _e = (call);                                                                     \
    if (_e != cudaSuccess)                                                                       \
      return fail(std::string(#call) + ": " + cudaGetErrorString(_e) + " (" __FILE__ ":" +      \
                  std::to_string(__LINE__) + ")");                                               \
  } while (0)

// Restores the caller's current device when an entry point returns (the library switches to the handle's).
struct DeviceGuard {
  int prev = -1;
  bool armed = false;
  cudaError_t set(int device) {
    cudaError_t e = cudaGetDevice(&prev);
    if (e != cudaSuccess) return e;
    armed = (prev != device);
    return armed ? cudaSetDevice(device) : cudaSuccess;
  }
  ~DeviceGuard() { if (armed) cudaSetDevice(prev); }
};

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  cudaError_t ensure(size_t need) {
    if (need <= bytes) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; bytes = 0;
    cudaError_t e = cudaMalloc(&p, need);
    if (e == cudaSuccess) bytes = need;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
};

struct lcpb200_handle_s {
  int dtype, n, m, e, device;
  int num_sms, smem_optin;
  Plan plan;
  int max_grid;            // resident CTAs (occupancy * SMs) of the dual-form kernels
  CPlan cplan;             // condensed-KKT kernels (lcp_condensed.cuh); cplan.ok == 0: not available
  int cond_grid = 0;       // resident CTAs of the condensed kernels
  static const int NSLOT = 2;   // independent workspace slices (one per pipeline stream)
  void* ws = nullptr;      // dual-form workspace, grown on demand: ws_ctas CTAs x NSLOT slices
  size_t ws_bytes = 0;
  int ws_ctas = 0;
  DevBuf d_flag[NSLOT];    // per-scene "gradients already written" flags of the backward pass
  DevBuf d_ph;             // engine path: p and h of every scene ([B,n] + [B,m])
  bool dual_ok = true;     // false: the dense API is not available for these sizes (engine entry points only)
  bnd::BPlan bplan;        // banded large-scene kernel (lcp_banded.cuh), planned on the first engine call
  int bplan_mode = -1;     // mode the plan was made for
  DevBuf d_bwsd, d_bwsi;   // its per-CTA L2 workspace
  int bws_ctas = 0;
  // host-buffer pipeline state
  cudaStream_t streams[NSLOT] = {nullptr, nullptr};
  DevBuf d_in[7], d_out[6], d_bwd[16];
  long long* prof = nullptr;      // optional per-CTA phase cycle counters [NSLOT*max_grid][PH_COUNT]
  long long* cprof = nullptr;     // same for the condensed kernels [NSLOT*cond_grid][CPH_COUNT]
  DevBuf d_struct;                // [struct_B][cplan.sbytes]: structure of every scene of the last lcpb200_forward
  int struct_B = 0;               // ... and its batch size (0 = nothing saved)
  DevBuf d_R;                     // host pipeline: R of every scene, kept for backward_host
  int retained_B = 0;             // scenes whose inputs/results forward_host left on the device
  bool retained_R = false;        // ... and whether R of those scenes is in d_R
};

static int pad_ld(int cols, int elem_bytes) {
  // leading dimension (elements): >= cols, a multiple of the 16-byte vector, and == 4 (mod 32) in
  // 32-bit words so that 4 consecutive rows tile all 32 banks (lcp_lu.cuh)
  const int wpe = elem_bytes / 4;             // words per element
  int ld = cols;
  while ((ld * wpe) % 32 != 4 || (ld * elem_bytes) % 16 != 0) ++ld;
  return ld;
}

template <typename T>
static int make_plan(lcpb200_handle_s* h) {
  Plan& P = h->plan;
  const int n = h->n, m = h->m, e = h->e;
  constexpr int NB = Blk<T>::NB, VC = VecOf<T>::VC;
  const int w = (int)sizeof(T);
  memset(&P, 0, sizeof(P));
  P.n = n; P.m = m; P.e = e;
  P.mp = ((m + NB - 1) / NB) * NB;
  const int mp = P.mp;
  P.nt = (mp >= 96 || n >= 96) ? 512 : (mp >= 64 ? 256 : 128);
  Vecs<T> vv;
  P.lds = pad_ld(NB, w);
  const long long vec_elems = vv.carve(nullptr, n, mp, e, P.nt, NB, P.lds);
  long long budget = (long long)h->smem_optin - 1024 - vec_elems * w;   // bytes
  if (budget < 0) return fail("problem too large: the shared-memory vectors alone exceed the per-CTA limit");
  auto al4 = [](long long x) { return (x + 3) & ~3LL; };
  long long off = 0;
  // ---- residency of T
  const int ldfull = pad_ld(mp, w);
  if ((long long)mp * ldfull * w <= budget) {
    P.mode = 0; P.m1 = mp; P.ldT = ldfull; P.ldL = 0;
    P.off_T = (int)off; off += al4((long long)mp * ldfull);
  } else {
    const int m1 = (((mp / 2) + NB - 1) / NB) * NB, n2 = mp - m1;
    const int ldl = pad_ld(m1, w);
    const int tiles = ((n2 + 15) / 16) * ((n2 + 16 * VC - 1) / (16 * VC));
    const long long need = ((long long)m1 * ldfull + (long long)n2 * ldl) * w;
    if (n2 > 0 && n2 <= m1 && need <= budget && tiles <= P.nt / 32) {
      P.mode = 1; P.m1 = m1; P.ldT = ldfull; P.ldL = ldl;
      P.off_T = (int)off; off += al4((long long)m1 * ldfull);
      P.off_L = (int)off; off += al4((long long)n2 * ldl);
    } else {
      P.mode = 2; P.m1 = mp; P.ldT = ((mp + VC - 1) / VC) * VC; P.ldL = 0;
    }
  }
  P.stage_ld = 0;
  P.prefetch = getenv("LCPB200_NO_PREFETCH") ? 0 : 1;
  if (P.mode != 2) {
    const int lds = pad_ld(n, w);
    if ((long long)m * lds <= (long long)P.m1 * P.ldT) P.stage_ld = lds;
  }
  budget -= off * w;
  P.ldG = n;
  P.ldQi = ((n + VC - 1) / VC) * VC;
  const long long Gb = al4((long long)m * P.ldG), Qb = al4((long long)n * P.ldQi);
  if (Gb * w <= budget) { P.G_smem = 1; P.off_G = (int)off; off += Gb; budget -= Gb * w; }
  if (Qb * w <= budget) { P.Qi_smem = 1; P.off_Qi = (int)off; off += Qb; budget -= Qb * w; }
  P.off_vec = (int)off;
  P.smem_bytes = (int)((off + vec_elems) * w);
  long long ws = 0;
  P.w_Qi = ws; ws += Qb;
  P.w_R = ws; ws += al4((long long)m * m);
  P.w_T = ws; ws += (P.mode == 2) ? al4((long long)mp * P.ldT) : 0;
  P.w_U12 = ws; ws += (P.mode == 1) ? al4((long long)P.m1 * (mp - P.m1)) : 0;
  P.w_X = ws; ws += al4((long long)n * m);
  P.w_XA = ws; ws += al4((long long)n * e);
  P.w_S11 = ws; ws += al4((long long)e * e);
  P.w_V = ws; ws += al4((long long)m * e);
  P.w_W = ws; ws += al4((long long)e * m);
  P.w_Fell = ws; ws += al4((long long)m * 8);          // F in ELL form: 4 values + 4 column indices per row
  P.w_Gell = ws; ws += al4((long long)16 * m + (long long)64 * n);   // G in row-ELL (8/row) and column-ELL (32/column) form
  P.ws_per_cta = ws;
  return 0;
}

template <typename T>
static int configure_kernels(lcpb200_handle_s* h) {
  const Plan& P = h->plan;
  const int dyn_max = h->smem_optin - 1024;
  int occ = 0;
  cudaError_t ce = P.mode == 0 ? configure_t<T, 0>(P.nt, P.smem_bytes, dyn_max, &occ)
                 : P.mode == 1 ? configure_t<T, 1>(P.nt, P.smem_bytes, dyn_max, &occ)
                               : configure_t<T, 2>(P.nt, P.smem_bytes, dyn_max, &occ);
  if (ce != cudaSuccess) return fail(std::string("kernel configuration: ") + cudaGetErrorString(ce));
  if (occ < 1) return fail("kernel cannot be resident with the planned shared memory");
  occ = std::min(occ, 8);
  h->max_grid = occ * h->num_sms;
  h->plan.grid = h->max_grid;
  return 0;
}


// ------------------------------------------------------------------ condensed-KKT plan (lcp_condensed.cuh)
#define LCPB200_NS_DISPATCH(NSV, CALL)                                  \
  ((NSV) == 2 ? CALL(2) : (NSV) == 3 ? CALL(3) : (NSV) == 4 ? CALL(4) : (NSV) == 6 ? CALL(6) : CALL(8))

template <typename T>
static int make_cplan(lcpb200_handle_s* h) {
  CPlan& C = h->cplan;
  memset(&C, 0, sizeof(C));
  if (getenv("LCPB200_NO_CONDENSED")) return 0;
  const int n = h->n, m = h->m, e = h->e, N = n + e;
  if (N > 128 || n > 255 || m > 4 * cnd::NT) return 0;
  static const int sizes[5] = {2, 3, 4, 6, 8};
  int NS = 8;
  for (int k = 4; k >= 0; --k) if (16 * sizes[k] >= N) NS = sizes[k];
  C.n = n; C.m = m; C.e = e; C.N = N; C.NS = NS; C.NP = 16 * NS;
  C.pcap = (m + 7) & ~7;
  C.flags = getenv("LCPB200_COND_FLAGS") ? atoi(getenv("LCPB200_COND_FLAGS")) : 3;
  const int dyn_max = h->smem_optin - 1024;
  const int target = NS <= 6 ? 2 : 1;                              // CTAs per SM the kernels are bounded for
  // shared memory per SM: 228 KB, 1 KB reserved per resident CTA
  const int per_cta_target = (228 * 1024) / target - 1024 - 64;
  int best = -1;
  for (int want = target; want >= 1 && best < 0; --want) {
    const int lim = std::min(dyn_max, want == target ? per_cta_target : (228 * 1024) / want - 1024 - 64);
    for (int mult = cnd::CSMAX; mult >= 1; --mult) {            // capacity of W / Fd: mult * pcap elements
      C.wcap = mult * C.pcap;
      const size_t bytes = cnd::carve_plan(C, (int)sizeof(T));
      if ((long long)bytes <= lim) { best = (int)bytes; break; }
      if (mult <= 4) break;                                     // the engine's fd = 2 blocks need 4
    }
  }
  if (best < 0) return 0;
  C.smem_bytes = best;
  int occ = 0;
#define CALL_CFG(NSV) cnd::configure_cond_t<T, NSV>(C.smem_bytes, dyn_max, &occ)
  const cudaError_t ce = LCPB200_NS_DISPATCH(NS, CALL_CFG);
#undef CALL_CFG
  if (ce != cudaSuccess) return fail(std::string("condensed kernel configuration: ") + cudaGetErrorString(ce));
  if (occ < 1) return 0;
  C.ctas_per_sm = occ;
  h->cond_grid = occ * h->num_sms;
  C.ok = 1;
  return 0;
}

extern "C" int lcpb200_version(void) { return LCPB200_VERSION; }
extern "C" const char* lcpb200_last_error_string(void) { return g_err.c_str(); }

extern "C" int lcpb200_create(int dtype, int n, int m, int e, int device, lcpb200_handle_t* out) {
  if (!out) return fail("out == NULL");
  *out = nullptr;
  if (dtype != LCPB200_F32 && dtype != LCPB200_F64) return fail("dtype must be LCPB200_F32 or LCPB200_F64");
  if (n <= 0 || m <= 0 || e < 0) return fail("need n > 0, m > 0, e >= 0");
  DeviceGuard dg_;
  CK(dg_.set(device));
  lcpb200_handle_s* h = new (std::nothrow) lcpb200_handle_s();
  if (!h) return fail("out of host memory");
  h->dtype = dtype; h->n = n; h->m = m; h->e = e; h->device = device;
  cudaError_t ce;
  if ((ce = cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device)) != cudaSuccess ||
      (ce = cudaDeviceGetAttribute(&h->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device)) != cudaSuccess) {
    delete h;
    return fail(std::string("cudaDeviceGetAttribute: ") + cudaGetErrorString(ce));
  }
  int rc = (dtype == LCPB200_F32) ? make_plan<float>(h) : make_plan<double>(h);
  if (!rc) rc = (dtype == LCPB200_F32) ? configure_kernels<float>(h) : configure_kernels<double>(h);
  if (rc) {
    // too large for the dense API: the handle still serves the engine entry points (banded kernel, fp64)
    if (dtype != LCPB200_F64 || n % 3 != 0 || e > bnd::BD) { delete h; return rc; }
    h->dual_ok = false;
    h->max_grid = h->num_sms;
    rc = 0;
  }
  if (!rc) rc = (dtype == LCPB200_F32) ? make_cplan<float>(h) : make_cplan<double>(h);
  if (rc) { delete h; return rc; }
  memset(&h->bplan, 0, sizeof(h->bplan));
  *out = h;
  return 0;
}

// The dual-form kernels keep U12 / ELL copies / small blocks in a per-CTA L2 workspace. It is sized
// for the CTAs a call can actually use (min(B, resident CTAs)) and grown on demand, so that a
// batch-of-one engine call on a large scene does not allocate 148 CTAs' worth.
static int ensure_ws(lcpb200_handle_s* h, int B) {
  const int ctas = std::min(B, h->max_grid);
  if (ctas <= h->ws_ctas) return 0;
  const size_t esz = h->dtype == LCPB200_F32 ? 4 : 8;
  const size_t need = (size_t)h->plan.ws_per_cta * esz * (size_t)ctas * lcpb200_handle_s::NSLOT;
  if (h->ws) { CK(cudaDeviceSynchronize()); CK(cudaFree(h->ws)); h->ws = nullptr; h->ws_bytes = 0; h->ws_ctas = 0; }
  CK(cudaMalloc(&h->ws, need));
  h->ws_bytes = need;
  h->ws_ctas = ctas;
  return 0;
}

extern "C" int lcpb200_destroy(lcpb200_handle_t h) {
  if (!h) return 0;
  DeviceGuard dg_;
  dg_.set(h->device);
  if (h->ws) cudaFree(h->ws);
  h->d_struct.release();
  if (h->prof) cudaFree(h->prof);
  if (h->cprof) cudaFree(h->cprof);
  for (auto& s : h->streams) if (s) cudaStreamDestroy(s);
  for (auto& b : h->d_in) b.release();
  for (auto& b : h->d_out) b.release();
  for (auto& b : h->d_bwd) b.release();
  for (auto& b : h->d_flag) b.release();
  h->d_ph.release();
  h->d_bwsd.release();
  h->d_bwsi.release();
  h->d_R.release();
  delete h;
  return 0;
}

extern "C" size_t lcpb200_workspace_bytes(lcpb200_handle_t h) { return h ? h->ws_bytes : 0; }

extern "C" int lcpb200_describe(lcpb200_handle_t h, char* buf, size_t len) {
  if (!h || !buf) return fail("null argument");
  const Plan& P = h->plan;
  static const char* modes[3] = {"smem", "smem-split(U12 in L2)", "L2"};
  const CPlan& C = h->cplan;
  char cbuf[256];
  if (C.ok)
    snprintf(cbuf, sizeof(cbuf), "condensed KKT: N=%d(pad %d) fp64 LU in registers, threads=%d smem=%dB CTAs/SM=%d grid<=%d "
             "(forward%s; unstructured scenes fall back to dual)", C.N, C.NP, cnd::NT, C.smem_bytes, C.ctas_per_sm,
             h->cond_grid, h->dtype == LCPB200_F32 ? "+backward" : "");
  else
    snprintf(cbuf, sizeof(cbuf), "condensed KKT: n/a");
  snprintf(buf, len,
           "dtype=%s n=%d m=%d(pad %d) e=%d | %s | dual: threads=%d smem=%dB T:%s m1=%d ldT=%d ldL=%d G:%s Qinv:%s grid<=%d "
           "ws/CTA=%lldB sms=%d",
           h->dtype == LCPB200_F32 ? "f32" : "f64", P.n, P.m, P.mp, P.e, cbuf, P.nt, P.smem_bytes, modes[P.mode], P.m1,
           P.ldT, P.ldL, P.G_smem ? "smem" : "L2", P.Qi_smem ? "smem" : "L2", h->max_grid,
           (long long)(P.ws_per_cta * (h->dtype == LCPB200_F32 ? 4 : 8)), h->num_sms);
  return 0;
}

template <typename T>
static int launch_forward(lcpb200_handle_s* h, int slot, int B, const void* Q, const void* p, const void* G,
                          const void* hv, const void* A, const void* b, const void* F, double eps,
                          int not_improved_lim, int max_iter, void* zhat, void* nu, void* lam, void* slack,
                          int32_t* status, int32_t* iters, void* resid, void* Rsave, cudaStream_t st,
                          unsigned char* ssave = nullptr) {
  const bool cond = h->cplan.ok != 0;
  if (cond) {
    // structured scenes: condensed-KKT kernel; it flags the others (status = -100) for the dual-form kernel below
    cnd::CFwdArgs<T> c;
    c.P = h->cplan;
    c.B = B;
    c.Q = (const T*)Q; c.p = (const T*)p; c.G = (const T*)G; c.h = (const T*)hv;
    c.A = (const T*)A; c.b = (const T*)b; c.F = (const T*)F;
    c.zhat = (T*)zhat; c.nu = (T*)nu; c.lam = (T*)lam; c.slack = (T*)slack; c.resid = (T*)resid;
    c.status = status; c.iters = iters;
    c.eps = (T)eps; c.not_improved_lim = not_improved_lim; c.max_iter = max_iter;
    memset(&c.soa, 0, sizeof(c.soa));
    c.ssave = ssave;
    c.prof = h->cprof ? h->cprof + (size_t)slot * h->cond_grid * cnd::CPH_COUNT : nullptr;
    const int cgrid = std::min(B, h->cond_grid);
#define CALL_FWD(NSV) cnd::launch_cond_forward_t<T, NSV>(c, cgrid, st)
    const cudaError_t ce = LCPB200_NS_DISPATCH(h->cplan.NS, CALL_FWD);
#undef CALL_FWD
    CK(ce);
    Rsave = nullptr;          // the condensed kernel does not form R; the dual-form backward recomputes it
  }
  if (int rc = ensure_ws(h, B)) return rc;
  FwdArgs<T> a;
  a.P = h->plan;
  a.B = B;
  a.Q = (const T*)Q; a.p = (const T*)p; a.G = (const T*)G; a.h = (const T*)hv;
  a.A = (const T*)A; a.b = (const T*)b; a.F = (const T*)F;
  a.zhat = (T*)zhat; a.nu = (T*)nu; a.lam = (T*)lam; a.slack = (T*)slack; a.resid = (T*)resid;
  a.status = status; a.iters = iters;
  a.eps = (T)eps; a.not_improved_lim = not_improved_lim; a.max_iter = max_iter;
  a.Rsave = (T*)Rsave;
  a.fallback_only = cond ? 1 : 0;
  a.ws = (T*)h->ws + (size_t)slot * h->plan.ws_per_cta * h->ws_ctas;
  a.prof = h->prof ? h->prof + (size_t)slot * h->max_grid * PH_COUNT : nullptr;
  const int grid = std::min(B, h->ws_ctas);
  const int mode = h->plan.mode;
  const cudaError_t le = mode == 0   ? launch_forward_t<T, 0>(a, grid, st)
                         : mode == 1 ? launch_forward_t<T, 1>(a, grid, st)
                                     : launch_forward_t<T, 2>(a, grid, st);
  CK(le);
  return 0;
}

template <typename T>
static int launch_backward(lcpb200_handle_s* h, int slot, int B, const void* Q, const void* G, const void* A,
                           const void* F, const void* zhat, const void* nu, const void* lam, const void* slack,
                           const void* g, void* dQ, void* dp, void* dG, void* dh, void* dA, void* db, void* dF,
                           const void* Rsave, unsigned flags, cudaStream_t st, const unsigned char* sload = nullptr) {
  // fp32: condensed-KKT backward first, the dual form only for the scenes it flags as unstructured.
  // fp64: the dual form first -- at the fp64 round-off floor (lambda, s ~ 1e-16, d = lambda/s spanning
  // 1e+-16) the condensed matrix loses dx (DESIGN.md "Parity") -- and the condensed kernel only as a rescue
  // for scenes on which the dual LU (pivoting restricted to its diagonal blocks) broke down (non-finite dx).
  const bool have_cond = h->cplan.ok != 0;
  const bool cond_first = have_cond && sizeof(T) == 4 && !getenv("LCPB200_DUAL_BACKWARD");
  int* flagbuf = nullptr;
  if (have_cond) {
    CK(h->d_flag[slot].ensure(sizeof(int) * (size_t)B));
    flagbuf = (int*)h->d_flag[slot].p;
  }
  cnd::CBwdArgs<T> c;
  if (have_cond) {
    c.P = h->cplan;
    c.B = B;
    c.Q = (const T*)Q; c.G = (const T*)G; c.A = (const T*)A; c.F = (const T*)F;
    c.zhat = (const T*)zhat; c.nu = (const T*)nu; c.lam = (const T*)lam; c.slack = (const T*)slack;
    c.g = (const T*)g;
    c.dQ = (T*)dQ; c.dp = (T*)dp; c.dG = (T*)dG; c.dh = (T*)dh; c.dA = (T*)dA; c.db = (T*)db; c.dF = (T*)dF;
    c.done = cond_first ? flagbuf : nullptr;
    c.only = cond_first ? nullptr : flagbuf;
    c.flags = flags;
    c.sload = sload;
    memset(&c.soa, 0, sizeof(c.soa));
    c.dmass = c.dinertia = c.dv = c.dfext = c.dnormal = c.dp1 = c.dp2 = c.dmu = c.drest = nullptr;
    c.prof = h->cprof ? h->cprof + (size_t)slot * h->cond_grid * cnd::CPH_COUNT : nullptr;
  }
  const int cgrid = std::min(B, std::max(h->cond_grid, 1));
  if (cond_first) {
#define CALL_BWD(NSV) cnd::launch_cond_backward_t<T, NSV>(c, cgrid, st)
    const cudaError_t ce = LCPB200_NS_DISPATCH(h->cplan.NS, CALL_BWD);
#undef CALL_BWD
    CK(ce);
  }
  if (int rc = ensure_ws(h, B)) return rc;
  BwdArgs<T> a;
  a.P = h->plan;
  a.B = B;
  a.Q = (const T*)Q; a.G = (const T*)G; a.A = (const T*)A; a.F = (const T*)F;
  a.zhat = (const T*)zhat; a.nu = (const T*)nu; a.lam = (const T*)lam; a.slack = (const T*)slack;
  a.g = (const T*)g;
  a.dQ = (T*)dQ; a.dp = (T*)dp; a.dG = (T*)dG; a.dh = (T*)dh; a.dA = (T*)dA; a.db = (T*)db; a.dF = (T*)dF;
  a.flags = flags;
  a.Rsave = have_cond ? nullptr : (const T*)Rsave;    // R is only formed when the forward ran on the dual form
  a.skip = cond_first ? flagbuf : nullptr;
  a.bad = (have_cond && !cond_first) ? flagbuf : nullptr;
  a.ws = (T*)h->ws + (size_t)slot * h->plan.ws_per_cta * h->ws_ctas;
  a.prof = h->prof ? h->prof + (size_t)slot * h->max_grid * PH_COUNT : nullptr;
  const int grid = std::min(B, h->ws_ctas);
  const int mode = h->plan.mode;
  const cudaError_t le = mode == 0   ? launch_backward_t<T, 0>(a, grid, st)
                         : mode == 1 ? launch_backward_t<T, 1>(a, grid, st)
                                     : launch_backward_t<T, 2>(a, grid, st);
  CK(le);
  if (have_cond && !cond_first) {
#define CALL_BWD(NSV) cnd::launch_cond_backward_t<T, NSV>(c, cgrid, st)
    const cudaError_t ce = LCPB200_NS_DISPATCH(h->cplan.NS, CALL_BWD);
#undef CALL_BWD
    CK(ce);
  }
  return 0;
}

static int check_fwd_args(lcpb200_handle_t h, int B, const void* Q, const void* p, const void* G, const void* hv,
                          const void* A, const void* b, const void* F, const void* zhat, const void* nu,
                          const void* lam, const void* slack, const void* status, const void* iters,
                          int max_iter) {
  if (!h) return fail("null handle");
  if (B < 0) return fail("B < 0");
  if (!Q || !p || !G || !hv || !F) return fail("Q, p, G, h, F must be non-NULL");
  if (h->e > 0 && (!A || !b)) return fail("handle was created with e > 0 but A or b is NULL");
  if (!zhat || !lam || !slack || !status || !iters) return fail("zhat, lam, slack, status, iters must be non-NULL");
  if (h->e > 0 && !nu) return fail("nu must be non-NULL when e > 0");
  if (max_iter < 0) return fail("max_iter < 0");
  return 0;
}

extern "C" int lcpb200_forward(lcpb200_handle_t h, int B, const void* Q, const void* p, const void* G,
                               const void* hv, const void* A, const void* b, const void* F, double eps,
                               int not_improved_lim, int max_iter, void* zhat, void* nu, void* lam, void* slack,
                               int32_t* status, int32_t* iters, void* resid, void* Rsave, void* stream) {
  if (int rc = check_fwd_args(h, B, Q, p, G, hv, A, b, F, zhat, nu, lam, slack, status, iters, max_iter)) return rc;
  if (!h->dual_ok) return fail("this handle serves the engine entry points only (problem too large for the dense API)");
  if (B == 0) return 0;
  DeviceGuard dg_;
  CK(dg_.set(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  // the structure of every scene is kept for a backward of the same inputs (LCPB200_BWD_REUSE_STRUCTURE)
  unsigned char* ssave = nullptr;
  h->struct_B = 0;
  if (h->cplan.ok) {
    if ((size_t)B * h->cplan.sbytes > h->d_struct.bytes) CK(cudaDeviceSynchronize());    // (an earlier launch may still read it)
    CK(h->d_struct.ensure((size_t)B * h->cplan.sbytes));
    ssave = (unsigned char*)h->d_struct.p;
  }
  const int rc = h->dtype == LCPB200_F32
             ? launch_forward<float>(h, 0, B, Q, p, G, hv, A, b, F, eps, not_improved_lim, max_iter, zhat, nu, lam,
                                     slack, status, iters, resid, Rsave, st, ssave)
             : launch_forward<double>(h, 0, B, Q, p, G, hv, A, b, F, eps, not_improved_lim, max_iter, zhat, nu, lam,
                                      slack, status, iters, resid, Rsave, st, ssave);
  if (rc == 0 && ssave) h->struct_B = B;
  return rc;
}

extern "C" int lcpb200_backward(lcpb200_handle_t h, int B, const void* Q, const void* G, const void* A,
                                const void* F, const void* zhat, const void* nu, const void* lam,
                                const void* slack, const void* g, void* dQ, void* dp, void* dG, void* dh, void* dA,
                                void* db, void* dF, const void* Rsave, unsigned flags, void* stream) {
  if (!h) return fail("null handle");
  if (!h->dual_ok) return fail("this handle serves the engine entry points only (problem too large for the dense API)");
  if (B < 0) return fail("B < 0");
  if (!Q || !G || !F || !zhat || !lam || !slack || !g) return fail("Q, G, F, zhat, lam, slack, dl_dzhat must be non-NULL");
  if (h->e > 0 && (!A || !nu)) return fail("A and nu must be non-NULL when e > 0");
  if (flags & ~(LCPB200_BWD_EXACT_ADJOINT | LCPB200_BWD_REUSE_STRUCTURE))
    return fail("flags: LCPB200_BWD_EXACT_ADJOINT | LCPB200_BWD_REUSE_STRUCTURE are the defined bits");
  if (B == 0) return 0;
  DeviceGuard dg_;
  CK(dg_.set(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  // LCPB200_BWD_REUSE_STRUCTURE: the caller states that (Q, G, A, F) are the inputs of the last lcpb200_forward on
  // this handle; ignored when nothing (or another batch size) was saved
  const unsigned char* sload = ((flags & LCPB200_BWD_REUSE_STRUCTURE) && h->cplan.ok && h->struct_B == B)
                                   ? (const unsigned char*)h->d_struct.p : nullptr;
  const unsigned kf = flags & LCPB200_BWD_EXACT_ADJOINT;
  return h->dtype == LCPB200_F32
             ? launch_backward<float>(h, 0, B, Q, G, A, F, zhat, nu, lam, slack, g, dQ, dp, dG, dh, dA, db, dF, Rsave, kf, st, sload)
             : launch_backward<double>(h, 0, B, Q, G, A, F, zhat, nu, lam, slack, g, dQ, dp, dG, dh, dA, db, dF, Rsave, kf, st, sload);
}

extern "C" int lcpb200_profile(lcpb200_handle_t h, int enable, long long* out) {
  // Development aid: per-phase SM cycle counters (thread 0 of every CTA), summed over CTAs.
  // enable = 1 allocates + zeroes the counters, 0 frees them; `out` receives 24 values: the 14
  // dual-form phases (see the header) followed by the 10 condensed-kernel phases.
  if (!h) return fail("null handle");
  DeviceGuard dg_;
  CK(dg_.set(h->device));
  const size_t cnt = (size_t)lcpb200_handle_s::NSLOT * h->max_grid * PH_COUNT;
  const size_t ccnt = (size_t)lcpb200_handle_s::NSLOT * std::max(h->cond_grid, h->num_sms) * cnd::CPH_COUNT;
  if (out) {
    for (int i = 0; i < PH_COUNT + cnd::CPH_COUNT; ++i) out[i] = 0;
    if (h->prof) {
      std::vector<long long> tmp(cnt);
      CK(cudaMemcpy(tmp.data(), h->prof, cnt * sizeof(long long), cudaMemcpyDeviceToHost));
      for (size_t i = 0; i < cnt; ++i) out[i % PH_COUNT] += tmp[i];
    }
    if (h->cprof) {
      std::vector<long long> tmp(ccnt);
      CK(cudaMemcpy(tmp.data(), h->cprof, ccnt * sizeof(long long), cudaMemcpyDeviceToHost));
      for (size_t i = 0; i < ccnt; ++i) out[PH_COUNT + i % cnd::CPH_COUNT] += tmp[i];
    }
  }
  if (enable && !h->prof) CK(cudaMalloc(&h->prof, cnt * sizeof(long long)));
  if (enable && !h->cprof) CK(cudaMalloc(&h->cprof, ccnt * sizeof(long long)));
  if (enable) { CK(cudaMemset(h->prof, 0, cnt * sizeof(long long))); CK(cudaMemset(h->cprof, 0, ccnt * sizeof(long long))); }
  if (!enable && h->prof) { cudaFree(h->prof); h->prof = nullptr; }
  if (!enable && h->cprof) { cudaFree(h->cprof); h->cprof = nullptr; }
  return 0;
}

// ------------------------------------------------------------------ host-buffer pipeline
// Chunks of scenes are copied in on one of two streams, solved on the same stream and copied
// back, so the H2D copy of chunk k+1 overlaps the solve of chunk k (each stream has its own
// workspace slice).
static int ensure_streams(lcpb200_handle_s* h) {
  for (auto& s : h->streams)
    if (!s) CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  return 0;
}

static int chunk_scenes(const lcpb200_handle_s* h, int B) {
  // at least two waves of CTAs per chunk, at most 8 chunks
  int c = std::max(2 * h->max_grid, (B + 7) / 8);
  return std::max(1, std::min(c, B));
}

extern "C" int lcpb200_forward_host(lcpb200_handle_t h, int B, const void* Q, const void* p, const void* G,
                                    const void* hv, const void* A, const void* b, const void* F, double eps,
                                    int not_improved_lim, int max_iter, void* zhat, void* nu, void* lam,
                                    void* slack, int32_t* status, int32_t* iters, void* resid) {
  if (int rc = check_fwd_args(h, B, Q, p, G, hv, A, b, F, zhat, nu, lam, slack, status, iters, max_iter)) return rc;
  if (!h->dual_ok) return fail("this handle serves the engine entry points only (problem too large for the dense API)");
  if (B == 0) return 0;
  DeviceGuard dg_;
  CK(dg_.set(h->device));
  if (int rc = ensure_streams(h)) return rc;
  const size_t w = h->dtype == LCPB200_F32 ? 4 : 8;
  const size_t n = h->n, m = h->m, e = h->e;
  const size_t in_sz[7] = {n * n * w, n * w, m * n * w, m * w, e * n * w, e * w, m * m * w};
  const void* in_src[7] = {Q, p, G, hv, A, b, F};
  const size_t out_sz[6] = {n * w, e * w, m * w, m * w, 4, 4};
  void* out_dst[6] = {zhat, nu, lam, slack, status, iters};
  for (int i = 0; i < 7; ++i) if (in_sz[i]) CK(h->d_in[i].ensure(in_sz[i] * B));
  for (int i = 0; i < 6; ++i) if (out_sz[i]) CK(h->d_out[i].ensure(out_sz[i] * B));
  DevBuf& d_resid = h->d_bwd[15];
  if (resid) CK(d_resid.ensure(w * B));
  h->retained_B = 0;
  // keep R for backward_host (<= 8 GiB) -- only the dual-form forward produces it
  const bool keepR = !h->cplan.ok && (m * m * w * (size_t)B) <= ((size_t)8 << 30);
  if (keepR) CK(h->d_R.ensure(m * m * w * (size_t)B));
  const int C = chunk_scenes(h, B);
  int k = 0;
  for (int s0 = 0; s0 < B; s0 += C, ++k) {
    const int cb = std::min(C, B - s0);
    const int slot = k % lcpb200_handle_s::NSLOT;
    cudaStream_t st = h->streams[slot];
    for (int i = 0; i < 7; ++i)
      if (in_sz[i] && in_src[i])
        CK(cudaMemcpyAsync((char*)h->d_in[i].p + in_sz[i] * s0, (const char*)in_src[i] + in_sz[i] * s0,
                           in_sz[i] * cb, cudaMemcpyHostToDevice, st));
    auto at = [&](DevBuf& bf, size_t per) -> void* { return per ? (char*)bf.p + per * s0 : nullptr; };
    int rc = h->dtype == LCPB200_F32
                 ? launch_forward<float>(h, slot, cb, at(h->d_in[0], in_sz[0]), at(h->d_in[1], in_sz[1]),
                                         at(h->d_in[2], in_sz[2]), at(h->d_in[3], in_sz[3]), at(h->d_in[4], in_sz[4]),
                                         at(h->d_in[5], in_sz[5]), at(h->d_in[6], in_sz[6]), eps, not_improved_lim,
                                         max_iter, at(h->d_out[0], out_sz[0]), at(h->d_out[1], out_sz[1]),
                                         at(h->d_out[2], out_sz[2]), at(h->d_out[3], out_sz[3]),
                                         (int32_t*)at(h->d_out[4], 4), (int32_t*)at(h->d_out[5], 4),
                                         resid ? (char*)d_resid.p + w * s0 : nullptr,
                                         keepR ? (char*)h->d_R.p + m * m * w * s0 : nullptr, st)
                 : launch_forward<double>(h, slot, cb, at(h->d_in[0], in_sz[0]), at(h->d_in[1], in_sz[1]),
                                          at(h->d_in[2], in_sz[2]), at(h->d_in[3], in_sz[3]), at(h->d_in[4], in_sz[4]),
                                          at(h->d_in[5], in_sz[5]), at(h->d_in[6], in_sz[6]), eps, not_improved_lim,
                                          max_iter, at(h->d_out[0], out_sz[0]), at(h->d_out[1], out_sz[1]),
                                          at(h->d_out[2], out_sz[2]), at(h->d_out[3], out_sz[3]),
                                          (int32_t*)at(h->d_out[4], 4), (int32_t*)at(h->d_out[5], 4),
                                          resid ? (char*)d_resid.p + w * s0 : nullptr,
                                          keepR ? (char*)h->d_R.p + m * m * w * s0 : nullptr, st);
    if (rc) return rc;
    for (int i = 0; i < 6; ++i)
      if (out_sz[i] && out_dst[i])
        CK(cudaMemcpyAsync((char*)out_dst[i] + out_sz[i] * s0, (char*)h->d_out[i].p + out_sz[i] * s0,
                           out_sz[i] * cb, cudaMemcpyDeviceToHost, st));
    if (resid)
      CK(cudaMemcpyAsync((char*)resid + w * s0, (char*)d_resid.p + w * s0, w * cb, cudaMemcpyDeviceToHost, st));
  }
  for (auto& s : h->streams) CK(cudaStreamSynchronize(s));
  h->retained_B = B;
  h->retained_R = keepR;
  return 0;
}

extern "C" int lcpb200_backward_host(lcpb200_handle_t h, int B, const void* Q, const void* G, const void* A,
                                     const void* F, const void* zhat, const void* nu, const void* lam,
                                     const void* slack, const void* g, void* dQ, void* dp, void* dG, void* dh,
                                     void* dA, void* db, void* dF, unsigned flags) {
  if (!h) return fail("null handle");
  if (!h->dual_ok) return fail("this handle serves the engine entry points only (problem too large for the dense API)");
  if (B < 0) return fail("B < 0");
  // Q == NULL: reuse the device copies (inputs, results and R) that the last forward_host on this
  // handle left behind -- the save_for_backward of lcp.py:34 without a second upload.
  const bool retained = (Q == nullptr);
  if (retained) {
    if (h->retained_B != B || B == 0) return fail("backward_host: no retained forward state for this batch");
    if (!g) return fail("dl_dzhat must be non-NULL");
  } else {
    if (!G || !F || !zhat || !lam || !slack || !g) return fail("Q, G, F, zhat, lam, slack, dl_dzhat must be non-NULL");
    if (h->e > 0 && (!A || !nu)) return fail("A and nu must be non-NULL when e > 0");
  }
  if (flags != LCPB200_BWD_BUG_COMPATIBLE && flags != LCPB200_BWD_EXACT_ADJOINT)
    return fail("flags must be LCPB200_BWD_BUG_COMPATIBLE or LCPB200_BWD_EXACT_ADJOINT");
  if (B == 0) return 0;
  DeviceGuard dg_;
  CK(dg_.set(h->device));
  if (int rc = ensure_streams(h)) return rc;
  const size_t w = h->dtype == LCPB200_F32 ? 4 : 8;
  const size_t n = h->n, m = h->m, e = h->e;
  // inputs: Q G A F zhat nu lam slack g ; outputs: dQ dp dG dh dA db dF
  const size_t in_sz[9] = {n * n * w, m * n * w, e * n * w, m * m * w, n * w, e * w, m * w, m * w, n * w};
  const void* in_src[9] = {Q, G, A, F, zhat, nu, lam, slack, g};
  // Q, G, A, F may already be resident from forward_host (same buffers d_in[0,2,4,6]); we re-copy for safety.
  // retained: zhat/nu/lam/slack live in the forward's result buffers d_out[0..3]
  DevBuf* in_buf[9] = {&h->d_in[0], &h->d_in[2], &h->d_in[4], &h->d_in[6],
                       retained ? &h->d_out[0] : &h->d_bwd[0], retained ? &h->d_out[1] : &h->d_bwd[1],
                       retained ? &h->d_out[2] : &h->d_bwd[2], retained ? &h->d_out[3] : &h->d_bwd[3], &h->d_bwd[4]};
  const bool resident[9] = {retained, retained, retained, retained, retained, retained, retained, retained, false};
  const size_t out_sz[7] = {n * n * w, n * w, m * n * w, m * w, e * n * w, e * w, m * m * w};
  void* out_dst[7] = {dQ, dp, dG, dh, dA, db, dF};
  DevBuf* out_buf[7] = {&h->d_bwd[5], &h->d_bwd[6], &h->d_bwd[7], &h->d_bwd[8], &h->d_bwd[9], &h->d_bwd[10],
                        &h->d_bwd[11]};
  if (!retained) h->retained_B = 0;       // the input buffers are about to be overwritten
  for (int i = 0; i < 9; ++i) if (in_sz[i] && (in_src[i] || resident[i])) CK(in_buf[i]->ensure(in_sz[i] * B));
  for (int i = 0; i < 7; ++i) if (out_sz[i] && out_dst[i]) CK(out_buf[i]->ensure(out_sz[i] * B));
  const int C = chunk_scenes(h, B);
  int k = 0;
  for (int s0 = 0; s0 < B; s0 += C, ++k) {
    const int cb = std::min(C, B - s0);
    const int slot = k % lcpb200_handle_s::NSLOT;
    cudaStream_t st = h->streams[slot];
    for (int i = 0; i < 9; ++i)
      if (in_sz[i] && in_src[i] && !resident[i])
        CK(cudaMemcpyAsync((char*)in_buf[i]->p + in_sz[i] * s0, (const char*)in_src[i] + in_sz[i] * s0,
                           in_sz[i] * cb, cudaMemcpyHostToDevice, st));
    auto ai = [&](int i) -> void* {
      return (in_sz[i] && (in_src[i] || resident[i])) ? (char*)in_buf[i]->p + in_sz[i] * s0 : nullptr;
    };
    const void* rs = (retained && h->retained_R) ? (const char*)h->d_R.p + m * m * w * s0 : nullptr;
    auto ao = [&](int i) -> void* { return (out_sz[i] && out_dst[i]) ? (char*)out_buf[i]->p + out_sz[i] * s0 : nullptr; };
    int rc = h->dtype == LCPB200_F32
                 ? launch_backward<float>(h, slot, cb, ai(0), ai(1), ai(2), ai(3), ai(4), ai(5), ai(6), ai(7), ai(8),
                                          ao(0), ao(1), ao(2), ao(3), ao(4), ao(5), ao(6), rs, flags, st)
                 : launch_backward<double>(h, slot, cb, ai(0), ai(1), ai(2), ai(3), ai(4), ai(5), ai(6), ai(7), ai(8),
                                           ao(0), ao(1), ao(2), ao(3), ao(4), ao(5), ao(6), rs, flags, st);
    if (rc) return rc;
    for (int i = 0; i < 7; ++i)
      if (out_sz[i] && out_dst[i])
        CK(cudaMemcpyAsync((char*)out_dst[i] + out_sz[i] * s0, (char*)out_buf[i]->p + out_sz[i] * s0,
                           out_sz[i] * cb, cudaMemcpyDeviceToHost, st));
  }
  for (auto& s : h->streams) CK(cudaStreamSynchronize(s));
  return 0;
}


// ------------------------------------------------------------------ fused engine entry points
// Contact list in, velocities out: the condensed kernels take their structure straight from the
// structure-of-arrays the engine holds; no dense Q / G / F is written to or read from HBM, and the
// backward returns the gradients w.r.t. the contact list (the chain rule through the assembly is
// applied to the factored gradients inside the kernel).
template <typename T>
static void fill_soa(cnd::EngineSoA<T>& s, lcpb200_handle_s* h, int B, int nb, int nc, int mode, double dt,
                     const void* mass, const void* inertia, const void* v, const void* fext, const void* normal,
                     const void* p1, const void* p2, const int32_t* b1, const int32_t* b2, const void* mu,
                     const void* rest, const int32_t* nc_s = nullptr) {
  s.mass = (const T*)mass; s.inertia = (const T*)inertia; s.v = (const T*)v; s.fext = (const T*)fext;
  s.normal = (const T*)normal; s.p1 = (const T*)p1; s.p2 = (const T*)p2; s.mu = (const T*)mu; s.rest = (const T*)rest;
  s.b1 = b1; s.b2 = b2; s.nc_s = nc_s; s.nb = nb; s.nc = nc; s.mode = mode; s.dt = (T)dt;
  s.p_s = (T*)h->d_ph.p;
  s.h_s = s.p_s + (size_t)B * h->n;
}

// Which kernel family serves the engine entry points of this handle: the condensed-KKT kernels (n + e <= 128,
// both dtypes) or the banded large-scene kernel (fp64; LCPB200_FORCE_BANDED=1 routes small fp64 scenes there
// too -- used by the tests to cross-check the two).
static bool use_banded(const lcpb200_handle_s* h) {
  if (h->dtype != LCPB200_F64) return false;
  return !h->cplan.ok || getenv("LCPB200_FORCE_BANDED") != nullptr;
}

static int ensure_bplan(lcpb200_handle_s* h, int B, int nb, int nc, int mode) {
  if (h->bplan_mode != mode) {
    bnd::BPlan& P = h->bplan;
    memset(&P, 0, sizeof(P));
    P.nb = nb; P.n = h->n; P.ncap = nc; P.cs = mode == 0 ? 4 : 1; P.m = h->m; P.e = h->e;
    if (h->e > bnd::BD) return fail("large-scene kernel: more than 16 equality rows");
    const int dyn_max = h->smem_optin - 1024;
    if (!bnd::carve_bplan(P, dyn_max)) return fail("large-scene kernel: the scene does not fit (shared memory)");
    int occ = 0;
    CK(bnd::configure_band(P.smem_bytes, dyn_max, &occ));
    if (occ < 1) return fail("large-scene kernel cannot be resident");
    P.ok = 1;
    h->bplan_mode = mode;
    h->bws_ctas = 0;
  }
  const int ctas = std::min(B, h->num_sms);
  if (ctas > h->bws_ctas) {
    CK(cudaDeviceSynchronize());
    CK(h->d_bwsd.ensure((size_t)ctas * h->bplan.g_doubles * sizeof(double)));
    CK(h->d_bwsi.ensure((size_t)ctas * h->bplan.i_ints * sizeof(int)));
    h->bws_ctas = ctas;
  }
  return 0;
}

static int check_engine(lcpb200_handle_t h, int B, int nb, int nc, int mode) {
  if (!h) return fail("null handle");
  if (B < 0 || nb <= 0 || nc <= 0) return fail("need B >= 0, nb > 0, nc > 0");
  if (mode != 0 && mode != 1) return fail("mode must be 0 (solve_dynamics) or 1 (post_stabilization)");
  if (!h->cplan.ok && h->dtype != LCPB200_F64)
    return fail("engine entry points: n + e > 128 needs the large-scene kernel, which is fp64 only");
  if (h->n != 3 * nb || h->m != (mode == 0 ? 4 : 1) * nc)
    return fail("handle was created for other sizes: need n = 3 nb and m = 4 nc (mode 0) or nc (mode 1)");
  return 0;
}

template <typename T>
static int engine_forward_t(lcpb200_handle_s* h, int B, int nb, int nc, int mode, double dt, const void* mass,
                            const void* inertia, const void* v, const void* fext, const void* normal, const void* p1,
                            const void* p2, const int32_t* b1, const int32_t* b2, const int32_t* ncs, const void* mu,
                            const void* rest, const void* A, const void* b, double eps, int not_improved_lim, int max_iter, void* zhat,
                            void* nu, void* lam, void* slack, int32_t* status, int32_t* iters, void* resid,
                            cudaStream_t st) {
  CK(h->d_ph.ensure(sizeof(T) * (size_t)B * (h->n + h->m)));
  cnd::CFwdArgs<T> c;
  c.P = h->cplan;
  c.B = B;
  c.Q = nullptr; c.G = nullptr; c.F = nullptr;
  c.A = (const T*)A; c.b = (const T*)b;
  fill_soa<T>(c.soa, h, B, nb, nc, mode, dt, mass, inertia, v, fext, normal, p1, p2, b1, b2, mu, rest, ncs);
  c.ssave = nullptr;
  c.p = c.soa.p_s; c.h = c.soa.h_s;
  c.zhat = (T*)zhat; c.nu = (T*)nu; c.lam = (T*)lam; c.slack = (T*)slack; c.resid = (T*)resid;
  c.status = status; c.iters = iters;
  c.eps = (T)eps; c.not_improved_lim = not_improved_lim; c.max_iter = max_iter;
  c.prof = h->cprof;
  const int cgrid = std::min(B, h->cond_grid);
#define CALL_FWD(NSV) cnd::launch_cond_forward_t<T, NSV>(c, cgrid, st)
  const cudaError_t ce = LCPB200_NS_DISPATCH(h->cplan.NS, CALL_FWD);
#undef CALL_FWD
  CK(ce);
  return 0;
}

extern "C" int lcpb200_engine_forward(lcpb200_handle_t h, int B, int nb, int nc, int mode, double dt,
                                      const void* mass, const void* inertia, const void* v, const void* fext,
                                      const void* normal, const void* p1, const void* p2, const int32_t* body1,
                                      const int32_t* body2, const int32_t* contact_count, const void* mu,
                                      const void* restitution, const void* A, const void* b, double eps, int not_improved_lim, int max_iter, void* zhat,
                                      void* nu, void* lam, void* slack, int32_t* status, int32_t* iters, void* resid,
                                      void* stream) {
  if (int rc = check_engine(h, B, nb, nc, mode)) return rc;
  if (!mass || !inertia || !v || !normal || !p1 || !p2 || !body1 || !body2 || !restitution) return fail("engine_forward: NULL input");
  if (mode == 0 && (!fext || !mu)) return fail("engine_forward: fext and mu are needed for mode 0");
  if (h->e > 0 && (!A || !b || !nu)) return fail("handle was created with e > 0 but A, b or nu is NULL");
  if (!zhat || !lam || !slack || !status || !iters) return fail("zhat, lam, slack, status, iters must be non-NULL");
  if (B == 0) return 0;
  DeviceGuard dg_;
  CK(dg_.set(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (use_banded(h)) {
    if (int rc = ensure_bplan(h, B, nb, nc, mode)) return rc;
    bnd::BArgs a;
    a.P = h->bplan;
    a.B = B;
    memset(&a.soa, 0, sizeof(a.soa));
    a.soa.mass = (const double*)mass; a.soa.inertia = (const double*)inertia; a.soa.v = (const double*)v;
    a.soa.fext = (const double*)fext; a.soa.normal = (const double*)normal; a.soa.p1 = (const double*)p1;
    a.soa.p2 = (const double*)p2; a.soa.mu = (const double*)mu; a.soa.rest = (const double*)restitution;
    a.soa.b1 = body1; a.soa.b2 = body2; a.soa.nc_s = contact_count; a.soa.nb = nb; a.soa.nc = nc; a.soa.mode = mode;
    a.soa.dt = dt;
    a.A = (const double*)A; a.b = (const double*)b;
    a.zhat = (double*)zhat; a.nu = (double*)nu; a.lam = (double*)lam; a.slack = (double*)slack; a.resid = (double*)resid;
    a.status = status; a.iters = iters;
    a.eps = eps; a.not_improved_lim = not_improved_lim; a.max_iter = max_iter;
    a.wsd = (double*)h->d_bwsd.p; a.wsi = (int*)h->d_bwsi.p;
    a.prof = h->cprof;
    CK(bnd::launch_band_forward(a, std::min(B, h->num_sms), st));
    return 0;
  }
  return h->dtype == LCPB200_F32
             ? engine_forward_t<float>(h, B, nb, nc, mode, dt, mass, inertia, v, fext, normal, p1, p2, body1, body2,
                                       contact_count, mu, restitution, A, b, eps, not_improved_lim, max_iter, zhat, nu, lam, slack, status,
                                       iters, resid, st)
             : engine_forward_t<double>(h, B, nb, nc, mode, dt, mass, inertia, v, fext, normal, p1, p2, body1, body2,
                                        contact_count, mu, restitution, A, b, eps, not_improved_lim, max_iter, zhat, nu, lam, slack, status,
                                        iters, resid, st);
}

template <typename T>
static int engine_backward_t(lcpb200_handle_s* h, int B, int nb, int nc, int mode, double dt, const void* mass,
                             const void* inertia, const void* v, const void* fext, const void* normal, const void* p1,
                             const void* p2, const int32_t* b1, const int32_t* b2, const int32_t* ncs, const void* mu,
                             const void* rest, const void* A, const void* zhat, const void* nu, const void* lam, const void* slack,
                             const void* g, void* dmass, void* dinertia, void* dv, void* dfext, void* dnormal,
                             void* dp1, void* dp2, void* dmu, void* drest, void* dA, void* db, unsigned flags,
                             cudaStream_t st) {
  CK(h->d_ph.ensure(sizeof(T) * (size_t)B * (h->n + h->m)));
  cnd::CBwdArgs<T> c;
  c.P = h->cplan;
  c.B = B;
  c.Q = nullptr; c.G = nullptr; c.F = nullptr; c.A = (const T*)A;
  c.zhat = (const T*)zhat; c.nu = (const T*)nu; c.lam = (const T*)lam; c.slack = (const T*)slack; c.g = (const T*)g;
  c.dQ = c.dp = c.dG = c.dh = c.dF = nullptr;
  c.dA = (T*)dA; c.db = (T*)db;
  c.done = nullptr; c.only = nullptr; c.flags = flags; c.sload = nullptr;
  c.prof = h->cprof;
  fill_soa<T>(c.soa, h, B, nb, nc, mode, dt, mass, inertia, v, fext, normal, p1, p2, b1, b2, mu, rest, ncs);
  c.dmass = (T*)dmass; c.dinertia = (T*)dinertia; c.dv = (T*)dv; c.dfext = (T*)dfext; c.dnormal = (T*)dnormal;
  c.dp1 = (T*)dp1; c.dp2 = (T*)dp2; c.dmu = (T*)dmu; c.drest = (T*)drest;
  const int cgrid = std::min(B, h->cond_grid);
#define CALL_BWD(NSV) cnd::launch_cond_backward_t<T, NSV>(c, cgrid, st)
  const cudaError_t ce = LCPB200_NS_DISPATCH(h->cplan.NS, CALL_BWD);
#undef CALL_BWD
  CK(ce);
  return 0;
}

extern "C" int lcpb200_engine_backward(lcpb200_handle_t h, int B, int nb, int nc, int mode, double dt,
                                       const void* mass, const void* inertia, const void* v, const void* fext,
                                       const void* normal, const void* p1, const void* p2, const int32_t* body1,
                                       const int32_t* body2, const int32_t* contact_count, const void* mu,
                                       const void* restitution, const void* A, const void* zhat, const void* nu, const void* lam, const void* slack,
                                       const void* dl_dzhat, void* dmass, void* dinertia, void* dv, void* dfext,
                                       void* dnormal, void* dp1, void* dp2, void* dmu, void* drestitution, void* dA,
                                       void* db, unsigned flags, void* stream) {
  if (int rc = check_engine(h, B, nb, nc, mode)) return rc;
  if (!mass || !inertia || !v || !normal || !p1 || !p2 || !body1 || !body2 || !restitution) return fail("engine_backward: NULL input");
  if (mode == 0 && !mu) return fail("engine_backward: mu is needed for mode 0");
  if (!zhat || !lam || !slack || !dl_dzhat) return fail("zhat, lam, slack, dl_dzhat must be non-NULL");
  if (h->e > 0 && (!A || !nu)) return fail("A and nu must be non-NULL when e > 0");
  if (flags != LCPB200_BWD_BUG_COMPATIBLE && flags != LCPB200_BWD_EXACT_ADJOINT)
    return fail("flags must be LCPB200_BWD_BUG_COMPATIBLE or LCPB200_BWD_EXACT_ADJOINT");
  if (B == 0) return 0;
  DeviceGuard dg_;
  CK(dg_.set(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (use_banded(h)) {
    if (flags != LCPB200_BWD_BUG_COMPATIBLE) return fail("engine_backward: the large-scene kernel implements the bug-compatible adjoint only");
    if (int rc = ensure_bplan(h, B, nb, nc, mode)) return rc;
    bnd::BBwdArgs a;
    a.P = h->bplan;
    a.B = B;
    memset(&a.soa, 0, sizeof(a.soa));
    a.soa.mass = (const double*)mass; a.soa.inertia = (const double*)inertia; a.soa.v = (const double*)v;
    a.soa.fext = (const double*)fext; a.soa.normal = (const double*)normal; a.soa.p1 = (const double*)p1;
    a.soa.p2 = (const double*)p2; a.soa.mu = (const double*)mu; a.soa.rest = (const double*)restitution;
    a.soa.b1 = body1; a.soa.b2 = body2; a.soa.nc_s = contact_count; a.soa.nb = nb; a.soa.nc = nc; a.soa.mode = mode;
    a.soa.dt = dt;
    a.A = (const double*)A;
    a.zhat = (const double*)zhat; a.nu = (const double*)nu; a.lam = (const double*)lam; a.slack = (const double*)slack;
    a.g = (const double*)dl_dzhat;
    a.dmass = (double*)dmass; a.dinertia = (double*)dinertia; a.dv = (double*)dv; a.dfext = (double*)dfext;
    a.dnormal = (double*)dnormal; a.dp1 = (double*)dp1; a.dp2 = (double*)dp2; a.dmu = (double*)dmu;
    a.drest = (double*)drestitution; a.dA = (double*)dA; a.db = (double*)db;
    a.wsd = (double*)h->d_bwsd.p; a.wsi = (int*)h->d_bwsi.p;
    a.prof = h->cprof;
    CK(bnd::launch_band_backward(a, std::min(B, h->num_sms), st));
    return 0;
  }
  return h->dtype == LCPB200_F32
             ? engine_backward_t<float>(h, B, nb, nc, mode, dt, mass, inertia, v, fext, normal, p1, p2, body1, body2,
                                        contact_count, mu, restitution, A, zhat, nu, lam, slack, dl_dzhat, dmass, dinertia, dv, dfext,
                                        dnormal, dp1, dp2, dmu, drestitution, dA, db, flags, st)
             : engine_backward_t<double>(h, B, nb, nc, mode, dt, mass, inertia, v, fext, normal, p1, p2, body1, body2,
                                         contact_count, mu, restitution, A, zhat, nu, lam, slack, dl_dzhat, dmass, dinertia, dv, dfext,
                                         dnormal, dp1, dp2, dmu, drestitution, dA, db, flags, st);
}

// ------------------------------------------------------------------ assembly
extern "C" int lcpb200_find_contacts_masked(int dtype, int B, int nb, int cap, double eps, const void* pos,
                                            const void* rad, const uint32_t* skip, int32_t* body1, int32_t* body2,
                                            int32_t* counts, void* stream) {
  if (dtype != LCPB200_F32 && dtype != LCPB200_F64) return fail("bad dtype");
  if (B < 0 || nb <= 0 || cap <= 0) return fail("find_contacts: need B >= 0, nb > 0, cap > 0");
  if (!pos || !rad || !body1 || !body2 || !counts) return fail("find_contacts: NULL argument");
  if (B == 0) return 0;
  int dev = 0, sms = 0;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == LCPB200_F32)
    cts::launch_find_contacts<float>(B, nb, cap, (float)eps, (const float*)pos, (const float*)rad, skip, body1, body2,
                                     counts, sms, st);
  else
    cts::launch_find_contacts<double>(B, nb, cap, eps, (const double*)pos, (const double*)rad, skip, body1, body2,
                                      counts, sms, st);
  CK(cudaGetLastError());
  return 0;
}

extern "C" int lcpb200_find_contacts(int dtype, int B, int nb, int cap, double eps, const void* pos, const void* rad,
                                     int32_t* body1, int32_t* body2, int32_t* counts, void* stream) {
  return lcpb200_find_contacts_masked(dtype, B, nb, cap, eps, pos, rad, nullptr, body1, body2, counts, stream);
}

extern "C" int lcpb200_joint_rows(int dtype, int B, int nb, int e, int nj, const int32_t* rows, const void* pos,
                                  const void* pos1, const void* v, void* A, void* ge, void* stream) {
  if (dtype != LCPB200_F32 && dtype != LCPB200_F64) return fail("bad dtype");
  if (B < 0 || nb <= 0 || e <= 0 || nj < 0) return fail("joint_rows: need B >= 0, nb > 0, e > 0, nj >= 0");
  if (e > jnt::MAX_ROWS) return fail("joint_rows: more than " + std::to_string(jnt::MAX_ROWS) + " rows");
  if (!rows || !pos || !A || (nj > 0 && !pos1)) return fail("joint_rows: NULL argument");
  if (ge && !v) return fail("joint_rows: ge needs v");
  if (B == 0) return 0;
  int dev = 0, sms = 0;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == LCPB200_F32)
    jnt::launch_joint_rows<float>(B, nb, e, nj, rows, (const float*)pos, (const float*)pos1, (const float*)v, (float*)A,
                                  (float*)ge, sms, st);
  else
    jnt::launch_joint_rows<double>(B, nb, e, nj, rows, (const double*)pos, (const double*)pos1, (const double*)v,
                                   (double*)A, (double*)ge, sms, st);
  CK(cudaGetLastError());
  return 0;
}

extern "C" int lcpb200_joint_move(int dtype, int B, int nb, int nj, const int32_t* joint_body, const void* rot1_start,
                                  const void* r1, const void* v, const void* dts, const uint8_t* done, void* rot1,
                                  void* pos1, void* stream) {
  if (dtype != LCPB200_F32 && dtype != LCPB200_F64) return fail("bad dtype");
  if (B < 0 || nb <= 0 || nj < 0) return fail("joint_move: need B >= 0, nb > 0, nj >= 0");
  if (B == 0 || nj == 0) return 0;
  if (!joint_body || !rot1_start || !r1 || !v || !dts || !rot1 || !pos1) return fail("joint_move: NULL argument");
  int dev = 0, sms = 0;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == LCPB200_F32)
    jnt::launch_joint_move<float>(B, nb, nj, joint_body, (const float*)rot1_start, (const float*)r1, (const float*)v,
                                  (const float*)dts, done, (float*)rot1, (float*)pos1, sms, st);
  else
    jnt::launch_joint_move<double>(B, nb, nj, joint_body, (const double*)rot1_start, (const double*)r1,
                                   (const double*)v, (const double*)dts, done, (double*)rot1, (double*)pos1, sms, st);
  CK(cudaGetLastError());
  return 0;
}

extern "C" int lcpb200_contact_geometry(int dtype, int B, int nb, int cap, const void* pos, const void* rad,
                                        const void* fric, const void* rest, const int32_t* body1, const int32_t* body2,
                                        const int32_t* counts, void* normal, void* p1, void* p2, void* pen, void* mu,
                                        void* rest_c, void* stream) {
  if (dtype != LCPB200_F32 && dtype != LCPB200_F64) return fail("bad dtype");
  if (B < 0 || nb <= 0 || cap <= 0) return fail("contact_geometry: need B >= 0, nb > 0, cap > 0");
  if (!pos || !rad || !fric || !rest || !body1 || !body2 || !counts || !normal || !p1 || !p2 || !pen || !mu || !rest_c)
    return fail("contact_geometry: NULL argument");
  if (B == 0) return 0;
  int dev = 0, sms = 0;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == LCPB200_F32)
    cts::launch_contact_geometry<float>(B, nb, cap, (const float*)pos, (const float*)rad, (const float*)fric,
                                        (const float*)rest, body1, body2, counts, (float*)normal, (float*)p1, (float*)p2,
                                        (float*)pen, (float*)mu, (float*)rest_c, sms, st);
  else
    cts::launch_contact_geometry<double>(B, nb, cap, (const double*)pos, (const double*)rad, (const double*)fric,
                                         (const double*)rest, body1, body2, counts, (double*)normal, (double*)p1,
                                         (double*)p2, (double*)pen, (double*)mu, (double*)rest_c, sms, st);
  CK(cudaGetLastError());
  return 0;
}

extern "C" int lcpb200_assemble(int dtype, int B, int nb, int nc, double dt, const void* mass, const void* inertia,
                                const void* v, const void* fext, const void* normal, const void* p1,
                                const void* p2, const int32_t* body1, const int32_t* body2, const void* mu,
                                const void* restitution, void* Q, void* p, void* G, void* hv, void* F,
                                void* stream) {
  if (dtype != LCPB200_F32 && dtype != LCPB200_F64) return fail("bad dtype");
  if (B < 0 || nb <= 0 || nc <= 0) return fail("need B >= 0, nb > 0, nc > 0");
  if (!mass || !inertia || !v || !fext || !normal || !p1 || !p2 || !body1 || !body2 || !mu || !restitution)
    return fail("assemble: NULL input");
  if (!Q || !p || !G || !hv || !F) return fail("assemble: NULL output");
  if (B == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == LCPB200_F32)
    launch_assemble<float>(B, nb, nc, (float)dt, (const float*)mass, (const float*)inertia, (const float*)v,
                           (const float*)fext, (const float*)normal, (const float*)p1, (const float*)p2, body1,
                           body2, (const float*)mu, (const float*)restitution, (float*)Q, (float*)p, (float*)G,
                           (float*)hv, (float*)F, st);
  else
    launch_assemble<double>(B, nb, nc, dt, (const double*)mass, (const double*)inertia, (const double*)v,
                            (const double*)fext, (const double*)normal, (const double*)p1, (const double*)p2,
                            body1, body2, (const double*)mu, (const double*)restitution, (double*)Q, (double*)p,
                            (double*)G, (double*)hv, (double*)F, st);
  CK(cudaGetLastError());
  return 0;
}

extern "C" int lcpb200_assemble_backward(int dtype, int B, int nb, int nc, double dt, const void* mass,
                                         const void* inertia, const void* v, const void* normal, const void* p1,
                                         const void* p2, const int32_t* body1, const int32_t* body2,
                                         const void* mu, const void* restitution, const void* dQ, const void* dp,
                                         const void* dG, const void* dh, const void* dF, void* dmass,
                                         void* dinertia, void* dv, void* dfext, void* dnormal, void* dp1,
                                         void* dp2, void* dmu, void* drestitution, void* stream) {
  if (dtype != LCPB200_F32 && dtype != LCPB200_F64) return fail("bad dtype");
  if (B < 0 || nb <= 0 || nc <= 0) return fail("need B >= 0, nb > 0, nc > 0");
  if (!mass || !inertia || !v || !normal || !p1 || !p2 || !body1 || !body2 || !mu || !restitution)
    return fail("assemble_backward: NULL input");
  if (!dQ || !dp || !dG || !dh || !dF) return fail("assemble_backward: NULL upstream gradient");
  if (B == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == LCPB200_F32)
    launch_assemble_backward<float>(B, nb, nc, (float)dt, (const float*)mass, (const float*)inertia,
                                    (const float*)v, (const float*)normal, (const float*)p1, (const float*)p2,
                                    body1, body2, (const float*)mu, (const float*)restitution, (const float*)dQ,
                                    (const float*)dp, (const float*)dG, (const float*)dh, (const float*)dF,
                                    (float*)dmass, (float*)dinertia, (float*)dv, (float*)dfext, (float*)dnormal,
                                    (float*)dp1, (float*)dp2, (float*)dmu, (float*)drestitution, st);
  else
    launch_assemble_backward<double>(B, nb, nc, dt, (const double*)mass, (const double*)inertia, (const double*)v,
                                     (const double*)normal, (const double*)p1, (const double*)p2, body1, body2,
                                     (const double*)mu, (const double*)restitution, (const double*)dQ,
                                     (const double*)dp, (const double*)dG, (const double*)dh, (const double*)dF,
                                     (double*)dmass, (double*)dinertia, (double*)dv, (double*)dfext,
                                     (double*)dnormal, (double*)dp1, (double*)dp2, (double*)dmu,
                                     (double*)drestitution, st);
  CK(cudaGetLastError());
  return 0;
}
