/* lcpb200.h -- C ABI of the B200-native batched LCP contact solver.
 *
 * The reference (locuslab/lcp-physics) is pure Python and has no FFI; this
 * header is the boundary a maintainer binds with ctypes (see INTEGRATION.md).
 * Every entry point replaces a reference interface on the hot path
 * (paths relative to the reference tree):
 *
 *   lcpb200_forward          lcp_physics/lcp/lcp.py:22-35   LCPFunction.forward
 *                            = lcp/solvers/pdipm.py:357-408 pre_factor_kkt
 *                            + lcp/solvers/pdipm.py:49-179  forward (PDIPM loop)
 *                            + pdipm.py:414-454 factor_kkt, :325-354 solve_kkt,
 *                              :182-186 get_step
 *   lcpb200_backward         lcp_physics/lcp/lcp.py:37-64   LCPFunction.backward
 *   lcpb200_assemble         lcp_physics/physics/world.py:144-234 (M,Jc,Jf,E,mu,
 *                            restitutions) + physics/engines.py:50-74 (G,F,h,p)
 *   lcpb200_assemble_backward  autograd through the same assembly
 *   lcpb200_forward_host / lcpb200_backward_host
 *                            the same calls with HOST buffers (pinned or
 *                            pageable); H2D/D2H copies are done inside, chunked
 *                            and overlapped with the kernels.
 *
 * Conventions
 *   - All matrices are dense, row-major, batch-major and contiguous, exactly
 *     the tensors LCPFunction receives: Q[B,n,n] p[B,n] G[B,m,n] h[B,m]
 *     A[B,e,n] b[B,e] F[B,m,m].  e == 0  <=>  A == b == NULL
 *     (the reference passes 1-D empty tensors, engines.py:59-60).
 *   - dtype: LCPB200_F32 or LCPB200_F64; all floating buffers share it.
 *   - Device pointers unless the function name ends in _host.
 *   - `stream` is a cudaStream_t passed as void*; NULL = legacy default stream.
 *   - Return value 0 = OK; non-zero = error, text via lcpb200_last_error_string().
 *     No exceptions cross the ABI.  Per-scene solver status is reported in
 *     `status[B]` (see LCPB200_STATUS_*): a singular Q sets
 *     LCPB200_STATUS_SINGULAR_Q and the caller raises the reference's
 *     RuntimeError (pdipm.py:361-368).
 *   - Scenes are independent: per-scene termination and per-scene get_step
 *     maximum (SURVEY.md F4: <= 1.5e-12 rel from the batch-coupled reference).
 *   - Two kernel families (DESIGN.md section 3). Scenes with the engine's structure (diagonal Q, sparse
 *     G, block-sparse F) are solved through the condensed n x n KKT system, formed / factored in fp64
 *     without pivoting (it is quasi-definite). Other scenes fall back, per scene, to the dual m x m
 *     form of the reference with threshold partial pivoting restricted to the LU's diagonal blocks
 *     (the reference pivots over whole columns on CPU tensors and not at all on CUDA tensors,
 *     pdipm.py:18 `pivot=not x.is_cuda`).
 *   - One stream at a time per handle (the handle owns the workspace).
 */
#ifndef LCPB200_H
#define LCPB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LCPB200_VERSION 200

#define LCPB200_F32 0
#define LCPB200_F64 1

/* per-scene status written by lcpb200_forward */
#define LCPB200_STATUS_MAX_ITER      0  /* ran all max_iter iterations            */
#define LCPB200_STATUS_NOT_IMPROVED  1  /* not_improved_lim non-improving iters   */
#define LCPB200_STATUS_CONVERGED     2  /* best residual < eps                    */
#define LCPB200_STATUS_DIVERGED      3  /* mu > 1e100                             */
#define LCPB200_STATUS_SINGULAR_Q   -1  /* zero / non-finite pivot factoring Q    */

/* flags for lcpb200_backward */
#define LCPB200_BWD_BUG_COMPATIBLE   0u /* reference behaviour: un-transposed KKT (SURVEY.md F6) */
#define LCPB200_BWD_EXACT_ADJOINT    1u /* transposed KKT system (true adjoint)                  */
#define LCPB200_BWD_REUSE_STRUCTURE  2u /* lcpb200_backward only: (Q, G, A, F) are the inputs of the
                                          * last lcpb200_forward on this handle (same B): reuse the
                                          * block structure it found instead of scanning the dense
                                          * matrices again (19 KB instead of 0.4 MB per scene at
                                          * config 3). Ignored when nothing matching was saved.    */

typedef struct lcpb200_handle_s* lcpb200_handle_t;

int         lcpb200_version(void);
const char* lcpb200_last_error_string(void);

/* Create a solver for problems of size (n, m, e) in `dtype` on CUDA device
 * `device`. The handle owns a small per-CTA workspace (independent of B). */
int lcpb200_create(int dtype, int n, int m, int e, int device, lcpb200_handle_t* out);
int lcpb200_destroy(lcpb200_handle_t h);
size_t lcpb200_workspace_bytes(lcpb200_handle_t h);
/* Describe the launch plan (threads, dynamic smem, grid, which matrices are
 * smem-resident) into `buf` -- for logs and DESIGN.md. */
int lcpb200_describe(lcpb200_handle_t h, char* buf, size_t len);

/* Development aid: per-phase SM cycle counters of the solver kernels, summed over CTAs.
 * enable=1 allocates/zeroes them, 0 frees; out (may be NULL) receives 24 values: the 14 dual-form phases below
 * followed by the 10 condensed-kernel phases {structure, block inverses, assembly of K, LU, solve: right-hand
 * side, solve: substitution, solve: back-substitution of the multipliers, residuals, step rules, gradients}:
 * {prefactor, load T, LU, KKT solves, residuals, step rules,
 *  LU: diagonal blocks (look-ahead warp), LU: panel solves, LU: trailing updates,
 *  LU: diagonal-block inverses, number of diagonal blocks with row interchanges, number of
 *  diagonal blocks, LU: look-ahead warp's panel pieces + block update, LU: other warps waiting
 *  for the look-ahead warp}. */
int lcpb200_profile(lcpb200_handle_t h, int enable, long long* out);

/* LCPFunction.forward. Outputs: zhat[B,n], nu[B,e] (NULL if e==0), lam[B,m],
 * slack[B,m], status[B] int32, iters[B] int32 (PDIPM iterations executed),
 * resid[B] (best residual, same dtype; may be NULL), Rsave[B,m,m] (may be NULL):
 * the Schur matrix R = G Q^-1 G^T + F - ... of every scene (the `self.R` the
 * reference keeps for backward, lcp.py:28); pass it to lcpb200_backward to skip
 * the re-factorisation of Q and the Schur GEMM there. */
int lcpb200_forward(lcpb200_handle_t h, int B,
                    const void* Q, const void* p, const void* G, const void* hvec,
                    const void* A, const void* b, const void* F,
                    double eps, int not_improved_lim, int max_iter,
                    void* zhat, void* nu, void* lam, void* slack,
                    int32_t* status, int32_t* iters, void* resid, void* Rsave,
                    void* stream);

/* LCPFunction.backward. Inputs: the forward inputs it needs (Q,G,A,F), the
 * saved forward results (zhat, nu, lam, slack) and dl_dzhat[B,n].
 * Outputs (any may be NULL = skip): dQ[B,n,n] dp[B,n] dG[B,m,n] dh[B,m]
 * dA[B,e,n] db[B,e] dF[B,m,m]. */
int lcpb200_backward(lcpb200_handle_t h, int B,
                     const void* Q, const void* G, const void* A, const void* F,
                     const void* zhat, const void* nu, const void* lam, const void* slack,
                     const void* dl_dzhat,
                     void* dQ, void* dp, void* dG, void* dh, void* dA, void* db, void* dF,
                     const void* Rsave /* from lcpb200_forward, or NULL = recompute */,
                     unsigned flags, void* stream);

/* Same two calls with HOST buffers: copies in, solves, copies out. The timed
 * "e2e" path of bench.py. Synchronous on return. forward_host leaves its inputs,
 * results and R on the device; backward_host with Q == NULL (then G, A, F, zhat,
 * nu, lam, slack are ignored) reuses them instead of uploading them again -- the
 * save_for_backward of lcp.py:34. Any other call on the handle drops that state. */
int lcpb200_forward_host(lcpb200_handle_t h, int B,
                         const void* Q, const void* p, const void* G, const void* hvec,
                         const void* A, const void* b, const void* F,
                         double eps, int not_improved_lim, int max_iter,
                         void* zhat, void* nu, void* lam, void* slack,
                         int32_t* status, int32_t* iters, void* resid);
int lcpb200_backward_host(lcpb200_handle_t h, int B,
                          const void* Q, const void* G, const void* A, const void* F,
                          const void* zhat, const void* nu, const void* lam, const void* slack,
                          const void* dl_dzhat,
                          void* dQ, void* dp, void* dG, void* dh, void* dA, void* db, void* dF,
                          unsigned flags);

/* Contact detection for B scenes of nb circles (replaces the pair loop of World.find_contacts,
 * physics/world.py:139-142, with the circle-circle test of physics/contacts.py:68-80: a pair (i < j) is a
 * contact iff rad_i + rad_j - |pos_i - pos_j| >= -eps). Device pointers:
 *   pos[B,nb,2] rad[B,nb]                      body centres and radii (dtype)
 *   body1[B,cap] body2[B,cap] int32            OUT: the touching pairs of every scene in lexicographic pair
 *                                              order (the order the reference appends contacts in), padded
 *                                              with the pair (0, 1)
 *   counts[B] int32                            OUT: number of touching pairs (may exceed cap: then the lists
 *                                              hold the first cap pairs and the caller must grow cap)
 * The contact geometry (normal, p1, p2, penetration) of the selected pairs is the caller's (it is O(cap) and,
 * in the torch mirror, differentiable). */
int lcpb200_find_contacts(int dtype, int B, int nb, int cap, double eps, const void* pos, const void* rad,
                          int32_t* body1, int32_t* body2, int32_t* counts, void* stream);

/* lcpb200_find_contacts with pairs that never produce a contact (bodies.py:104-106 `add_no_contact`,
 * contacts.py:60-61): skip is a bitmask over the lexicographic pair index q of (i < j), q = i (2 nb - i - 1) / 2 +
 * j - i - 1, bit q & 31 of word q >> 5 (ceil(nb (nb - 1) / 64) words, shared by the batch). A skipped pair is
 * neither counted nor listed; the order of the others is unchanged. skip == NULL is lcpb200_find_contacts. */
int lcpb200_find_contacts_masked(int dtype, int B, int nb, int cap, double eps, const void* pos, const void* rad,
                                 const uint32_t* skip, int32_t* body1, int32_t* body2, int32_t* counts, void* stream);

/* Equality rows of joints (World.Je(), physics/world.py:156-170, Jacobians of physics/constraints.py) for B
 * scenes with one constraint topology. Device pointers:
 *   rows[e,4] int32        one {kind, body1, body2 or -1, aux} per row: kind 0 = unit row on dof aux of body1
 *                          (X / Y / Rot / TotalConstraint), 1 / 2 = first / second row of a revolute Joint
 *                          (J1 = [-y1, 1, 0] / [x1, 0, 1], J2 = [y2, -1, 0] / [-x2, 0, -1]) with pos1 = the lever
 *                          of revolute joint aux (aux = -1: pos1 = 0, the FixedJoint's), 3 = [1,0,0] / [-1,0,0]
 *                          (the FixedJoint's rotation row); pos2 = p_body1 + pos1 - p_body2
 *   pos[B,nb,2]            body centres;  pos1[B,nj,2]: levers of the nj revolute joints (NULL if nj == 0)
 *   A[B,e,3nb]             OUT: dense rows, every element written
 *   v[B,3nb], ge[B,e]      optional (both or neither): ge = A v, the b of post-stabilisation (engines.py:87)
 * e <= 256. */
int lcpb200_joint_rows(int dtype, int B, int nb, int e, int nj, const int32_t* rows, const void* pos,
                       const void* pos1, const void* v, void* A, void* ge, void* stream);

/* Joint.move (constraints.py:38-45) of the nj revolute joints of B scenes:
 *   rot1[s,k] = rot1_start[s,k] + v[s, 3 joint_body[k]] dts[s],  pos1[s,k] = r1[s,k] (cos, sin)(rot1[s,k])
 * joint_body[nj] int32 (body 1 of each joint), rot1_start / r1 / rot1 [B,nj], v[B,3nb], dts[B], pos1[B,nj,2].
 * done[B] (uint8, may be NULL): scenes with done[s] != 0 keep rot1 and pos1. rot1_start may alias rot1. */
int lcpb200_joint_move(int dtype, int B, int nb, int nj, const int32_t* joint_body, const void* rot1_start,
                       const void* r1, const void* v, const void* dts, const uint8_t* done, void* rot1, void* pos1,
                       void* stream);

/* Geometry and material of the pairs selected by lcpb200_find_contacts (contacts.py:69-77, world.py:144-151,
 * :213-224), for callers that do not differentiate through the contact generation:
 *   normal[B,cap,2] = (pos1 - pos2) / dist, penetration[B,cap] = r1 + r2 - dist (-1e30 in unused slots),
 *   p1 = -normal (r1 - pen / 2), p2 = normal (r2 - pen / 2), mu / restitution[B,cap] = mean of the two bodies'
 *   fric_coeff[B,nb] / restitution[B,nb]. */
int lcpb200_contact_geometry(int dtype, int B, int nb, int cap, const void* pos, const void* rad,
                             const void* fric_coeff, const void* restitution, const int32_t* body1,
                             const int32_t* body2, const int32_t* counts, void* normal, void* p1, void* p2,
                             void* penetration, void* mu, void* restitution_c, void* stream);

/* Contact-list -> dense LCP assembly for B scenes of nb bodies (3 dofs each,
 * n = 3 nb), nc contacts, fd = 2 friction directions (world.py:191-192),
 * m = nc (2 + fd). Structure-of-arrays inputs:
 *   mass[B,nb] inertia[B,nb] v[B,n] fext[B,n]           bodies
 *   normal[B,nc,2] p1[B,nc,2] p2[B,nc,2]                contact geometry
 *   body1[nc] body2[nc] int32 (shared by the batch)     contact topology
 *   mu[B,nc] restitution[B,nc]                          contact material
 * Outputs: Q[B,n,n] p[B,n] G[B,m,n] h[B,m] F[B,m,m]  with
 *   p = M v + dt fext,  h = [(Jc v) restitution, 0, 0]  (engines.py:32,53,74). */
int lcpb200_assemble(int dtype, int B, int nb, int nc, double dt,
                     const void* mass, const void* inertia, const void* v, const void* fext,
                     const void* normal, const void* p1, const void* p2,
                     const int32_t* body1, const int32_t* body2,
                     const void* mu, const void* restitution,
                     void* Q, void* p, void* G, void* hvec, void* F, void* stream);

/* Adjoint of lcpb200_assemble: given dQ dp dG dh dF, accumulate gradients
 * w.r.t. mass, inertia, v, fext, normal, p1, p2, mu, restitution (any NULL = skip). */
int lcpb200_assemble_backward(int dtype, int B, int nb, int nc, double dt,
                              const void* mass, const void* inertia, const void* v,
                              const void* normal, const void* p1, const void* p2,
                              const int32_t* body1, const int32_t* body2,
                              const void* mu, const void* restitution,
                              const void* dQ, const void* dp, const void* dG,
                              const void* dh, const void* dF,
                              void* dmass, void* dinertia, void* dv, void* dfext,
                              void* dnormal, void* dp1, void* dp2,
                              void* dmu, void* drestitution, void* stream);

/* Fused engine entry points (SURVEY.md 8(b): lcpb200_assemble_solve). They replace, in ONE kernel per pass,
 *   mode 0: PdipmEngine.solve_dynamics' LCP (physics/engines.py:50-76) incl. the assembly of
 *           world.py:144-234:  zhat = LCP(M, M v + dt f, [Jc; Jf; 0], [(Jc v) rest, 0, 0], A, b, F(E, mu));
 *           the engine returns -zhat (engines.py:76);
 *   mode 1: PdipmEngine.post_stabilization's LCP (physics/engines.py:80-116):
 *           zhat = LCP(M, 0, Jc, (Jc v)(1 - rest), A, b, 0).
 * Inputs are the contact structure-of-arrays of lcpb200_assemble (+ optional equality rows A[B,e,n], b[B,e],
 * e.g. World.Je()); nothing dense is written to or read from HBM. The handle must have been created with
 * n = 3 nb, m = 4 nc (mode 0) or nc (mode 1). n + e <= 128: the condensed-KKT kernels (fp32 / fp64); larger
 * scenes (fp64 only, e.g. BASELINE config 4: 512 bodies): the banded large-scene kernels (lcp_banded.cuh), which
 * order the bodies so that the condensed matrix is an arrow matrix (half bandwidth <= 128 after the ordering, <= 16
 * border rows: pinned bodies, bodies with > 12 contacts, equality rows). A scene whose contact topology the kernel
 * cannot take (a contact of a body with itself, > 16 contacts on one body for the condensed kernels, a band or
 * border beyond the limits above) gets status -100 and no result: assemble it with lcpb200_assemble and call
 * lcpb200_forward.
 * contact_count == NULL: every scene has the nc contacts body1[nc], body2[nc] (one topology for the batch).
 * contact_count[B] != NULL (batched worlds): scene s uses its first contact_count[s] <= nc contacts, body1 /
 * body2 are [B,nc] and all per-contact arrays are strided by nc; a scene with 0 contacts gets the
 * equality-constrained solve of engines.py:35-49; lam / slack rows of scene s are laid out for ITS count
 * (normal rows [0,c), friction [c,3c), gamma [3c,4c)), the arrays keep the stride m.
 * lcpb200_engine_backward: the chain rule through the assembly applied to the factored gradients of
 * lcp.py:52-63 (dG = dlam (x) zhat + lam (x) dx, ...): gradients w.r.t. the contact list, any may be NULL. */
int lcpb200_engine_forward(lcpb200_handle_t h, int B, int nb, int nc, int mode, double dt,
                           const void* mass, const void* inertia, const void* v, const void* fext,
                           const void* normal, const void* p1, const void* p2,
                           const int32_t* body1, const int32_t* body2, const int32_t* contact_count,
                           const void* mu, const void* restitution, const void* A, const void* b,
                           double eps, int not_improved_lim, int max_iter,
                           void* zhat, void* nu, void* lam, void* slack,
                           int32_t* status, int32_t* iters, void* resid, void* stream);
int lcpb200_engine_backward(lcpb200_handle_t h, int B, int nb, int nc, int mode, double dt,
                            const void* mass, const void* inertia, const void* v, const void* fext,
                            const void* normal, const void* p1, const void* p2,
                            const int32_t* body1, const int32_t* body2, const int32_t* contact_count,
                            const void* mu, const void* restitution, const void* A,
                            const void* zhat, const void* nu, const void* lam, const void* slack,
                            const void* dl_dzhat,
                            void* dmass, void* dinertia, void* dv, void* dfext,
                            void* dnormal, void* dp1, void* dp2, void* dmu, void* drestitution,
                            void* dA, void* db, unsigned flags, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LCPB200_H */
