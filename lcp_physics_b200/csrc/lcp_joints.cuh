// lcp_joints.cuh -- equality rows of joints for batched worlds of circles (BatchedWorld joints=).
//
// Restates World.Je() (physics/world.py:156-170) for B scenes that share one constraint topology, with the
// Jacobians of physics/constraints.py:
//     Joint (revolute, :29-36)    J1 = [[-y1, 1, 0], [x1, 0, 1]],  J2 = [[y2, -1, 0], [-x2, 0, -1]]
//     FixedJoint (:70-77)         pos1 = 0, pos2 = p_b1 - p_b2, the two rows above and [1,0,0] / [-1,0,0]
//     X / Y / Rot / TotalConstraint   unit rows on one dof of body 1
// with pos1 the revolute joint's lever on body 1 (the per-scene state) and pos2 = p_b1 + pos1 - p_b2 at the current
// positions. The topology is a row table built once on the host: one int4 {kind, body1, body2 or -1, aux} per row,
// aux = the dof of a unit row or the revolute-joint index of a lever row (-1: the FixedJoint's pos1 = 0).
//
// joint_rows_kernel: one CTA per scene (persistent grid). The rows' two 3-vectors are formed in shared memory,
// then the dense A[scene] (e x 3 nb, every element including the zeros) is written with consecutive threads on
// consecutive elements. With v != NULL it also writes ge = A v (the b of post-stabilisation, engines.py:87), from
// the non-zero entries only.
// joint_move_kernel: Joint.move (constraints.py:38-45) for every scene and revolute joint,
//     rot1 = rot1_start + v[3 b1] dts,  pos1 = r1 (cos rot1, sin rot1),
// except in scenes flagged done, which keep their state (step_dt's per-scene dt halving, world.py:88-107).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace lcpb200 {
namespace jnt {

constexpr int NT = 256;
constexpr int MAX_ROWS = 256;       // shared-memory capacity per scene (the engine kernels take <= 128 rows)

enum RowKind { UNIT = 0, LEVER_X = 1, LEVER_Y = 2, ROT = 3 };

template <typename T>
__global__ void __launch_bounds__(NT) joint_rows_kernel(int B, int nb, int e, int nj, const int32_t* __restrict__ rows,
                                                        const T* __restrict__ pos, const T* __restrict__ pos1,
                                                        const T* __restrict__ v, T* __restrict__ A, T* __restrict__ ge) {
  __shared__ T vals[MAX_ROWS * 6];  // J1 (3), J2 (3) of every row
  __shared__ int rb1[MAX_ROWS], rb2[MAX_ROWS];
  const int n = 3 * nb;
  const long long en = (long long)e * n;
  for (int sc = blockIdx.x; sc < B; sc += gridDim.x) {
    const T* P = pos + (size_t)sc * nb * 2;
    for (int r = threadIdx.x; r < e; r += NT) {
      const int kind = rows[4 * r], b1 = rows[4 * r + 1], b2 = rows[4 * r + 2], aux = rows[4 * r + 3];
      T j1[3] = {T(0), T(0), T(0)}, j2[3] = {T(0), T(0), T(0)};
      if (kind == UNIT) {
        j1[0] = T(aux == 0); j1[1] = T(aux == 1); j1[2] = T(aux == 2);
      } else if (kind == ROT) {
        j1[0] = T(1); j2[0] = T(-1);
      } else {
        T x1 = T(0), y1 = T(0), x2 = T(0), y2 = T(0);
        if (aux >= 0) { x1 = pos1[((size_t)sc * nj + aux) * 2]; y1 = pos1[((size_t)sc * nj + aux) * 2 + 1]; }
        if (b2 >= 0) { x2 = (P[2 * b1] + x1) - P[2 * b2]; y2 = (P[2 * b1 + 1] + y1) - P[2 * b2 + 1]; }
        if (kind == LEVER_X) { j1[0] = -y1; j1[1] = T(1); j2[0] = y2; j2[1] = T(-1); }
        else                 { j1[0] = x1; j1[2] = T(1); j2[0] = -x2; j2[2] = T(-1); }
      }
#pragma unroll
      for (int q = 0; q < 3; ++q) { vals[6 * r + q] = j1[q]; vals[6 * r + 3 + q] = j2[q]; }
      rb1[r] = b1; rb2[r] = b2;
      if (ge != nullptr) {
        const T* V = v + (size_t)sc * n;
        T acc = j1[0] * V[3 * b1] + j1[1] * V[3 * b1 + 1] + j1[2] * V[3 * b1 + 2];
        if (b2 >= 0) acc += j2[0] * V[3 * b2] + j2[1] * V[3 * b2 + 1] + j2[2] * V[3 * b2 + 2];
        ge[(size_t)sc * e + r] = acc;
      }
    }
    __syncthreads();
    T* Asc = A + (size_t)sc * en;
    for (long long k = threadIdx.x; k < en; k += NT) {
      const int r = (int)(k / n), c = (int)(k - (long long)r * n);
      const int body = c / 3, q = c - 3 * body;
      Asc[k] = body == rb1[r] ? vals[6 * r + q] : body == rb2[r] ? vals[6 * r + 3 + q] : T(0);
    }
    __syncthreads();                                             // vals / rb* are rewritten for the next scene
  }
}

template <typename T>
__global__ void __launch_bounds__(NT) joint_move_kernel(int B, int nb, int nj, const int32_t* __restrict__ joint_body,
                                                        const T* rot1_start, const T* __restrict__ r1,
                                                        const T* __restrict__ v, const T* __restrict__ dts,
                                                        const uint8_t* __restrict__ done, T* rot1, T* __restrict__ pos1) {
  // rot1_start may alias rot1 (post-stabilisation moves the state in place): every element is read before it is written
  const long long total = (long long)B * nj;
  for (long long t = blockIdx.x * (long long)NT + threadIdx.x; t < total; t += (long long)gridDim.x * NT) {
    const int sc = (int)(t / nj), k = (int)(t - (long long)sc * nj);
    if (done != nullptr && done[sc]) continue;
    const T rot = rot1_start[t] + v[(size_t)sc * 3 * nb + 3 * joint_body[k]] * dts[sc];
    rot1[t] = rot;
    pos1[2 * t] = cos(rot) * r1[t];
    pos1[2 * t + 1] = sin(rot) * r1[t];
  }
}

template <typename T>
static void launch_joint_rows(int B, int nb, int e, int nj, const int32_t* rows, const T* pos, const T* pos1, const T* v,
                              T* A, T* ge, int num_sms, cudaStream_t st) {
  const int grid = B < 8 * num_sms ? B : 8 * num_sms;
  joint_rows_kernel<T><<<grid, NT, 0, st>>>(B, nb, e, nj, rows, pos, pos1, v, A, ge);
}

template <typename T>
static void launch_joint_move(int B, int nb, int nj, const int32_t* joint_body, const T* rot1_start, const T* r1,
                              const T* v, const T* dts, const uint8_t* done, T* rot1, T* pos1, int num_sms,
                              cudaStream_t st) {
  const long long total = (long long)B * nj;
  long long grid = (total + NT - 1) / NT;
  if (grid > 8LL * num_sms) grid = 8LL * num_sms;
  joint_move_kernel<T><<<(int)grid, NT, 0, st>>>(B, nb, nj, joint_body, rot1_start, r1, v, dts, done, rot1, pos1);
}

}  // namespace jnt
}  // namespace lcpb200
