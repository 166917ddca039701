// lcp_contacts.cuh -- batched contact detection for scenes of circles (SURVEY.md section 8 row f-2).
//
// Restates the circle-circle branch of the reference's contact handler (physics/contacts.py:68-80) together
// with the pair enumeration of World.find_contacts (physics/world.py:139-142: the broadphase callback visits
// every pair of geoms once):
//     r = rad_i + rad_j;  dist = |pos_i - pos_j|;  penetration = r - dist;  contact iff penetration >= -eps.
// One CTA per scene walks all nb (nb - 1) / 2 pairs (i < j) in lexicographic order -- the order in which the
// reference appends to world.contacts for circle scenes, which fixes the row order of Jc / Jf / E and therefore
// the LCP the engine builds -- and compacts the touching pairs IN THAT ORDER with a block-wide exclusive scan
// (ballot prefix inside a warp, warp totals through shared memory): deterministic, no atomics, no sort.
// Outputs: the pair list body1 / body2 [B, cap] (padded with the pair (0, 1)), and the TRUE number of touching
// pairs per scene (which may exceed cap: the caller checks). An optional skip bitmask over the pair index q (bit
// q & 31 of word q >> 5, shared by the batch) removes pairs that never produce a contact (`add_no_contact`,
// bodies.py:104-106, contacts.py:60-61): a skipped pair is neither counted nor listed. The contact geometry (normal, p1, p2, penetration)
// is evaluated by the caller on the selected pairs only (O(cap), differentiable in torch), so this kernel
// replaces the O(nb^2) part: at nb = 513 it tests 131 328 pairs per scene.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace lcpb200 {
namespace cts {

constexpr int NT = 256;
constexpr int ITEMS = 4;            // consecutive pairs per thread and chunk

// number of pairs (i', j') with i' < i, i.e. index of pair (i, i + 1)
__device__ __forceinline__ long long pairs_before(long long i, long long nb) { return i * (2 * nb - i - 1) / 2; }

template <typename T>
__global__ void __launch_bounds__(NT) find_contacts_kernel(int B, int nb, int cap, T eps, const T* __restrict__ pos,
                                                           const T* __restrict__ rad, const uint32_t* __restrict__ skip,
                                                           int32_t* __restrict__ body1, int32_t* __restrict__ body2,
                                                           int32_t* __restrict__ counts) {
  __shared__ int warp_tot[NT / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long npairs = (long long)nb * (nb - 1) / 2;
  for (int sc = blockIdx.x; sc < B; sc += gridDim.x) {
    const T* P = pos + (size_t)sc * nb * 2;
    const T* R = rad + (size_t)sc * nb;
    int32_t* o1 = body1 + (size_t)sc * cap;
    int32_t* o2 = body2 + (size_t)sc * cap;
    int base = 0;                                                // touching pairs found in the previous chunks
    for (long long q0 = 0; q0 < npairs; q0 += (long long)NT * ITEMS) {
      const long long q = q0 + (long long)tid * ITEMS;
      int i = 0, j = 0;
      if (q < npairs) {                                          // (i, j) of pair q: closed form + exact fix-up
        const double t = 2.0 * nb - 1.0;
        long long ii = (long long)floor((t - sqrt(t * t - 8.0 * (double)q)) * 0.5);
        if (ii < 0) ii = 0;
        if (ii > nb - 2) ii = nb - 2;
        while (ii + 1 <= nb - 2 && pairs_before(ii + 1, nb) <= q) ++ii;
        while (ii > 0 && pairs_before(ii, nb) > q) --ii;
        i = (int)ii;
        j = (int)(q - pairs_before(ii, nb)) + i + 1;
      }
      unsigned hit = 0;
      int pi[ITEMS], pj[ITEMS];
#pragma unroll
      for (int u = 0; u < ITEMS; ++u) {
        pi[u] = i; pj[u] = j;
        if (q + u < npairs) {
          const long long qu = q + u;
          if (skip == nullptr || !((skip[qu >> 5] >> (qu & 31)) & 1u)) {   // `if geom1 in geom2.no_contact: return`
            const T dx = P[2 * i] - P[2 * j], dy = P[2 * i + 1] - P[2 * j + 1];
            const T dist = sqrt(dx * dx + dy * dy);
            const T pen = R[i] + R[j] - dist;                    // contacts.py:70-73
            if (!(pen < -eps)) hit |= 1u << u;                   // `if penetration < -eps: return`
          }
          if (++j == nb) { ++i; j = i + 1; }
        }
      }
      const int mine = __popc(hit);
      int incl = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
      if (lane == 31) warp_tot[warp] = incl;
      __syncthreads();
      int before = base, total = 0;
#pragma unroll
      for (int w = 0; w < NT / 32; ++w) { const int v = warp_tot[w]; if (w < warp) before += v; total += v; }
      int at = before + incl - mine;
#pragma unroll
      for (int u = 0; u < ITEMS; ++u)
        if (hit & (1u << u)) { if (at < cap) { o1[at] = pi[u]; o2[at] = pj[u]; } ++at; }
      base += total;
      __syncthreads();                                           // warp_tot is rewritten by the next chunk
    }
    for (int k = base + tid; k < cap; k += NT) { o1[k] = 0; o2[k] = nb > 1 ? 1 : 0; }      // padding: a valid pair
    if (tid == 0) counts[sc] = base;
  }
}

// Geometry of the selected pairs (contacts.py:69-77, world.py:144-151, :213-224), for callers that do not need
// autograd through the contact generation: normal = (pos1 - pos2) / dist, penetration = r1 + r2 - dist,
// p1 = -normal (r1 - pen / 2), p2 = normal (r2 - pen / 2), mu / restitution = mean of the two bodies'. Unused slots
// (k >= counts[scene]) get the geometry of the padding pair and penetration = -1e30.
template <typename T>
__global__ void __launch_bounds__(NT) contact_geometry_kernel(int B, int nb, int cap, const T* __restrict__ pos,
                                                              const T* __restrict__ rad, const T* __restrict__ fric,
                                                              const T* __restrict__ rest, const int32_t* __restrict__ body1,
                                                              const int32_t* __restrict__ body2,
                                                              const int32_t* __restrict__ counts, T* __restrict__ normal,
                                                              T* __restrict__ p1, T* __restrict__ p2, T* __restrict__ pen,
                                                              T* __restrict__ mu, T* __restrict__ rest_c) {
  const long long total = (long long)B * cap;
  for (long long t = blockIdx.x * (long long)NT + threadIdx.x; t < total; t += (long long)gridDim.x * NT) {
    const int sc = (int)(t / cap), k = (int)(t - (long long)sc * cap);
    const int i = body1[t], j = body2[t];
    const T* P = pos + (size_t)sc * nb * 2;
    const T* R = rad + (size_t)sc * nb;
    const T dx = P[2 * i] - P[2 * j], dy = P[2 * i + 1] - P[2 * j + 1];
    const T dist = sqrt(dx * dx + dy * dy);
    const T r1 = R[i], r2 = R[j];
    const T pn = r1 + r2 - dist;
    const T nx = dx / dist, ny = dy / dist;
    const T a1 = r1 - pn / 2, a2 = r2 - pn / 2;
    normal[2 * t] = nx; normal[2 * t + 1] = ny;
    p1[2 * t] = -nx * a1; p1[2 * t + 1] = -ny * a1;
    p2[2 * t] = nx * a2; p2[2 * t + 1] = ny * a2;
    pen[t] = k < counts[sc] ? pn : T(-1e30);
    mu[t] = T(0.5) * (fric[(size_t)sc * nb + i] + fric[(size_t)sc * nb + j]);
    rest_c[t] = T(0.5) * (rest[(size_t)sc * nb + i] + rest[(size_t)sc * nb + j]);
  }
}

template <typename T>
static void launch_contact_geometry(int B, int nb, int cap, const T* pos, const T* rad, const T* fric, const T* rest,
                                    const int32_t* body1, const int32_t* body2, const int32_t* counts, T* normal, T* p1,
                                    T* p2, T* pen, T* mu, T* rest_c, int num_sms, cudaStream_t st) {
  const long long total = (long long)B * cap;
  long long grid = (total + NT - 1) / NT;
  if (grid > 8LL * num_sms) grid = 8LL * num_sms;
  contact_geometry_kernel<T><<<(int)grid, NT, 0, st>>>(B, nb, cap, pos, rad, fric, rest, body1, body2, counts, normal, p1, p2,
                                                        pen, mu, rest_c);
}

template <typename T>
static void launch_find_contacts(int B, int nb, int cap, T eps, const T* pos, const T* rad, const uint32_t* skip,
                                 int32_t* body1, int32_t* body2, int32_t* counts, int num_sms, cudaStream_t st) {
  const int grid = B < 8 * num_sms ? B : 8 * num_sms;
  find_contacts_kernel<T><<<grid, NT, 0, st>>>(B, nb, cap, eps, pos, rad, skip, body1, body2, counts);
}

}  // namespace cts
}  // namespace lcpb200
