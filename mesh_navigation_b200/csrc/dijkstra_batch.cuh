// Batches of full-field Dijkstra plans (mnb_dijkstra_batch): one goal per CTA, or per cluster of CS CTAs, persistent groups
// pull goal indices from an atomic counter -- the shape of k_cvp_batch, without the band engine.
//
// Why a label-correcting loop reproduces the heap loop bit for bit: edge weights are >= 0, so without a robot cutoff the
// final distance of DijkstraMeshPlanner::dijkstra does not depend on pop order.  It is the least fixed point of
//   d[seed] = 0,   d[c] = min over expandable neighbours u of fl(d[u] + w(u,c))   (c valid, c != seed)
// with expandable(u) = !((double)cost[u] > cost_limit) (dijkstra:302) and invalid vertices never relaxed (:328).  fl(x + w)
// is monotone in x, so relaxing from +inf in any order, until nothing improves, ends at exactly that fixed point.  The
// predecessor depends on pop order only through exact ties; the reference's strict `<` in pop order makes it the argmin of
// (fl(d[u] + w), d[u], u) over the expandable neighbours (DijkstraProblem::recompute), evaluated once on the converged row.
// (Zero-weight edges between equal labels are the one case where that order is not the pop order: DESIGN.md §7.)
//
// A round: every candidate whose current label lies below the bucket end (smallest label pushed in the previous round plus
// the band width) relaxes its edges with atomicMin on the float bits (non-negative floats order like their bits; NaN and
// +inf sums never pass `tmp < d`); improved, expandable vertices and the candidates beyond the bucket end go to the next
// round's list, once each (per-vertex round stamp).  Scratch per group: stamp + two lists = 12 B per vertex; the labels are
// the goal's output row itself.
#pragma once
#include "band_engine.cuh"

namespace mnb {

struct DijkstraBatchArgs {
  uint32_t V;
  const uint32_t* adj_ptr; const uint2* adj_nw; const uint4* ell_adj;
  const float* cost; const uint8_t* invalid;
  double cost_limit;
  float delta;                  // bucket width (potential units)
  uint32_t n_queries;
  const uint32_t* seeds;        // [n_queries] device
  float* out_dist;              // [n_queries][V]: the labels live here
  uint32_t* out_pred;           // [n_queries][V] or null
  uint32_t* scratch;            // per group g: 3 V words at g * 3 V: stamp, list0, list1
  GroupCtl* ctl;                // [groups]
  unsigned int* next_query;
  const int* cancel_flag;
  uint32_t max_rounds;
};

using DijkstraBatchStage = StageT<4096>;

// calls f(neighbour, weight) for every edge of u: the 8-slot ELL row, the CSR list beyond 8 neighbours
template <class F>
__device__ __forceinline__ void djb_edges(const DijkstraBatchArgs& a, uint32_t u, F f) {
  const uint4 r0 = __ldg(&a.ell_adj[(size_t)u * ELL_W]);
  const uint32_t deg = r0.w;
  if (deg <= ELL_W) {
    if (deg) f(r0.x, __uint_as_float(r0.y));
    for (uint32_t k = 1; k < deg; ++k) {
      const uint4 r = __ldg(&a.ell_adj[(size_t)u * ELL_W + k]);
      f(r.x, __uint_as_float(r.y));
    }
  } else {
    const uint32_t kb = __ldg(&a.adj_ptr[u]), ke = __ldg(&a.adj_ptr[u + 1]);
    for (uint32_t k = kb; k < ke; ++k) {
      const uint2 nw = __ldg(&a.adj_nw[k]);
      f(nw.x, __uint_as_float(nw.y));
    }
  }
}

__device__ __forceinline__ bool djb_expandable(const DijkstraBatchArgs& a, uint32_t u) {
  return !((double)__ldg(&a.cost[u]) > a.cost_limit);       // dijkstra:302
}

constexpr int DJB_THREADS = 256, DJB_MINBLOCKS = 4;     // 48 registers: four CTAs per SM

template <int CS>
__global__ void __launch_bounds__(DJB_THREADS, DJB_MINBLOCKS) k_dijkstra_batch(const DijkstraBatchArgs a) {
  constexpr unsigned FULL = 0xffffffffu;
  const float INF = __uint_as_float(INF_BITS);
  __shared__ DijkstraBatchStage st;
  uint32_t g, gthreads, gtid;
  group_coords<CS>(g, gthreads, gtid);
  const uint32_t V = a.V, lane = threadIdx.x & 31;
  uint32_t* const stamp = a.scratch + (size_t)g * 3 * V;
  uint32_t* const list0 = stamp + V;
  uint32_t* const list1 = list0 + V;
  GroupCtl* const ctl = a.ctl + g;
  if (threadIdx.x == 0) { st.n = 0; st.m_tau = INF_BITS; st.lo = INF_BITS; }
  __syncthreads();
  for (;;) {
    if (gtid == 0) ctl->query = atomicAdd(a.next_query, 1u);
    group_sync<CS>();
    const uint32_t q = __ldcg(&ctl->query);
    if (q >= a.n_queries) break;
    const uint32_t seed = a.seeds[q];
    uint32_t* const dist = reinterpret_cast<uint32_t*>(a.out_dist + (size_t)q * V);   // float bits
    for (uint32_t v = gtid; v < V; v += gthreads) { dist[v] = INF_BITS; stamp[v] = 0u; }
    group_sync<CS>();
    if (gtid == 0) {
      dist[seed] = 0u;                                     // dijkstra:276 (an invalid seed too, as the reference does)
      stamp[seed] = 1u; list0[0] = seed;
      ctl->count[0] = 1u; ctl->count[1] = 0u;
      ctl->lo[0] = 0u; ctl->lo[1] = INF_BITS;
      ctl->stop_ring[0] = 0u; ctl->stop_ring[1] = 0u;
    }
    group_sync<CS>();
    unsigned int my_reached = gtid == 0 ? 1u : 0u;         // (the seed)
    unsigned long long my_relax = 0;
    uint32_t r = 0;
    for (;; ++r) {
      // round r reads slot r % 3 and fills slot (r + 1) % 3; slot (r + 2) % 3 was last read in round r - 1, before the barrier
      const uint32_t slot = r % 3, next = (r + 1) % 3;
      const unsigned int n = __ldcg(&ctl->count[slot]);
      const float lo = __uint_as_float(__ldcg(&ctl->lo[slot]));
      const unsigned int stop = __ldcg(&ctl->stop_ring[r & 1]);
      if (n == 0 || stop || r > a.max_rounds) break;       // group-uniform: the watchdog cannot deadlock the barrier
      float bucket_end = lo + a.delta;
      if (!(bucket_end > lo)) bucket_end = nextafterf(lo, INF);   // the smallest pushed label is always expanded
      if (gtid == 0) {
        ctl->count[(r + 2) % 3] = 0u; ctl->lo[(r + 2) % 3] = INF_BITS;
        ctl->stop_ring[(r + 1) & 1] = (a.cancel_flag && (r & 31) == 0 && *(const volatile int*)a.cancel_flag) ? 1u : 0u;
      }
      const uint32_t* const list_r = (r & 1) ? list1 : list0;
      uint32_t* const list_n = (r & 1) ? list0 : list1;
      unsigned int* const count_next = &ctl->count[next];
      const uint32_t tag = r + 2u;                         // stamp of the vertices in the next round's list
      float my_lo = INF;
      auto push = [&](uint32_t v, float d) {
        my_lo = fminf(my_lo, d);
        if (__ldcg(&stamp[v]) == tag || atomicExch(&stamp[v], tag) == tag) return;
        const unsigned int p = atomicAdd(&st.n, 1u);
        if (p < (unsigned)DijkstraBatchStage::CAP) st.buf[p] = v;
        else list_n[atomicAdd(count_next, 1u)] = v;        // overflow: straight to global
      };
      for (uint32_t i = gtid; i < n; i += gthreads) {
        const uint32_t u = __ldcg(&list_r[i]);
        const float du = __uint_as_float(__ldcg(&dist[u]));
        if (!(du < bucket_end)) { push(u, du); continue; }  // beyond the bucket: next round
        if (!djb_expandable(a, u)) continue;
        djb_edges(a, u, [&](uint32_t c, float w) {
          if (a.invalid && a.invalid[c]) return;            // dijkstra:328
          ++my_relax;
          const float tmp = __fadd_rn(du, w);               // dijkstra:331
          if (!(tmp < __uint_as_float(__ldcg(&dist[c])))) return;
          const uint32_t old = atomicMin(&dist[c], __float_as_uint(tmp));
          if (__float_as_uint(tmp) >= old) return;
          if (old == INF_BITS) ++my_reached;
          if (djb_expandable(a, c)) push(c, tmp);
        });
      }
      const unsigned int wl = __reduce_min_sync(FULL, __float_as_uint(my_lo));
      if (lane == 0 && wl != INF_BITS) atomicMin(&st.lo, wl);
      stage_flush(st, list_n, count_next, &ctl->m_tau[next], &ctl->lo[next]);
      group_sync<CS>();
    }
    {
      const unsigned int wr = __reduce_add_sync(FULL, my_reached);
      unsigned long long wx = my_relax;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) wx += __shfl_xor_sync(FULL, wx, o);
      if (lane == 0) { if (wr) atomicAdd(&ctl->settled, (unsigned long long)wr); if (wx) atomicAdd(&ctl->recomputes, wx); }
    }
    if (gtid == 0) { ctl->rounds += r; if (r > a.max_rounds) ctl->watchdog = 1; }
    group_sync<CS>();
    if (a.out_pred) {
      // predecessors from the converged row (DijkstraProblem::recompute's argmin): seed -> itself, unreached / invalid -> self
      uint32_t* const pred = a.out_pred + (size_t)q * V;
      for (uint32_t c = gtid; c < V; c += gthreads) {
        uint32_t best_u = c;
        if (c != seed && __ldcg(&dist[c]) != INF_BITS && !(a.invalid && a.invalid[c])) {
          float best = INF, best_du = INF;
          djb_edges(a, c, [&](uint32_t u, float w) {
            if (!djb_expandable(a, u)) return;
            const float du = __uint_as_float(__ldcg(&dist[u]));
            const float tmp = __fadd_rn(du, w);
            if (DijkstraEllProblem::better(tmp, du, u, best, best_du, best_u)) { best = tmp; best_du = du; best_u = u; }
          });
          if (__float_as_uint(best) == INF_BITS) best_u = c;
        }
        pred[c] = best_u;
      }
    }
    group_sync<CS>();
  }
}

}  // namespace mnb
