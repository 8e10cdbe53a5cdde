// binpack.cu — K3: BinpackingNodeEstimator.Estimate (estimator/binpacking_estimator.go:97-247) on the GPU.
//
// One THREAD BLOCK per template (templates are independent simulations; inside one, placement order is
// sequential by construction), persistent with an atomic work counter over a longest-first work order.
// A thread owns the nodes j = tid, tid + TPB, ... of the simulation ("thread per node"): the running
// state of the nodes the estimate adds (free[A] int64, pod slots, used host ports, has-pods flag) lives
// in SHARED memory, every per-group pass is one sweep of the block over the open nodes followed by a
// block reduction; the state of the pre-existing cluster nodes (touched only by the hostname-spread
// fallback) stays in a per-block global slab.
//
// Plain groups (identical pods, no topology spread / inter-pod affinity involvement): CLOSED FORM
//   * tryToScheduleOnExistingNodes (:141-164): SchedulePodOnAnyNodeMatching scans cyclically from
//     lastIndex (predicate/plugin_runner.go:81,123), so identical pods are dealt round-robin over the
//     added nodes with spare capacity k_j: every node gets min(k_j, L), the first `rem` nodes in cyclic
//     order with k_j > L get one more (L = largest lap count with sum min(k_j, L) <= n).
//   * tryToScheduleOnNewNodes (:168-247): only the last added node is tried, so each new node takes
//     min(remaining, k_new) until the limiter denies (:222); an empty last node stops the group (:212);
//     a pod that fits no fresh node still adds one (:227-240).
// Groups under topology counters (dyn.cuh) take the CAPACITY FORM when every counter is a per-node capacity or a budget:
//   * hostname-key counters see one domain per node: a DoNotSchedule spread constraint whose global minimum is PINNED
//     at 0 (proved per group) admits (maxSkew - self - count) / weight + 1 pods on a node, an (existing-)anti-affinity
//     counter one pod; the same round-robin closed form then applies to the added nodes AND to the fallback of
//     :186-205, which deals the pods the last node refuses FOR SKEW over the CLUSTER nodes in cyclic order;
//   * counters on any other key see ONE domain for all added nodes and bound the pods the group can place at all.
// Every other group runs the reference's per-pod loop against incremental counters (copy-on-write over the cluster
// base counts): per pod one block-wide evaluation of every open node, a block-wide arg-min of the cyclic distance,
// one placement.
// Per (template, group) step the block reads ONE 144-byte group record that travelled one group ahead (cp.async);
// groups that provably find no room (per-template capacity bounds, a ring of dead requests) skip their sweep.
// FM = true is HintingSimulator.TrySchedulePods on the cluster nodes (the filter-out-schedulable pass), see the
// kernel's comment.  The file is compiled in three parts (BP_PART) so that build() can run them in parallel.
#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "engine.h"

namespace cae {

struct BpParams {
  int E, T, N, U, t_begin, t_end, cap, has_dyn, dstride, log_cap;
  int win;                 // added nodes resident in shared memory (= cap), 0 when they do not fit
  const int32_t *order, *order_n;
  const GroupRec* grec;    // [E] one record per pending pod group
  const int32_t* perm;     // work order of the templates
  const uint8_t* pre_code;
  const int32_t *spec_sc, *spec_dc;
  const int64_t* tmpl_free;  // [A][T]
  const int32_t *tmpl_slots, *max_nodes, *pc_of;
  const unsigned long long* port_conf;
  const int64_t* c_free;  // [A][N]
  const int32_t* c_slots;
  int act_dim[CAE_MAX_RES];
  int32_t *node_count, *pod_count, *sched, *work_counter, *status;
  const int32_t* last_index_in;   // [T] or NULL: the plugin runner's lastIndex when the Estimate of template t starts
  int32_t* last_index_out;        // [T] or NULL: ... and when it returns
  long long* prof;         // optional [16] counters (CAE_PACK_PROF)
  // filter-out-schedulable pass (FM): HintingSimulator.TrySchedulePods on the cluster nodes; `grec` then holds one record
  // per RUN of consecutive identical pods (pad[0] = offset of the run in fm_pods)
  int fm_runs, fm_last_index, fm_break, fm_nctrl;
  const int32_t *fm_pods, *fm_hint, *fm_class, *fm_class_ctrl;
  const uint8_t* fm_node_ok;
  int32_t *fm_assigned, *fm_out;          // [P] node or -1; {lastIndex, overflowing controllers, pods scheduled, moved}
  int32_t* fm_ctrl_cnt;                   // [controllers] classes stored per controller (zeroed)
  uint8_t *fm_class_mark, *fm_ctrl_over;  // [classes] known unschedulable, [controllers] overflowing (zeroed)
  // batched scale-down (FM with sim_n > 0): RemovalSimulator.SimulateNodeRemoval for sim_n candidates in turn, see the kernel
  int sim_n, sim_persist, sim_max_removable, sim_trace_cap;
  const int32_t *sim_cand, *sim_pod_off, *sim_pods, *sim_run_off;   // [n] node, [n+1] own pods (CSR), [n+1] own runs in grec
  const GroupRec* sim_rec_pod;            // [P] one-pod record of every pending pod (pods moved in by an earlier candidate)
  int32_t *sim_result, *sim_trace_off, *sim_trace_pod, *sim_trace_node;
  int32_t* sim_st;                             // [SIM_WORDS] state of the candidate loop (SIM_LI = lastIndex in, raw)
  const uint8_t* sim_dest;                     // [N] destination map or NULL; fm_node_ok then points at sim_nok
  uint8_t *sim_present, *sim_nok, *sim_seen;   // [N] node in the snapshot (init 1), present && destination, candidate seen
  int32_t *sim_pos, *sim_at, *sim_gone;        // [N] list position of a present node, node at a position; [n] nodes taken out
  int32_t *sim_mv_head, *sim_mv_tail, *sim_mv_next;   // pods placed on a node by persisted simulations, in placement order
  int64_t* sim_bk_free;                        // [A1][N] node state before the running simulation (undo)
  unsigned long long* sim_bk_ports;
  int32_t* sim_bk_slots;
  unsigned char* scratch;
  size_t scratch_per_cta;
};

constexpr int BP_HIST = 256;   // capacities up to this use the histogram; above, a binary search

// description of the dynamic group being placed (shared memory, uniform reads)
struct GroupDyn {
  int nq;
  int qid[DYN_MAX_Q], kind[DYN_MAX_Q], k[DYN_MAX_Q], host[DYN_MAX_Q], Dc[DYN_MAX_Q], tslot[DYN_MAX_Q];
  int wown[DYN_MAX_Q], self[DYN_MAX_Q], maxskew[DYN_MAX_Q], mindom[DYN_MAX_Q], elig_new[DYN_MAX_Q], dsw[DYN_MAX_Q];
  int minv[DYN_MAX_Q], nmin[DYN_MAX_Q], ndom[DYN_MAX_Q], tot[DYN_MAX_Q], boff[DYN_MAX_Q], nfeed[DYN_MAX_Q];
  int aff_self;
};

struct BpShared {
  GroupRec rec[2];            // record of the current group / the next one (in flight)
  GroupDyn wd;
  int flag[DYN_MAX_Q];        // counters whose minimum must be recomputed
  long long rl[2][32];
  long long rb[2][32][CAE_MAX_RES];   // refresh of the per-template capacity bounds
  int ri[2][32][3];
  int hist[BP_HIST + 1];      // #nodes per capacity value (closed-form lap count)
  int t, L, rem, pre_s, log_n, overflow, newly, need_log, mlast, lastnode;
  long long dead[4][CAE_MAX_RES];   // requests (no host ports) whose sweep found no room since the node state last changed
};

__device__ __forceinline__ int bp_wsum(int v) { return __reduce_add_sync(0xffffffffu, v); }   // REDUX: one instruction
__device__ __forceinline__ long long bp_wsum_ll(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ long long bp_wmax_ll(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int bp_wmax(int v) { return __reduce_max_sync(0xffffffffu, v); }
__device__ __forceinline__ int bp_wmin(int v) { return __reduce_min_sync(0xffffffffu, v); }

// Block reductions: one barrier each.  Two scratch rows alternate (`par`), so a row is rewritten only
// after every thread has passed the barrier of the reduction in between.
template <int NW>
__device__ __forceinline__ void blk_sum_ll_max(BpShared& S, int& par, long long& a, int& b) {
  a = bp_wsum_ll(a); b = bp_wmax(b);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) { S.rl[par][w] = a; S.ri[par][w][0] = b; }
  __syncthreads();
  a = bp_wsum_ll(lane < NW ? S.rl[par][lane] : 0ll);
  b = bp_wmax(lane < NW ? S.ri[par][lane][0] : INT_MIN);
  par ^= 1;
}
template <int NW>
__device__ __forceinline__ void blk_sum_sum_max(BpShared& S, int& par, int& a, int& b, int& c) {
  a = bp_wsum(a); b = bp_wsum(b); c = bp_wmax(c);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) { S.ri[par][w][0] = a; S.ri[par][w][1] = b; S.ri[par][w][2] = c; }
  __syncthreads();
  a = bp_wsum(lane < NW ? S.ri[par][lane][0] : 0);
  b = bp_wsum(lane < NW ? S.ri[par][lane][1] : 0);
  c = bp_wmax(lane < NW ? S.ri[par][lane][2] : INT_MIN);
  par ^= 1;
}
// a: sum of per-thread values each <= clampv (<= 2^26), clamped to clampv after every stage; b: max; c: sum
template <int NW>
__device__ __forceinline__ void blk_csum_max_sum(BpShared& S, int& par, int clampv, int& a, int& b, int& c) {
  a = min(bp_wsum(a), clampv); b = bp_wmax(b); c = bp_wsum(c);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) { S.ri[par][w][0] = a; S.ri[par][w][1] = b; S.ri[par][w][2] = c; }
  __syncthreads();
  a = min(bp_wsum(lane < NW ? S.ri[par][lane][0] : 0), clampv);
  b = bp_wmax(lane < NW ? S.ri[par][lane][1] : INT_MIN);
  c = bp_wsum(lane < NW ? S.ri[par][lane][2] : 0);
  par ^= 1;
}
template <int NW>
__device__ __forceinline__ void blk_sum_max(BpShared& S, int& par, int& a, int& b) {
  a = bp_wsum(a); b = bp_wmax(b);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) { S.ri[par][w][0] = a; S.ri[par][w][1] = b; }
  __syncthreads();
  a = bp_wsum(lane < NW ? S.ri[par][lane][0] : 0);
  b = bp_wmax(lane < NW ? S.ri[par][lane][1] : INT_MIN);
  par ^= 1;
}
template <int NW>
__device__ __forceinline__ void blk_min_sum(BpShared& S, int& par, int& a, int& b) {
  a = bp_wmin(a); b = bp_wsum(b);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) { S.ri[par][w][0] = a; S.ri[par][w][1] = b; }
  __syncthreads();
  a = bp_wmin(lane < NW ? S.ri[par][lane][0] : INT_MAX);
  b = bp_wsum(lane < NW ? S.ri[par][lane][1] : 0);
  par ^= 1;
}
template <int NW>
__device__ __forceinline__ long long blk_sum_ll(BpShared& S, int& par, long long a) {
  a = bp_wsum_ll(a);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) S.rl[par][w] = a;
  __syncthreads();
  a = bp_wsum_ll(lane < NW ? S.rl[par][lane] : 0ll);
  par ^= 1;
  return a;
}

#ifndef BP_UNROLL
#define BP_UNROLL 1
#endif
constexpr int kBpUnroll = BP_UNROLL;   // unroll factor of the per-node sweeps
#ifndef BP_MIN_CTAS
#define BP_MIN_CTAS 4
#endif

__device__ __forceinline__ void bp_cp_async16(void* smem_dst, const void* gmem_src) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem_src));
}
__device__ __forceinline__ void bp_cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void bp_cp_async_wait() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

// floor(f / r) for f >= r > 0 with a quotient below 2^31: one double division + an exact +-1 correction
// (|double error| < 2^-20 of the quotient), instead of the ~100-instruction 64-bit integer division
__device__ __forceinline__ int bp_div(int64_t f, int64_t r) {
  long long q = (long long)(__ll2double_rn(f) / __ll2double_rn(r));
  if (q * r > f) --q;
  else if ((q + 1) * r <= f) ++q;
  return (int)q;
}

// the same with a precomputed float reciprocal of r, for quotients below `kbound` <= 2^20: the float estimate is
// within 1 of the true quotient (relative error < 2^-21), the correction makes it exact
__device__ __forceinline__ int bp_div_f(int64_t f, int64_t r, float rinv, int kbound) {
  if (kbound > (1 << 20)) return bp_div(f, r);
  int q = (int)(__ll2float_rz(f) * rinv);
  const long long qr = (long long)q * r;
  if (qr > f) --q;
  else if (qr + r <= f) ++q;
  return q;
}

// FM = true: the same machinery as HintingSimulator.TrySchedulePods on the CLUSTER snapshot
// (simulator/scheduling/hinting_simulator.go:53-135; filterOutSchedulableByPacking, core/podlistprocessor/
// filter_out_schedulable.go:96-126): ONE simulation on one thread block, no template, the node list is the N cluster nodes,
// pods arrive as runs of consecutive identical pods in the caller's order.  Plain runs are dealt in closed form (lap by lap,
// because every pod's node is reported), hinted pods and pods under topology counters one by one, with the
// SimilarPodsScheduling shortcut (similar_pods.go:59-104).
// With p.sim_n > 0 the same block runs the planner's scale-down loop (RemovalSimulator.SimulateNodeRemoval per candidate,
// simulator/cluster.go:126-217): candidates in order on one snapshot, each one's pods tried with breakOnFailure on the node
// list WITHOUT the candidate.  The node list is the cluster order minus the nodes taken out (presence mask + block prefix:
// scans and lastIndex use list positions); a taken-out node's residents and the pods logged on it stop counting and its
// domains lose one eligible node (replayed into the copy-on-write counters like the placement log).  A successful
// simulation with persist stays (its pods are appended to the pods-to-move of the nodes they landed on), any other one is
// undone from a copy of the node state and by truncating the log.  lastIndex runs through the whole loop.
template <int A, int TPB, bool WIN, bool FM>
__global__ void __launch_bounds__(TPB, FM ? 1 : BP_MIN_CTAS * 256 / TPB) binpack_kernel(DevObjects o, DynTables d, BpParams p) {
  constexpr int NW = TPB / 32;
  constexpr int A1 = A > 0 ? A : 1;
  extern __shared__ __align__(16) unsigned char bp_dsm[];
  __shared__ BpShared S;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int N = p.N, NT = p.N + p.T;
  const int Neff = (p.has_dyn || FM) ? N : 0;   // cluster nodes carry run state only when a placement can reach them
  const int win = p.win;
  const int Xg = Neff + (win ? 0 : p.cap);
  // ---- shared window: the nodes this estimate adds ----
  int64_t* s_free = reinterpret_cast<int64_t*>(bp_dsm);                                        // [A1][win]
  unsigned long long* s_ports = reinterpret_cast<unsigned long long*>(s_free + (size_t)A1 * win);  // [win]
  int32_t* s_slots = reinterpret_cast<int32_t*>(s_ports + win);                                // [win]
  int32_t* s_kc = s_slots + win;                                                               // [win] capacity for the current group
  int32_t* s_pre = s_kc + win;                                                                 // [win] ordered prefix (final-lap ranks)
  uint8_t* s_sched = reinterpret_cast<uint8_t*>(s_pre + win);                                  // [win] node holds a scheduled pod
  // ---- global slab: cluster nodes (and the added nodes when they do not fit the window) ----
  unsigned char* slab = p.scratch + (size_t)blockIdx.x * p.scratch_per_cta;
  int32_t* hdr = reinterpret_cast<int32_t*>(slab);   // version counter survives across launches
  int64_t* g_free = reinterpret_cast<int64_t*>(slab + 16);                                     // [A1][Xg]
  unsigned long long* g_ports = reinterpret_cast<unsigned long long*>(g_free + (size_t)A1 * Xg);
  int32_t* g_slots = reinterpret_cast<int32_t*>(g_ports + Xg);
  int32_t* g_kc = g_slots + Xg;
  int32_t* g_pre = g_kc + Xg;
  int32_t* wcnt = g_pre + Xg;                                                                  // [DYN_MAX_Q][dstride]
  int32_t* wpres = wcnt + (size_t)DYN_MAX_Q * p.dstride;
  int32_t* wver = wpres + (size_t)DYN_MAX_Q * p.dstride;                                       // slot version
  int32_t* logbuf = wver + (size_t)DYN_MAX_Q * p.dstride;                                      // [log_cap][3]
  int32_t* g_aux = logbuf + (size_t)p.log_cap * 3;                                            // [Xg] pods dealt to a node (FM)
  uint8_t* g_sched = reinterpret_cast<uint8_t*>(g_aux + Xg);                                   // [Xg]

  // added node j (shared window, or the slab behind the cluster nodes when the window does not fit)
  auto afr = [&](int a, int j) -> int64_t& { if constexpr (WIN) return s_free[a * win + j]; else return g_free[(size_t)a * Xg + Neff + j]; };
  auto apo = [&](int j) -> unsigned long long& { if constexpr (WIN) return s_ports[j]; else return g_ports[Neff + j]; };
  auto asl = [&](int j) -> int32_t& { if constexpr (WIN) return s_slots[j]; else return g_slots[Neff + j]; };
  auto akc = [&](int j) -> int32_t& { if constexpr (WIN) return s_kc[j]; else return g_kc[Neff + j]; };
  auto apr = [&](int j) -> int32_t& { if constexpr (WIN) return s_pre[j]; else return g_pre[Neff + j]; };
  auto asch = [&](int j) -> uint8_t& { if constexpr (WIN) return s_sched[j]; else return g_sched[Neff + j]; };
  // cluster node x < Neff
  auto cfr = [&](int a, int x) -> int64_t& { return g_free[(size_t)a * Xg + x]; };
  auto cpo = [&](int x) -> unsigned long long& { return g_ports[x]; };
  auto csl = [&](int x) -> int32_t& { return g_slots[x]; };
  auto csch = [&](int x) -> uint8_t& { return g_sched[x]; };
  // any node of the simulation, x < Neff: cluster, else added node x - Neff (per-pod loop only)
  auto fr = [&](int a, int x) -> int64_t& { return x >= Neff ? afr(a, x - Neff) : cfr(a, x); };
  auto po = [&](int x) -> unsigned long long& { return x >= Neff ? apo(x - Neff) : cpo(x); };
  auto sl_ = [&](int x) -> int32_t& { return x >= Neff ? asl(x - Neff) : csl(x); };
  auto sch = [&](int x) -> uint8_t& { return x >= Neff ? asch(x - Neff) : csch(x); };

  GroupDyn& wd = S.wd;
  int par = 0;                 // block-uniform parity of the reduction scratch
  // CAE_PACK_PROF=1: cycles per phase / event counts, thread 0 of every block, summed over the launch
  long long prof_t0 = 0;
#define BP_PROF_BEGIN() do { if (p.prof && tid == 0) prof_t0 = clock64(); } while (0)
#define BP_PROF_END(slot) do { if (p.prof && tid == 0) atomicAdd((unsigned long long*)&p.prof[slot], (unsigned long long)(clock64() - prof_t0)); } while (0)
#define BP_PROF_COUNT(slot, v) do { if (p.prof && tid == 0) atomicAdd((unsigned long long*)&p.prof[slot], (unsigned long long)(v)); } while (0)
  int gver_ctr = hdr[1] + 1;

  for (;;) {
    __syncthreads();
    if (tid == 0) {
      const int i = atomicAdd(p.work_counter, 1);
      if (FM) S.t = i == 0 ? 0 : p.t_end;
      else S.t = i >= p.t_end - p.t_begin ? p.t_end : (p.perm ? p.perm[i] : p.t_begin + i);
      S.log_n = 0; S.overflow = 0;
    }
    __syncthreads();
    const int t = S.t;
    if (t >= p.t_end) break;
    const long long prof_tmpl0 = (p.prof && tid == 0) ? clock64() : 0;

    int64_t tfree[A1];
#pragma unroll
    for (int a = 0; a < A; ++a) tfree[a] = FM ? 0 : p.tmpl_free[(size_t)a * p.T + t];
    const int tslots = FM ? 0 : p.tmpl_slots[t];
    const int max_nodes = (!FM && p.max_nodes) ? p.max_nodes[t] : 0;
    const int col_new = N + p.T + t;  // universe column of the sanitized template
    // lastIndex may come in RAW (left by a longer node list): plugin_runner.go:81 uses it modulo the CURRENT list length
    // until a scan places a pod (:123), so every scan start below is taken through li_eff()
    int n_new = 0, nodes_with_pods = 0, pods_total = 0, last_index = FM ? p.fm_last_index : (p.last_index_in ? p.last_index_in[t] : 0);
    auto li_eff = [&]() -> int { const int len = N + n_new; return len > 0 ? last_index % len : 0; };
    bool new_nodes_available = !FM, cl_init = false, fm_stop = false, fm_moved = false;
    auto ensure_cluster = [&]() {  // run state of the cluster nodes, needed once a placement can reach them
      if (cl_init) return;
      for (int x = tid; x < N; x += TPB) {
#pragma unroll
        for (int a = 0; a < A; ++a) g_free[(size_t)a * Xg + x] = p.c_free[(size_t)a * N + x];
        g_slots[x] = p.c_slots[x];
        g_ports[x] = 0ull;
        g_sched[x] = 0;
      }
      cl_init = true;
      __syncthreads();
    };
    if (FM) ensure_cluster();
    // batched scale-down: node list of the running simulation (identity for a single filter pass)
    const bool batch = FM && p.sim_n > 0;
    auto sv = [&](int i) -> int32_t& { return p.sim_st[i]; };   // state of the candidate loop (thread 0 writes, barriers publish)
    auto Ncur = [&]() -> int { return batch ? sv(SIM_NCUR) : N; };   // length of the node list
    auto pos_of = [&](int x) -> int { return batch ? p.sim_pos[x] : x; };
    auto node_at = [&](int i) -> int { return batch ? p.sim_at[i] : i; };
    // Upper bounds of what ANY added node still has (free only shrinks, so a stale bound stays valid): a group whose
    // request exceeds them skips its pass over the open nodes; tightened whenever such a pass finds no room at all.
    int64_t maxfree[A1];
    int maxslots = INT_MIN;
#pragma unroll
    for (int a = 0; a < A; ++a) maxfree[a] = LLONG_MIN;
    // A request that found NO room in a sweep stays dead until a node is ADDED (placements only shrink what is free): a later
    // plain group asking at least as much in every dimension skips its sweep.  Only port-free requests are remembered
    // (a request with host ports can fail for its ports alone); the last four, a ring.
    int n_dead = 0, dead_next = 0;
    auto refresh_bounds = [&]() {
      long long mf[A1];
      int msl = INT_MIN;
#pragma unroll
      for (int a = 0; a < A; ++a) mf[a] = LLONG_MIN;
      for (int j = tid; j < n_new; j += TPB) {
        msl = max(msl, asl(j));
#pragma unroll
        for (int a = 0; a < A; ++a) mf[a] = max(mf[a], (long long)afr(a, j));
      }
      msl = bp_wmax(msl);
#pragma unroll
      for (int a = 0; a < A; ++a) mf[a] = bp_wmax_ll(mf[a]);
      if (lane == 0) {
        S.ri[par][warp][0] = msl;
#pragma unroll
        for (int a = 0; a < A; ++a) S.rb[par][warp][a] = mf[a];
      }
      __syncthreads();
      maxslots = bp_wmax(lane < NW ? S.ri[par][lane][0] : INT_MIN);
#pragma unroll
      for (int a = 0; a < A; ++a) maxfree[a] = bp_wmax_ll(lane < NW ? S.rb[par][lane][a] : LLONG_MIN);
      par ^= 1;
    };
    const int n_groups0 = FM ? p.fm_runs : p.order_n[t];
    auto n_groups = [&]() -> int { return batch ? sv(SIM_RUNS_OWN) + sv(SIM_MOVED) : n_groups0; };
    // pod k of the pass (batch: of the running simulation's list in the trace: its own pods, then the pods moved in)
    auto run_pod = [&](int k) -> int { return batch ? p.sim_trace_pod[sv(SIM_SEG) + k] : p.fm_pods[k]; };

    auto log_append = [&](int x, int spec, int cnt) {  // any thread
      const int idx = atomicAdd(&S.log_n, 1);
      if (idx < p.log_cap) { logbuf[idx * 3] = x; logbuf[idx * 3 + 1] = spec; logbuf[idx * 3 + 2] = cnt; }
      else S.overflow = 1;
    };

    // Identical pods dealt round-robin over `cnt` nodes (node i of the range has capacity capfn(i), cyclic
    // scan order starts at node s): closed form of repeated SchedulePodOnAnyNodeMatching calls.
    // applyfn(i, m) books m pods on node i and returns 1 when the node held no scheduled pod before.
    // Returns pods placed, nodes newly holding pods, cyclic distance from s of the node that took the LAST pod.
    auto round_robin = [&](int cnt, int s, int npods, auto capfn, auto kcref, auto preref, auto applyfn,
                           int& got, int& newly, int& last_dist) {
      got = 0; newly = 0; last_dist = -1;
      // pass 1: capacities; their sum only matters up to npods + 1, so it travels as a clamped 32-bit value
      const int clampv = npods < (1 << 26) ? npods + 1 : (1 << 26);
      int total = 0, kmax = 0, npos = 0;
#pragma unroll kBpUnroll
      for (int i = tid; i < cnt; i += TPB) {
        const int k = capfn(i);
        kcref(i) = k;
        total = min(total + min(k, clampv), clampv);
        kmax = max(kmax, k);
        npos += k > 0;
      }
      blk_csum_max_sum<NW>(S, par, clampv, total, kmax, npos);
      if (total <= 0) return;
      int L, rem;
      bool exact = npods < (1 << 26);   // the clamped sum decides total <= npods
      if (!exact) {
        long long t2 = 0;
        for (int i = tid; i < cnt; i += TPB) t2 += kcref(i);
        t2 = blk_sum_ll<NW>(S, par, t2);
        total = t2 <= npods ? (int)t2 : INT_MAX;
      }
      if (total <= npods) { L = kmax; rem = 0; got = total; }            // every node takes its full capacity
      else if (npos >= npods) { L = 0; rem = npods; got = npods; }       // one pod each on the first npods nodes with room
      else if (kmax <= BP_HIST) {
        got = npods;
        // histogram of the capacities: lanes with the same value elect one writer
        for (int i = tid; i <= BP_HIST; i += TPB) S.hist[i] = 0;
        __syncthreads();
        for (int base = 0; base < cnt; base += TPB) {
          const int i = base + tid;
          const int k = i < cnt ? kcref(i) : 0;
          const bool cntd = k > 0;
          const unsigned peers = __match_any_sync(0xffffffffu, cntd ? k : 0);
          if (cntd && lane == __ffs(peers) - 1) atomicAdd(&S.hist[k], __popc(peers));
        }
        __syncthreads();
        // f(L) = sum_j min(k_j, L) = sum_{l <= L} G(l), G(l) = #{k_j >= l}: two warp scans over the histogram
        if (warp == 0) {
          constexpr int PB = BP_HIST / 32;
          int c[PB], G[PB];
          int lane_tot = 0;
#pragma unroll
          for (int i = 0; i < PB; ++i) { c[i] = S.hist[lane * PB + i + 1]; lane_tot += c[i]; }
          int suf = lane_tot;   // inclusive suffix sum over lanes
#pragma unroll
          for (int off = 1; off < 32; off <<= 1) {
            const int v = __shfl_down_sync(0xffffffffu, suf, off);
            if (lane + off < 32) suf += v;
          }
          int run = suf - lane_tot, gsum = 0;   // counts of the lanes above
#pragma unroll
          for (int i = PB - 1; i >= 0; --i) { run += c[i]; G[i] = run; gsum += run; }
          int pre = gsum;       // inclusive prefix sum over lanes
#pragma unroll
          for (int off = 1; off < 32; off <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, pre, off);
            if (lane >= off) pre += v;
          }
          int f = pre - gsum, cn = 0, fbest = 0;
#pragma unroll
          for (int i = 0; i < PB; ++i) {
            f += G[i];          // f(lane * PB + i + 1)
            if (f <= npods) { ++cn; fbest = f; }
          }
          cn = bp_wsum(cn);     // f is strictly increasing up to kmax and f(kmax) = total > npods
          fbest = bp_wmax(fbest);
          if (lane == 0) { S.L = cn; S.rem = npods - fbest; }
        }
        __syncthreads();
        L = S.L; rem = S.rem;
      } else {
        got = npods;
        int lo = 0, hi = kmax;  // f(lo) <= npods < f(hi)
        long long flo = 0;
        while (hi - lo > 1) {
          const int mid = (lo + hi) >> 1;
          long long f = 0;
          for (int i = tid; i < cnt; i += TPB) f += min(kcref(i), mid);
          f = blk_sum_ll<NW>(S, par, f);
          if (f <= npods) { lo = mid; flo = f; } else hi = mid;
        }
        L = lo;
        rem = (int)(npods - flo);
      }
      // final lap: the first `rem` nodes in cyclic order from s with k > L take one more
      int pre_s = 0, tot_extra = 0;
      if (rem > 0) {
        int basecnt = 0;
        for (int base = 0; base < cnt; base += TPB) {
          const int i = base + tid;
          const bool ex = i < cnt && kcref(i) > L;
          const unsigned m = __ballot_sync(0xffffffffu, ex);
          if (lane == 0) S.ri[par][warp][0] = __popc(m);
          __syncthreads();
          const int v = lane < NW ? S.ri[par][lane][0] : 0;
          int inc = v;          // inclusive scan over the warps' counts
#pragma unroll
          for (int off = 1; off < 32; off <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, inc, off);
            if (lane >= off) inc += u;
          }
          const int wpre = __shfl_sync(0xffffffffu, inc - v, warp);
          const int all = __shfl_sync(0xffffffffu, inc, 31);
          if (i < cnt) {
            const int pj = basecnt + wpre + __popc(m & ((1u << lane) - 1));
            preref(i) = pj;
            if (i == s) S.pre_s = pj;
          }
          basecnt += all;
          par ^= 1;
        }
        __syncthreads();
        pre_s = S.pre_s;
        tot_extra = basecnt;
      }
#pragma unroll kBpUnroll
      for (int i = tid; i < cnt; i += TPB) {
        const int k = kcref(i);
        if (k <= 0) continue;
        bool extra = false;
        if (rem > 0 && k > L) {
          int rank = preref(i) - pre_s;
          if (i < s) rank += tot_extra;
          extra = rank < rem;
        }
        const int mj = min(k, L) + (extra ? 1 : 0);
        if (mj > 0) {
          newly += applyfn(i, mj);
          // the pod placed last sits at the furthest position served in the final lap
          if (rem > 0 ? extra : (k >= L)) { int dd = i - s; if (dd < 0) dd += cnt; last_dist = max(last_dist, dd); }
        }
      }
      blk_sum_max<NW>(S, par, newly, last_dist);
    };

    // Group records travel one group ahead: warp 0 copies the next group's record into shared memory with cp.async
    // while the block works on the current one; the order row is read two entries ahead.
    const int32_t* order_row = FM ? nullptr : p.order + (size_t)t * p.E;   // FM: the runs in order
    auto fetch_rec = [&](int graw, int buf) {
      if (warp == 0) {
        const GroupRec* src = p.grec + (graw & ~ORDER_NOT_ON_FRESH);
        if (batch) {   // the simulation's own runs, then one run per pod moved in
          const int ro = sv(SIM_RUNS_OWN);
          src = graw < ro ? p.grec + sv(SIM_RUN0) + graw : p.sim_rec_pod + run_pod(sv(SIM_OWN_N) + graw - ro);
        }
        if (lane < 9) bp_cp_async16(reinterpret_cast<char*>(&S.rec[buf]) + lane * 16, reinterpret_cast<const char*>(src) + lane * 16);
        bp_cp_async_commit();
      }
    };
    // block-wide exclusive prefix of a per-node flag over x = 0..N-1 (ballots + one warp scan per TPB nodes); fn(x, rank)
    // is called for every x < N with the flag set; returns the count
    auto node_prefix = [&](auto flag, auto fn) -> int {
      int basecnt = 0;
      for (int base = 0; base < N; base += TPB) {
        const int x = base + tid;
        const bool ex = x < N && flag(x);
        const unsigned mm = __ballot_sync(0xffffffffu, ex);
        if (lane == 0) S.ri[par][warp][0] = __popc(mm);
        __syncthreads();
        const int v = lane < NW ? S.ri[par][lane][0] : 0;
        int inc = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
          const int u = __shfl_up_sync(0xffffffffu, inc, off);
          if (lane >= off) inc += u;
        }
        const int wpre = __shfl_sync(0xffffffffu, inc - v, warp);
        if (ex) fn(x, basecnt + wpre + __popc(mm & ((1u << lane) - 1)));
        basecnt += __shfl_sync(0xffffffffu, inc, 31);
        par ^= 1;
      }
      return basecnt;
    };

    for (;;) {   // candidates (a single filter pass runs once)
    if (batch) {
      // ---- next candidate: NoNodeInfo / not simulated / simulate (its pod list goes to the trace) ----
      if (sv(SIM_CAND) >= p.sim_n) break;
      __syncthreads();
      if (tid == 0) {
        const int cand = sv(SIM_CAND)++;
        const int c = p.sim_cand[cand], own0 = p.sim_pod_off[cand], own_n = p.sim_pod_off[cand + 1] - own0, trn = sv(SIM_TRN);
        int res = 3, moved = 0;   // 3 = simulate
        if (sv(SIM_CUT)) res = -1;
        else if (!p.sim_present[c] || p.sim_seen[c]) res = 2;   // removed by an earlier persisted simulation, or listed twice
        else {
          for (int q = p.sim_mv_head[c]; q >= 0; q = p.sim_mv_next[q]) ++moved;
          if ((long long)trn + own_n + moved > p.sim_trace_cap) res = 4;   // trace capacity: nothing is guessed
        }
        p.sim_trace_off[cand] = trn;
        if (res == 3) {
          p.sim_seen[c] = 1;
          p.sim_present[c] = 0;
          p.sim_gone[sv(SIM_NREM)] = c;
          int k = trn + own_n;   // pods placed on c by earlier persisted simulations follow its own pods, in placement order
          for (int q = p.sim_mv_head[c]; q >= 0; q = p.sim_mv_next[q]) { p.sim_trace_pod[k] = q; p.sim_trace_node[k] = -1; ++k; }
          sv(SIM_SEG) = trn; sv(SIM_TRN) = k;
          sv(SIM_RUN0) = p.sim_run_off[cand]; sv(SIM_RUNS_OWN) = p.sim_run_off[cand + 1] - p.sim_run_off[cand];
          sv(SIM_LOG0) = S.log_n;
        } else if (res != 4) p.sim_result[cand] = res;
        sv(SIM_RES) = res; sv(SIM_C) = c; sv(SIM_OWN0) = own0; sv(SIM_OWN_N) = own_n; sv(SIM_MOVED) = moved;
      }
      __syncthreads();
      const int res = sv(SIM_RES);
      if (res == 4) { if (tid == 0) atomicExch(p.status, 2); break; }
      if (res != 3) continue;
      {
        const int seg = sv(SIM_SEG), own0 = sv(SIM_OWN0), own_n = sv(SIM_OWN_N);
        for (int i = tid; i < own_n; i += TPB) { p.sim_trace_pod[seg + i] = p.sim_pods[own0 + i]; p.sim_trace_node[seg + i] = -1; }
      }
      // list positions of the nodes in the snapshot, and the node state to restore if the simulation does not stay
      const int ncur = node_prefix([&](int x) { return p.sim_present[x] != 0; }, [&](int x, int r) { p.sim_pos[x] = r; p.sim_at[r] = x; });
      for (int x = tid; x < N; x += TPB) {
        p.sim_nok[x] = p.sim_present[x] && (!p.sim_dest || p.sim_dest[x]);   // read back through fm_node_ok
#pragma unroll
        for (int a = 0; a < A; ++a) p.sim_bk_free[(size_t)a * N + x] = g_free[(size_t)a * Xg + x];
        p.sim_bk_slots[x] = g_slots[x];
        p.sim_bk_ports[x] = g_ports[x];
      }
      const int li = sv(SIM_LI);   // raw: a scan starts at lastIndex % (current list length)
      if (tid == 0) sv(SIM_NCUR) = ncur;
      last_index = ncur > 0 ? (int)((((long long)li % ncur) + ncur) % ncur) : 0;
      fm_moved = false; fm_stop = false; pods_total = 0;
      __syncthreads();
    }
    int ord_cur = n_groups() > 0 ? (FM ? 0 : order_row[0]) : 0, ord_next = n_groups() > 1 ? (FM ? 1 : order_row[1]) : 0;
    if (n_groups() > 0) fetch_rec(ord_cur, 0);
    if (warp == 0) bp_cp_async_wait();
    __syncthreads();

    for (int gi = 0; gi < n_groups(); ++gi) {
      const GroupRec& rc = S.rec[gi & 1];
      if (gi + 1 < n_groups()) fetch_rec(ord_next, (gi + 1) & 1);
      const int ord_next2 = gi + 2 < n_groups() ? (FM ? gi + 2 : order_row[gi + 2]) : 0;
      const int g = ord_cur & ~ORDER_NOT_ON_FRESH;
      int n = rc.n;
      const int spec = rc.spec;
      int64_t req[A1];
      float rinv[A1];
#pragma unroll
      for (int a = 0; a < A; ++a) { req[a] = rc.req[a]; rinv[a] = rc.rinv[a]; }
      const int sc = rc.sc;
      const int dc = rc.dc;
      const bool static_new = !(ord_cur & ORDER_NOT_ON_FRESH);
      const bool has_ports = (rc.flags & GREC_HAS_PORTS) != 0;
      const unsigned long long pconf = rc.pconf;  // port sets this pod collides with
      const unsigned long long pbit = rc.pbit;
      const bool feeds = (rc.flags & GREC_FEEDS) != 0;
      // FM: offset of the run in the pass's pod list (batch: own runs first, then the pods moved in, one run each)
      const int pb = !batch ? rc.pad[0] : gi < sv(SIM_RUNS_OWN) ? rc.pad[0] - sv(SIM_OWN0) : sv(SIM_OWN_N) + gi - sv(SIM_RUNS_OWN);
      bool can_existing = n_new > 0 && static_new && maxslots >= 1;   // some added node may still take this pod
#pragma unroll
      for (int a = 0; a < A; ++a) can_existing = can_existing && !(req[a] > 0 && req[a] > maxfree[a]);
      if (!FM && dc == 0 && can_existing) {
        for (int i = 0; i < n_dead; ++i) {
          bool dom = true;
#pragma unroll
          for (int a = 0; a < A; ++a) dom = dom && req[a] >= S.dead[i][a];
          if (dom) { can_existing = false; break; }
        }
      }
      int placed = 0;

      // spare capacity of node x for this pod by NodePorts + NodeResourcesFit alone (pod slots, free resources)
      auto res_cap_of = [&](auto frf, int slots, unsigned long long ports, int want) -> int {
        int k = min(slots, want);
        if (k > 0 && (ports & pconf)) k = 0;
#pragma unroll
        for (int a = 0; a < A; ++a) {
          if (req[a] > 0 && k > 0) {
            const int64_t f = frf(a);
            if (f < req[a]) k = 0;
            else if (f < (int64_t)k * req[a]) k = bp_div_f(f, req[a], rinv[a], k);
          }
        }
        if (has_ports) k = min(k, 1);
        return k;
      };
      auto res_cap_a = [&](int j, int want) -> int { return res_cap_of([&](int a) { return afr(a, j); }, asl(j), has_ports ? apo(j) : 0ull, want); };
      auto res_cap_c = [&](int x, int want) -> int { return res_cap_of([&](int a) { return cfr(a, x); }, csl(x), has_ports ? cpo(x) : 0ull, want); };
      // ForceAddPod x m on node x (owner thread); returns 1 when the node held no scheduled pod before
      auto book_a = [&](int j, int m) -> int {
#pragma unroll
        for (int a = 0; a < A; ++a) if (req[a] > 0) afr(a, j) -= (int64_t)m * req[a];
        asl(j) -= m;
        if (has_ports) apo(j) |= pbit;
        int nw = 0;
        if (!asch(j)) { asch(j) = 1; nw = 1; }
        if (feeds) log_append(Neff + j, spec, m);
        return nw;
      };
      auto book_c = [&](int x, int m) -> int {
#pragma unroll
        for (int a = 0; a < A; ++a) if (req[a] > 0) cfr(a, x) -= (int64_t)m * req[a];
        csl(x) -= m;
        if (has_ports) cpo(x) |= pbit;
        int nw = 0;
        if (!csch(x)) { csch(x) = 1; nw = 1; }
        if (feeds) log_append(x, spec, m);
        return nw;
      };
      // capacity of a FRESH node by NodePorts + NodeResourcesFit (DaemonSet port conflicts are part of static_new)
      auto fresh_cap = [&](int want) -> int {
        int k = 0;
        if (static_new) {
          k = min(tslots, want);
#pragma unroll
          for (int a = 0; a < A; ++a) {
            if (req[a] > 0 && k > 0) {
              if (tfree[a] < req[a]) k = 0;
              else if (tfree[a] < (int64_t)k * req[a]) k = bp_div_f(tfree[a], req[a], rinv[a], k);
            }
          }
          if (has_ports) k = min(k, 1);
        }
        return k;
      };
      // tryToScheduleOnNewNodes in closed form: every new node takes min(remaining, k_new) pods (k_new <= 0: the node
      // is added, the pod still fails on it, :235-240).  `one`: add a single node only (permission is asked once).
      auto add_new_nodes = [&](int k_new, bool one) {
        long long allowed = max_nodes < 0 ? 0 : (max_nodes == 0 ? (long long)INT_MAX : max((long long)max_nodes - n_new, 0ll));
        if (allowed > p.cap - n_new) allowed = p.cap - n_new;
        int add, fill = 0;
        if (k_new <= 0 || one) {
          add = allowed >= 1 ? 1 : 0;
          if (allowed < 1) new_nodes_available = false;   // PermissionToAddNode denied (:222)
          if (k_new > 0) fill = min(n, add * k_new);
        } else {
          const long long need = ((long long)n + k_new - 1) / k_new;
          if (need > allowed) { add = (int)allowed; new_nodes_available = false; }
          else add = (int)need;
          fill = (int)min((long long)n, (long long)add * k_new);
        }
        for (int i = tid; i < add; i += TPB) {
          const int j = n_new + i;
          const int mj = k_new <= 0 ? 0 : min(k_new, fill - i * k_new);
#pragma unroll
          for (int a = 0; a < A; ++a) afr(a, j) = tfree[a] - (req[a] > 0 ? (int64_t)mj * req[a] : 0);
          asl(j) = tslots - mj;
          apo(j) = mj > 0 ? pbit : 0ull;
          asch(j) = mj > 0;
          if (feeds && mj > 0) log_append(Neff + j, spec, mj);
        }
        if (k_new > 0) { nodes_with_pods += add; placed += fill; n -= fill; }
        n_new += add;
        if (add > 0) {
          n_dead = 0; dead_next = 0;
          maxslots = max(maxslots, tslots);
#pragma unroll
          for (int a = 0; a < A; ++a) maxfree[a] = max(maxfree[a], tfree[a]);
        }
        __syncthreads();
      };

      // SimilarPodsScheduling (similar_pods.go:59-104): a pod that fitted nowhere marks its (controller, spec) class, at most
      // 10 classes per controller; later pods of a marked class are not tried
      const int fm_cls = (FM && p.fm_class) ? p.fm_class[run_pod(pb)] : -1;
      bool fm_blocked = FM && fm_cls >= 0 && p.fm_class_mark[fm_cls] != 0;
      auto fm_mark_failed = [&]() {
        if (fm_cls < 0) return;
        const int ctrl = p.fm_class_ctrl[fm_cls];
        const int cnt = p.fm_ctrl_cnt[ctrl];
        __syncthreads();
        if (tid == 0) {
          if (cnt >= 10) p.fm_ctrl_over[ctrl] = 1;
          else { p.fm_ctrl_cnt[ctrl] = cnt + 1; p.fm_class_mark[fm_cls] = 1; }
        }
        if (cnt < 10) fm_blocked = true;
        __syncthreads();
      };
      // hinted pods are singleton runs; a pod moved in was placed on the candidate itself, so its hint names a node out of the list
      const int fm_hint = (FM && p.fm_hint && !(batch && gi >= sv(SIM_RUNS_OWN))) ? p.fm_hint[run_pod(pb)] : -1;
      auto fm_set = [&](int k, int x) {   // node of pod k of the list (run_pod)
        if (batch) p.sim_trace_node[sv(SIM_SEG) + k] = x;
        else p.fm_assigned[p.fm_pods[k]] = x;
      };
      // FM: deal m identical pods over the cluster nodes with capacities g_kc[x], lap by lap (lap l serves the nodes with
      // capacity >= l in cyclic order from lastIndex), reporting every pod's node; books the pods and moves lastIndex
      auto fm_deal = [&](int m) {
        const int s = node_at(last_index < Ncur() ? last_index : 0);
        for (int x = tid; x < N; x += TPB) g_aux[x] = 0;
        int done = 0, lap = 1;
        while (done < m) {
          int basecnt = 0;
          for (int base = 0; base < N; base += TPB) {
            const int x = base + tid;
            const bool ex = x < N && g_kc[x] >= lap;
            const unsigned mm = __ballot_sync(0xffffffffu, ex);
            if (lane == 0) S.ri[par][warp][0] = __popc(mm);
            __syncthreads();
            const int v = lane < NW ? S.ri[par][lane][0] : 0;
            int inc = v;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
              const int u = __shfl_up_sync(0xffffffffu, inc, off);
              if (lane >= off) inc += u;
            }
            const int wpre = __shfl_sync(0xffffffffu, inc - v, warp);
            const int all = __shfl_sync(0xffffffffu, inc, 31);
            if (x < N) {
              const int pj = basecnt + wpre + __popc(mm & ((1u << lane) - 1));
              g_pre[x] = pj;
              if (x == s) S.pre_s = pj;
            }
            basecnt += all;
            par ^= 1;
          }
          __syncthreads();
          const int pre_s = S.pre_s, tot = basecnt, take = min(tot, m - done);
          for (int x = tid; x < N; x += TPB) {
            if (g_kc[x] < lap) continue;
            int rank = g_pre[x] - pre_s;
            if (x < s) rank += tot;
            if (rank < take) {
              fm_set(pb + done + rank, x);
              g_aux[x] += 1;
              if (rank == take - 1) S.lastnode = x;
            }
          }
          done += take;
          ++lap;
          __syncthreads();
        }
        if (m > 0) {
          for (int x = tid; x < N; x += TPB) if (g_aux[x] > 0) book_c(x, g_aux[x]);
          last_index = (pos_of(S.lastnode) + 1) % Ncur();
          fm_moved = true;
          placed += m;
        }
        __syncthreads();
      };
      if (FM && dc == 0 && fm_hint < 0) {
        // ======================= plain run on the cluster nodes: dealt lap by lap ==================
        if (fm_stop || fm_blocked || Ncur() == 0) {
          if (p.fm_break && n > 0) fm_stop = true;     // every pod of the run stays unschedulable (breakOnFailure, :71-73)
        } else {
          int total = 0, zero = 0, zero2 = 0;
          const int clampv = n < (1 << 26) ? n + 1 : (1 << 26);
          for (int x = tid; x < N; x += TPB) {
            const bool ok = (p.pre_code[(size_t)sc * p.U + x] & 0x0F) == 0 && !o.node_unschedulable[x] && (!p.fm_node_ok || p.fm_node_ok[x]);
            const int k = ok ? res_cap_c(x, n) : 0;
            g_kc[x] = k;
            total = min(total + min(k, clampv), clampv);
          }
          blk_csum_max_sum<NW>(S, par, clampv, total, zero, zero2);
          const int m = min(n, total);     // pods that find a node
          fm_deal(m);
          if (m < n) {                      // the next pod fits nowhere: the identical pods behind it see the same state
            fm_mark_failed();
            if (p.fm_break) fm_stop = true;
          }
        }
      } else if (FM && dc == 0) {
        // ======================= hinted plain pod (singleton run) ==================================
        int where = -1;
        if (!fm_stop) {
          const int h = fm_hint;   // tryScheduleUsingHints (:80-106); lastIndex untouched
          if (h >= 0 && h < N && (!p.fm_node_ok || p.fm_node_ok[h]) && (p.pre_code[(size_t)sc * p.U + h] & 0x0F) == 0 && res_cap_c(h, 1) > 0) {
            __syncthreads();
            if (tid == 0) book_c(h, 1);
            __syncthreads();
            where = h;
            placed += 1;
          }
          if (where < 0 && !fm_blocked && Ncur() > 0) {   // SchedulePodOnAnyNodeMatching (:117): whole list, cyclic from lastIndex
            int best = INT_MAX, zero = 0;
            for (int x = tid; x < N; x += TPB) {
              if (o.node_unschedulable[x] || (p.fm_node_ok && !p.fm_node_ok[x]) || (p.pre_code[(size_t)sc * p.U + x] & 0x0F) != 0) continue;
              if (res_cap_c(x, 1) > 0) { int dd = pos_of(x) - last_index; if (dd < 0) dd += Ncur(); best = min(best, dd); }
            }
            blk_min_sum<NW>(S, par, best, zero);
            if (best != INT_MAX) {
              int hpos = last_index + best;
              if (hpos >= Ncur()) hpos -= Ncur();
              const int hit = node_at(hpos);
              if (tid == 0) book_c(hit, 1);
              __syncthreads();
              last_index = (hpos + 1) % Ncur();
              fm_moved = true;
              where = hit;
              placed += 1;
            } else fm_mark_failed();
          }
          if (where < 0 && p.fm_break) fm_stop = true;
        }
        if (tid == 0) fm_set(pb, where);
      } else if (dc == 0) {
        // ======================= plain group: closed form =======================================
        BP_PROF_COUNT(8, 1);
        BP_PROF_BEGIN();
        if (can_existing) {
          const int li0 = li_eff();
          const int s = li0 >= N ? li0 - N : 0;  // first added node in cyclic scan order
          int got, newly, last_dist;
          round_robin(n_new, s, n,
                      [&](int i) { return res_cap_a(i, n); },
                      [&](int i) -> int32_t& { return akc(i); },
                      [&](int i) -> int32_t& { return apr(i); },
                      [&](int i, int m) { return book_a(i, m); }, got, newly, last_dist);
          placed += got;
          nodes_with_pods += newly;
          n -= got;
          if (last_dist >= 0) {
            int jl = s + last_dist;
            if (jl >= n_new) jl -= n_new;
            last_index = (N + jl + 1) % (N + n_new);
          }
          if (got == 0) {
            refresh_bounds();
            if (!has_ports) {     // remember the dead request (ring of four)
#pragma unroll
              for (int a = 0; a < A; ++a) if (tid == a) S.dead[dead_next][a] = req[a];
              dead_next = (dead_next + 1) & 3;
              n_dead = min(n_dead + 1, 4);
              __syncthreads();
            }
          } else __syncthreads();
        }
        BP_PROF_END(0);
        BP_PROF_BEGIN();
        if (n > 0 && new_nodes_available) {
          // after the pass above no added node (the last one included) can take this pod any more
          const bool stop = (n_new > 0) && !asch(n_new - 1);  // last node still empty (:212)
          if (!stop) add_new_nodes(fresh_cap(n), false);
        }
        BP_PROF_END(1);
      } else if (!FM && !new_nodes_available && !can_existing) {
        // no node may be added any more and no added node has room: every pod of the group fails at once
      } else {
        // ======================= dynamic group ===================================================
        const bool host_spread = (rc.flags & GREC_HOST_SPREAD) != 0;
        const int gver = ++gver_ctr;      // version of this group's working counters (lazy copy-on-write)
        // ---- describe the group's counters ----
        BP_PROF_BEGIN();
        __syncthreads();
        {
          // warp 0, one lane per counter of the class: one 64-byte record + three template-dependent values each,
          // inactive counters are squeezed out with a ballot
          const int q0 = d.dc_q_off[dc], qn = d.dc_q_off[dc + 1] - q0;
          if (warp == 0) {
            QRec r{};
            int td = -1, en = 0, dsw = 0;
            const int q = q0 + lane;
            if (lane < qn) {
              const int4* src = reinterpret_cast<const int4*>(d.qrec + q);
              int4* dst = reinterpret_cast<int4*>(&r);
#pragma unroll
              for (int i = 0; i < 4; ++i) dst[i] = __ldg(src + i);
              if (!FM) {   // FM: no template, nothing is ever added
                td = d.dom[(size_t)r.k * NT + N + t];
                en = d.elig[(size_t)q * p.U + col_new];
                dsw = d.ds_w[(size_t)q * p.T + t];
              }
            }
            const unsigned act = __ballot_sync(0xffffffffu, lane < qn && r.active);
            if (lane < qn && r.active) {
              const int i = __popc(act & ((1u << lane) - 1));
              wd.qid[i] = q; wd.kind[i] = r.kind; wd.k[i] = r.k; wd.host[i] = r.host; wd.Dc[i] = r.Dc;
              wd.tslot[i] = td < 0 ? -1 : (td < r.Dc ? td : r.Dc);
              wd.wown[i] = r.wown; wd.self[i] = r.self; wd.maxskew[i] = r.maxskew; wd.mindom[i] = r.mindom;
              wd.elig_new[i] = en; wd.dsw[i] = dsw; wd.tot[i] = r.base_tot; wd.boff[i] = r.boff;
              wd.minv[i] = r.st_min1; wd.nmin[i] = r.st_nmin; wd.ndom[i] = r.st_ndom;
              wd.nfeed[i] = r.nfeed;
              S.flag[i] = 0;
            }
            if (lane == 0) { wd.nq = __popc(act); wd.aff_self = d.dc_aff_self[dc]; S.need_log = 0; }
          }
        }
        __syncthreads();
        const int nq = wd.nq;
        auto slot_of = [&](int q, int x) -> int {
          if (x < Neff) return d.dom[(size_t)wd.k[q] * NT + x];
          if (wd.host[q]) return wd.Dc[q] + 1 + (x - Neff);
          return wd.tslot[q];
        };
        auto elig_of = [&](int q, int x) -> bool {
          return x < Neff ? d.elig[(size_t)wd.qid[q] * p.U + x] != 0 : wd.elig_new[q] != 0;
        };
        // Working counters are copy-on-write over the cluster base counts: a slot is valid only when its
        // version equals this group's, otherwise it reads as its default (base count for cluster domains,
        // DaemonSet weight for the fresh hostname domain of an added node, 0 for a template-only value).
        auto def_cnt = [&](int q, int sl) -> int {
          const int Dc = wd.Dc[q];
          return sl < Dc ? d.base_cnt[wd.boff[q] + sl] : (sl == Dc ? 0 : (wd.elig_new[q] ? wd.dsw[q] : 0));
        };
        auto def_pres = [&](int q, int sl) -> int {
          const int Dc = wd.Dc[q];
          return sl < Dc ? d.base_pres[wd.boff[q] + sl] : (sl == Dc ? 0 : (wd.elig_new[q] ? 1 : 0));
        };
        auto rd_cnt = [&](int q, int sl) -> int {
          const size_t o2 = (size_t)q * p.dstride + sl;
          if (wver[o2] == gver) return wcnt[o2];
          return def_cnt(q, sl);
        };
        auto rd_pres = [&](int q, int sl) -> int {
          const size_t o2 = (size_t)q * p.dstride + sl;
          if (wver[o2] == gver) return wpres[o2];
          return def_pres(q, sl);
        };
        auto wr = [&](int q, int sl, int c, int prs) {  // single thread
          const size_t o2 = (size_t)q * p.dstride + sl;
          wcnt[o2] = c; wpres[o2] = prs; wver[o2] = gver;
        };
        // min / #domains over the present domains of a spread counter (block-wide; ends with a barrier)
        auto recompute = [&](int q) {
          const int len = wd.Dc[q] + 1 + (wd.host[q] ? n_new : 0);
          int mn = INT_MAX, nd = 0;
          for (int i = tid; i < len; i += TPB) if (rd_pres(q, i) > 0) { mn = min(mn, rd_cnt(q, i)); ++nd; }
          blk_min_sum<NW>(S, par, mn, nd);
          int nm = 0, zero = 0;
          for (int i = tid; i < len; i += TPB) if (rd_pres(q, i) > 0 && rd_cnt(q, i) == mn) ++nm;
          blk_min_sum<NW>(S, par, zero, nm);
          if (tid == 0) { wd.minv[q] = mn; wd.nmin[q] = nm; wd.ndom[q] = nd; S.flag[q] = 0; }
          __syncthreads();
        };
        auto run_flagged = [&]() {   // after a barrier: recompute the counters thread 0 flagged
          for (int q = 0; q < nq; ++q) if (S.flag[q]) recompute(q);
        };
        // ---- seed: nodes added so far (O(1) per counter) ----
        if (tid == 0) {
          int need_log = 0;
          for (int q = 0; q < nq; ++q) {
            if (wd.elig_new[q] && n_new > 0) {
              const int dsw = wd.dsw[q];
              if (wd.host[q]) {  // n_new fresh hostname domains, each holding the DaemonSet weight
                wd.tot[q] += n_new * dsw;
                if (wd.kind[q] == Q_PTS) {
                  wd.ndom[q] += n_new;
                  if (dsw < wd.minv[q]) { wd.minv[q] = dsw; wd.nmin[q] = n_new; }
                  else if (dsw == wd.minv[q]) wd.nmin[q] += n_new;
                }
              } else if (wd.tslot[q] >= 0) {  // all added nodes share the template's value of this key
                const int sl = wd.tslot[q];
                const int c0 = rd_cnt(q, sl), p0 = rd_pres(q, sl), c1 = c0 + n_new * dsw;
                wr(q, sl, c1, p0 + n_new);
                wd.tot[q] += n_new * dsw;
                if (wd.kind[q] == Q_PTS && p0 == 0) {
                  wd.ndom[q] += 1;
                  if (c1 < wd.minv[q]) { wd.minv[q] = c1; wd.nmin[q] = 1; }
                  else if (c1 == wd.minv[q]) wd.nmin[q] += 1;
                }
                if (wd.kind[q] == Q_PTS && p0 > 0 && dsw > 0) S.flag[q] = 1;
              }
            }
            if (FM || wd.nfeed[q] - (wd.wown[q] > 0 ? 1 : 0) > 0) need_log = 1;   // FM: earlier runs of this very spec count too
          }
          S.need_log = need_log;
        }
        __syncthreads();
        run_flagged();
        const bool need_log = S.need_log != 0;
        // ---- then the run's placement log if other groups feed us, and (batch) the nodes out of the list ----
        if ((need_log && S.log_n > 0) || batch) {
          const int nlog = min(S.log_n, p.log_cap);
          for (int q = 0; q < nq; ++q) {
            const int qid = wd.qid[q];
            // Pass 1 materialises the touched copy-on-write slots with their defaults (identical values from
            // every thread), pass 2 stamps the version and adds the weights atomically.  Batch: a placement logged on a
            // node out of the list no longer counts; a node out of the list takes its residents' weights and one eligible
            // node from its domain.
            int touched = 0;
            long long dt = 0;
            auto gone_w = [&](int x) -> int {
              int w = 0;
              for (int r = o.node_pod_off[x]; r < o.node_pod_off[x + 1]; ++r) w += d.wmat[(size_t)qid * d.S + o.node_pod_spec[r]];
              return w;
            };
            for (int i = tid; i < nlog; i += TPB) {
              const int x = logbuf[i * 3];
              const int w = d.wmat[(size_t)qid * d.S + logbuf[i * 3 + 1]];
              if (w == 0 || !elig_of(q, x) || (batch && !p.sim_present[x])) continue;
              const int sl = slot_of(q, x);
              if (sl < 0) continue;
              const size_t o2 = (size_t)q * p.dstride + sl;
              if (wver[o2] != gver) { wcnt[o2] = def_cnt(q, sl); wpres[o2] = def_pres(q, sl); }
              touched = 1;
              dt += w * logbuf[i * 3 + 2];
            }
            if (batch) {
              for (int i = tid; i <= sv(SIM_NREM); i += TPB) {   // the removed nodes, then the candidate
                const int x = p.sim_gone[i];
                if (!elig_of(q, x)) continue;
                const int sl = slot_of(q, x);
                if (sl < 0) continue;
                const size_t o2 = (size_t)q * p.dstride + sl;
                if (wver[o2] != gver) { wcnt[o2] = def_cnt(q, sl); wpres[o2] = def_pres(q, sl); }
                dt -= gone_w(x);
              }
            }
            __syncthreads();
            for (int i = tid; i < nlog; i += TPB) {
              const int x = logbuf[i * 3];
              const int w = d.wmat[(size_t)qid * d.S + logbuf[i * 3 + 1]];
              if (w == 0 || !elig_of(q, x) || (batch && !p.sim_present[x])) continue;
              const int sl = slot_of(q, x);
              if (sl < 0) continue;
              const size_t o2 = (size_t)q * p.dstride + sl;
              wver[o2] = gver;
              atomicAdd(&wcnt[o2], w * logbuf[i * 3 + 2]);
            }
            if (batch) {
              for (int i = tid; i <= sv(SIM_NREM); i += TPB) {   // the removed nodes, then the candidate
                const int x = p.sim_gone[i];
                if (!elig_of(q, x)) continue;
                const int sl = slot_of(q, x);
                if (sl < 0) continue;
                const size_t o2 = (size_t)q * p.dstride + sl;
                wver[o2] = gver;
                atomicAdd(&wcnt[o2], -gone_w(x));
                atomicAdd(&wpres[o2], -1);
              }
            }
            blk_sum_ll_max<NW>(S, par, dt, touched);
            if (tid == 0) wd.tot[q] += (int)dt;
            __syncthreads();
            if ((touched > 0 || batch) && wd.kind[q] == Q_PTS) recompute(q);
          }
        }

        BP_PROF_END(2);
        // ---- capacity form: every counter of the group is either a per-node capacity or a budget ----
        // Hostname counters (each node is its own domain): a spread constraint whose global minimum is pinned at 0
        // admits (maxSkew - self - count) / weight + 1 pods on a node, an anti-affinity / existing-anti-affinity
        // counter one pod (none if the domain already holds a match).  Counters on any other key see ONE domain for
        // all added nodes (the template's value), so they bound the number of pods the group can place at all.
        // Then the per-pod loop of the reference is the round-robin closed form over capacities, cut at the budget.
        BP_PROF_BEGIN();
        bool fast = false;
        {
          int hp = -1;           // the hostname spread constraint, if any
          bool any_z = false, ok = true;
          for (int q = 0; q < nq; ++q) {
            if (wd.host[q]) {
              if (wd.kind[q] == Q_PTS) { if (hp >= 0) ok = false; hp = q; }
              else if (wd.kind[q] == Q_AFF) ok = false;
            } else any_z = true;
          }
          // the fallback of :186-205 places onto cluster nodes, whose other-key domains differ: per-pod loop
          if (hp >= 0 && (any_z || wd.minv[hp] != 0)) ok = false;
          if (FM && (any_z || fm_hint >= 0)) ok = false;   // other-key domains differ between cluster nodes / hinted pod: one by one
          // capacity a hostname counter puts on a node whose domain (slot sl, -1 = label missing) holds c matches
          auto hq_cap = [&](int q, int sl, int c, bool counted) -> int {
            if (wd.kind[q] == Q_PTS) {
              if (sl < 0) return 0;                                          // filtering.go:329 missing label
              if (c + wd.self[q] > wd.maxskew[q]) return 0;                  // filtering.go:352 with minMatchNum = 0
              if (!counted) return INT_MAX;
              return (wd.maxskew[q] - wd.self[q] - c) / wd.wown[q] + 1;
            }
            if (sl >= 0 && c > 0) return 0;                                  // interpodaffinity/filtering.go:352-379
            return (counted && sl >= 0) ? 1 : INT_MAX;
          };
          // caps of node x (any node of the simulation) from the hostname counters, spread and inter-pod apart
          auto h_caps = [&](int x, int& cap_pts, int& cap_ipa) {
            cap_pts = INT_MAX; cap_ipa = INT_MAX;
            for (int q = 0; q < nq; ++q) {
              if (!wd.host[q]) continue;
              const int sl = slot_of(q, x);
              const int c = sl >= 0 ? rd_cnt(q, sl) : 0;
              const int v = hq_cap(q, sl, c, wd.wown[q] > 0 && elig_of(q, x));
              if (wd.kind[q] == Q_PTS) cap_pts = v; else cap_ipa = min(cap_ipa, v);
            }
          };
          // a FRESH node reads the defaults of its new hostname domain
          int Spts_new = INT_MAX, Sipa_new = INT_MAX;
          for (int q = 0; q < nq; ++q) {
            if (!wd.host[q]) continue;
            const int v = hq_cap(q, 0, wd.elig_new[q] ? wd.dsw[q] : 0, wd.wown[q] > 0 && wd.elig_new[q]);
            if (wd.kind[q] == Q_PTS) Spts_new = v; else Sipa_new = min(Sipa_new, v);
          }
          // ---- budget of the other-key counters (uniform: all added nodes sit in the template's domain) ----
          int B = INT_MAX;
          if (ok && any_z) {
            bool aff_any = false, pods_exist = true, aff_missing = false;
            long long aff_tot = 0;
            for (int q = 0; q < nq && ok; ++q) {
              if (wd.host[q]) continue;
              const int kind = wd.kind[q], sl = wd.tslot[q], w = wd.wown[q];
              const int c = sl >= 0 ? rd_cnt(q, sl) : 0;
              const bool counted = w > 0 && wd.elig_new[q] && sl >= 0;
              if (wd.elig_new[q] && wd.dsw[q] != 0) { ok = false; break; }   // adding a node moves the counter (DaemonSet pods match)
              if (kind == Q_PTS) {
                // ANY spread constraint refusing the last node sends a pod that names the hostname key in some constraint
                // (even a ScheduleAnyway one) through the any-node fallback of :186-205: per-pod loop
                if (host_spread) { ok = false; break; }
                if (sl < 0) { B = 0; continue; }
                const int prs = rd_pres(q, sl), self = wd.self[q], ms = wd.maxskew[q];
                if (wd.elig_new[q] && prs == 0) { ok = false; break; }         // the domain appears with the first added node
                long long lim;    // placements pass while count <= lim
                if (wd.ndom[q] < wd.mindom[q]) lim = (long long)ms - self;                       // minimum treated as 0
                else if (prs > 0) {
                  // minimum over the OTHER present domains (constant while this group runs)
                  if (c > wd.minv[q] || wd.nmin[q] > 1) lim = (long long)wd.minv[q] + ms - self;
                  else if (wd.ndom[q] == 1) lim = LLONG_MAX;                                     // the only domain: skew 0
                  else { ok = false; break; }                                                    // unique minimum: needs the runner-up
                  if (self > ms) lim = -1;
                } else lim = wd.ndom[q] == 0 ? LLONG_MAX : (long long)wd.minv[q] + ms - self;    // domain not counted at all
                if (c > lim) B = 0;
                else if (counted && lim != LLONG_MAX) B = (int)min((long long)B, (lim - c) / w + 1);
              } else if (kind == Q_AFF) {
                aff_any = true;
                if (sl < 0) aff_missing = true;
                if (c <= 0) pods_exist = false;
                aff_tot += wd.tot[q];
              } else {
                if (sl >= 0 && c > 0) B = 0;
                else if (counted) B = min(B, 1);
              }
            }
            if (ok && aff_any) {
              if (aff_missing) B = 0;
              else if (!pods_exist) { if (aff_tot == 0 && wd.aff_self) ok = false; else B = 0; }   // first-pod escape hatch: per-pod loop
            }
          }
          bool caps_done = false;
          // capacities of the cluster nodes for this pod (static filters, ports, resources, hostname counters) -> kc[x];
          // returns "a present empty domain of the spread constraint exists whose only eligible node can never take this pod"
          auto cluster_caps = [&]() -> bool {
            ensure_cluster();
            int blocked = 0;
            for (int x = tid; x < N; x += TPB) {
              const bool stat_ok = (p.pre_code[(size_t)sc * p.U + x] & 0x0F) == 0 && !o.node_unschedulable[x] &&
                                   !(FM && p.fm_node_ok && !p.fm_node_ok[x]);
              const int rc = stat_ok ? res_cap_c(x, n) : 0;
              int cp, ci;
              h_caps(x, cp, ci);
              const int k_other = min(rc, ci);
              g_kc[x] = min(k_other, cp);
              if (k_other == 0 && hp >= 0 && !(batch && !p.sim_present[x])) {
                const int sl = slot_of(hp, x);
                if (sl >= 0 && elig_of(hp, x) && rd_cnt(hp, sl) == 0 && rd_pres(hp, sl) == 1) blocked = 1;
              }
            }
            long long z = 0;
            blk_sum_ll_max<NW>(S, par, z, blocked);
            caps_done = true;
            BP_PROF_COUNT(14, 1);
            return blocked > 0;
          };
          if (ok && hp >= 0 && !(wd.wown[hp] == 0 || wd.nmin[hp] > n)) ok = Ncur() > 0 ? cluster_caps() : false;   // is the minimum pinned?
          if (FM && ok) {
            // hostname counters only: per-node capacities over the cluster nodes, dealt like a plain run
            fast = true;
            if (fm_stop || fm_blocked || Ncur() == 0) {
              if (p.fm_break && n > 0) fm_stop = true;
            } else {
              if (!caps_done) cluster_caps();
              const int clampv = n < (1 << 26) ? n + 1 : (1 << 26);
              int total = 0, zero = 0, zero2 = 0;
              for (int x = tid; x < N; x += TPB) total = min(total + min(g_kc[x], clampv), clampv);
              blk_csum_max_sum<NW>(S, par, clampv, total, zero, zero2);
              const int m = min(n, total);
              fm_deal(m);
              if (m < n) {
                fm_mark_failed();
                if (p.fm_break) fm_stop = true;
              }
            }
          } else if (ok) {
            fast = true;
            const bool uni = !need_log;   // no other group feeds these counters: every added node reads the defaults
            int b = B;                    // pods the budget still admits
            int m_last = 0;               // pods of this group on the last added node
            const int S_new = min(Spts_new, Sipa_new);
            // ---- tryToScheduleOnExistingNodes ----
            if (can_existing && min(n, b) > 0 && (!uni || S_new > 0)) {
              if (tid == 0) S.mlast = 0;
              const int li0 = li_eff();
              const int s = li0 >= N ? li0 - N : 0;
              const int lastj = n_new - 1, want = min(n, b);
              int got, newly, last_dist;
              round_robin(n_new, s, want,
                          [&](int i) {
                            const int k = res_cap_a(i, want);
                            if (k <= 0) return 0;
                            if (uni) return min(k, S_new);
                            int cp, ci;
                            h_caps(Neff + i, cp, ci);
                            return min(k, min(cp, ci));
                          },
                          [&](int i) -> int32_t& { return akc(i); },
                          [&](int i) -> int32_t& { return apr(i); },
                          [&](int i, int m) { if (i == lastj) S.mlast = m; return book_a(i, m); }, got, newly, last_dist);
              placed += got;
              nodes_with_pods += newly;
              n -= got;
              if (b != INT_MAX) b -= got;
              if (last_dist >= 0) {
                int jl = s + last_dist;
                if (jl >= n_new) jl -= n_new;
                last_index = (N + jl + 1) % (N + n_new);
              }
              if (got == 0) refresh_bounds(); else __syncthreads();
              m_last = S.mlast;
            }
            // the pods the last node refuses for skew go to the cluster nodes in cyclic order (:186-205)
            auto cluster_phase = [&]() {
              if (N == 0) return;
              BP_PROF_COUNT(15, 1);
              if (!caps_done) cluster_caps();
              const int li0 = li_eff();
              const int s = li0 < N ? li0 : 0;
              int got, newly, last_dist;
              round_robin(N, s, n,
                          [&](int i) { return g_kc[i]; },
                          [&](int i) -> int32_t& { return g_kc[i]; },
                          [&](int i) -> int32_t& { return g_pre[i]; },
                          [&](int i, int m) { return book_c(i, m); }, got, newly, last_dist);
              placed += got;
              nodes_with_pods += newly;
              n -= got;
              if (last_dist >= 0) {
                int jl = s + last_dist;
                if (jl >= N) jl -= N;
                last_index = jl + 1;   // < N + n_new: the list holds at least one added node here
              }
              __syncthreads();
            };
            // ---- tryToScheduleOnNewNodes ----
            if (n > 0 && new_nodes_available) {
              bool cluster_done = false;
              if (hp >= 0 && host_spread && n_new > 0) {
                // why the last node refuses the next pod (default plugin order): static, ports, fit, then skew
                const int jl = n_new - 1;
                bool skew = static_new && !(apo(jl) & pconf) && asl(jl) >= 1;
#pragma unroll
                for (int a = 0; a < A; ++a) skew = skew && !(req[a] > 0 && req[a] > afr(a, jl));
                const int c_last = uni ? (wd.elig_new[hp] ? wd.dsw[hp] : 0) : rd_cnt(hp, slot_of(hp, Neff + jl));
                skew = skew && (c_last + (wd.elig_new[hp] ? m_last * wd.wown[hp] : 0) + wd.self[hp] > wd.maxskew[hp]);
                if (skew) { cluster_phase(); cluster_done = true; }
              }
              if (n > 0) {
                const bool stop = (n_new > 0) && !asch(n_new - 1);  // last node still empty (:212)
                const int npl = min(n, b);                          // pods the budget still admits
                if (stop) {
                } else if (npl == 0) {
                  add_new_nodes(0, false);             // the node is added, the pod fails on it (:235-240)
                } else {
                  const int k_new = min(fresh_cap(npl), S_new);
                  // a full fresh node refuses the next pod for skew iff the skew capacity binds before ports / fit / inter-pod affinity
                  const bool fresh_skew = hp >= 0 && k_new > 0 && Spts_new < fresh_cap(INT_MAX) && Spts_new <= Sipa_new;
                  const int n_all = n;
                  n = npl;
                  if (fresh_skew && host_spread && !cluster_done) {
                    add_new_nodes(k_new, true);        // the first fresh node fills ...
                    if (n > 0 && new_nodes_available) {
                      cluster_phase();                 // ... then the fallback drains the cluster nodes ...
                      if (n > 0) add_new_nodes(k_new, false);   // ... and further nodes take the rest
                    }
                  } else add_new_nodes(k_new, false);
                  const int done = npl - n;
                  n = n_all - done;
                  if (b != INT_MAX) b -= done;
                  // the budget ran out with pods left: the next pod fails on the last node and on one more fresh node
                  if (k_new > 0 && n > 0 && b == 0 && new_nodes_available && n_new > 0 && asch(n_new - 1)) add_new_nodes(0, false);
                }
              }
            }
          }
        }
        if (fast) { BP_PROF_END(4); BP_PROF_COUNT(9, 1); }
        if (!fast) {
        BP_PROF_COUNT(10, 1);
        // ======================= per-pod loop on incremental counters =============================
        // RunFilterPlugins on node x (default plugin order), per thread
        auto eval = [&](int x) -> int {
          const int col = x < Neff ? x : col_new;
          const int code = p.pre_code[(size_t)sc * p.U + col] & 0x0F;
          if (code) return code;
          if (po(x) & pconf) return CAE_R_NODE_PORTS;
          bool fail = sl_(x) < 1;
#pragma unroll
          for (int a = 0; a < A; ++a) fail |= (req[a] > 0 && req[a] > fr(a, x));
          if (fail) return CAE_R_FIT;
          bool aff_any = false, pods_exist = true;
          long long aff_tot = 0;
          for (int q = 0; q < nq; ++q) {
            const int kind = wd.kind[q];
            const int sl = slot_of(q, x);
            const int c = sl >= 0 ? rd_cnt(q, sl) : 0;
            if (kind == Q_PTS) {  // podtopologyspread/filtering.go:314-359
              if (sl < 0) return CAE_R_PTS_MISSING_LABEL;
              const long long minm = wd.ndom[q] < wd.mindom[q] ? 0 : wd.minv[q];
              if ((long long)c + wd.self[q] - minm > wd.maxskew[q]) return CAE_R_PTS_SKEW;
            } else if (kind == Q_AFF) {  // interpodaffinity/filtering.go:382-408
              aff_any = true;
              if (sl < 0) return CAE_R_IPA_AFFINITY;
              if (c <= 0) pods_exist = false;
              aff_tot += wd.tot[q];
            } else {
              if (aff_any) {
                if (!pods_exist && !(aff_tot == 0 && wd.aff_self)) return CAE_R_IPA_AFFINITY;
                aff_any = false;
              }
              if (sl >= 0 && c > 0) return kind == Q_ANTI ? CAE_R_IPA_ANTI_AFFINITY : CAE_R_IPA_EXISTING_ANTI_AFFINITY;
            }
          }
          if (aff_any && !pods_exist && !(aff_tot == 0 && wd.aff_self)) return CAE_R_IPA_AFFINITY;
          return CAE_R_OK;
        };
        // ForceAddPod on node x (uniform x) + counter upkeep
        auto place = [&](int x) {
          __syncthreads();   // every thread has finished evaluating against the old state
          if (tid == 0) {
            S.newly = !sch(x);
#pragma unroll
            for (int a = 0; a < A; ++a) if (req[a] > 0) fr(a, x) -= req[a];
            sl_(x) -= 1;
            po(x) |= pbit;
            sch(x) = 1;
            for (int q = 0; q < nq; ++q) {
              const int w = wd.wown[q];
              if (w == 0 || !elig_of(q, x)) continue;
              const int sl = slot_of(q, x);
              if (sl < 0) continue;
              const int old = rd_cnt(q, sl), prs = rd_pres(q, sl);
              wr(q, sl, old + w, prs);
              wd.tot[q] += w;
              if (wd.kind[q] == Q_PTS && old == wd.minv[q]) {
                if (--wd.nmin[q] == 0) S.flag[q] = 1;
              }
            }
            if (feeds) log_append(x, spec, 1);
          }
          __syncthreads();
          if (S.newly) ++nodes_with_pods;
          run_flagged();
          ++placed;
          --n;
        };
        // addNewNodeToSnapshot (:249-265): a sanitized copy of the template joins the list
        auto add_node = [&]() {
          const int x = Neff + n_new;
          __syncthreads();
          if (tid == 0) {
#pragma unroll
            for (int a = 0; a < A; ++a) fr(a, x) = tfree[a];
            sl_(x) = tslots;
            po(x) = 0ull;
            sch(x) = 0;
            for (int q = 0; q < nq; ++q) {
              const int en = wd.elig_new[q], dsw = wd.dsw[q];
              const int sl = slot_of(q, x);
              const bool pts = wd.kind[q] == Q_PTS;
              if (wd.host[q]) {  // a brand-new hostname domain (its default already reads dsw / present)
                if (en) {
                  wd.tot[q] += dsw;
                  if (pts) {
                    wd.ndom[q] += 1;
                    if (dsw < wd.minv[q]) { wd.minv[q] = dsw; wd.nmin[q] = 1; }
                    else if (dsw == wd.minv[q]) wd.nmin[q] += 1;
                  }
                }
              } else if (en && sl >= 0) {
                const int c0 = rd_cnt(q, sl), p0 = rd_pres(q, sl);
                wr(q, sl, c0 + dsw, p0 + 1);
                wd.tot[q] += dsw;
                if (pts && p0 == 0) {
                  wd.ndom[q] += 1;
                  if (c0 + dsw < wd.minv[q]) { wd.minv[q] = c0 + dsw; wd.nmin[q] = 1; }
                  else if (c0 + dsw == wd.minv[q]) wd.nmin[q] += 1;
                }
                if (pts && p0 > 0 && dsw > 0) S.flag[q] = 1;
              }
            }
          }
          n_new += 1;       // recompute() below must see the new node's hostname domain
          n_dead = 0; dead_next = 0;
          maxslots = max(maxslots, tslots);
#pragma unroll
          for (int a = 0; a < A; ++a) maxfree[a] = max(maxfree[a], tfree[a]);
          __syncthreads();
          run_flagged();
        };

        if constexpr (FM) {
          // ---- HintingSimulator.TrySchedulePods over the cluster nodes, pod by pod ----
          const int run_n = n;
          bool run_failed = false;  // a pod of this run fitted nowhere: the identical pods behind it see the same state
          for (int i = 0; i < run_n; ++i) {
            int where = -1;
            if (!fm_stop) {
              const int h = fm_hint;   // tryScheduleUsingHints (:80-106); lastIndex untouched.  Only singleton runs carry a hint
              if (h >= 0 && h < N && (!p.fm_node_ok || p.fm_node_ok[h]) && eval(h) == CAE_R_OK) { place(h); where = h; }
              if (where < 0 && !fm_blocked && !run_failed && Ncur() > 0) {
                // SchedulePodOnAnyNodeMatching (:117): whole list, cyclic from lastIndex
                int best = INT_MAX, zero = 0;
                for (int x = tid; x < N; x += TPB) {
                  if (o.node_unschedulable[x] || (p.fm_node_ok && !p.fm_node_ok[x])) continue;
                  if (eval(x) == CAE_R_OK) { int dd = pos_of(x) - last_index; if (dd < 0) dd += Ncur(); best = min(best, dd); }
                }
                blk_min_sum<NW>(S, par, best, zero);
                if (best != INT_MAX) {
                  int hpos = last_index + best;
                  if (hpos >= Ncur()) hpos -= Ncur();
                  const int hit = node_at(hpos);
                  place(hit);
                  last_index = (hpos + 1) % Ncur();
                  fm_moved = true;
                  where = hit;
                } else {
                  run_failed = true;
                  fm_mark_failed();
                }
              }
              if (where < 0 && p.fm_break) fm_stop = true;   // breakOnFailure (:71-73)
            }
            if (tid == 0) fm_set(pb + i, where);
          }
        } else {
        // ---- tryToScheduleOnExistingNodes: per pod, first passing added node in cyclic order ----
        BP_PROF_BEGIN();
        while (n > 0 && can_existing) {
          BP_PROF_COUNT(12, 1);
          const int li0 = li_eff();
          const int s = li0 >= N ? li0 - N : 0;
          int best = INT_MAX, zero = 0;
          for (int j = tid; j < n_new; j += TPB)
            if (eval(Neff + j) == CAE_R_OK) { int dd = j - s; if (dd < 0) dd += n_new; best = min(best, dd); }
          blk_min_sum<NW>(S, par, best, zero);
          if (best == INT_MAX) break;  // first pod that fits nowhere ends this phase for the group (:158)
          int found = s + best;
          if (found >= n_new) found -= n_new;
          place(Neff + found);
          last_index = (N + found + 1) % (N + n_new);
        }
        BP_PROF_END(5);
        BP_PROF_BEGIN();
        // ---- tryToScheduleOnNewNodes ----
        while (n > 0 && new_nodes_available) {
          BP_PROF_COUNT(13, 1);
          bool found = false;
          if (n_new > 0) {
            const int xl = Neff + n_new - 1;
            const int r = eval(xl);
            if (r == CAE_R_OK) { place(xl); found = true; }
            else if (host_spread && r == CAE_R_PTS_SKEW) {
              // SchedulePodOnAnyNodeMatching(name != lastNodeName) (:190-205): whole list, cyclic from lastIndex
              ensure_cluster();
              const int len = N + n_new, lastpos = N + n_new - 1, li0 = li_eff();
              int best = INT_MAX, zero = 0;
              for (int idx = tid; idx < len; idx += TPB) {
                if (idx == lastpos) continue;
                if (idx < N && o.node_unschedulable[idx]) continue;   // plugin_runner.go:92-94
                const int x = idx < N ? idx : Neff + (idx - N);
                if (eval(x) == CAE_R_OK) { int dd = idx - li0; if (dd < 0) dd += len; best = min(best, dd); }
              }
              blk_min_sum<NW>(S, par, best, zero);
              if (best != INT_MAX) {
                int hit = li0 + best;
                if (hit >= len) hit -= len;
                place(hit < N ? hit : Neff + (hit - N));
                last_index = (hit + 1) % len;
                found = true;
              }
            }
          }
          if (!found) {
            if (n_new > 0 && !sch(Neff + n_new - 1)) break;  // last node still empty (:212)
            const bool permit = !(max_nodes < 0 || (max_nodes > 0 && n_new >= max_nodes)) && n_new < p.cap;
            if (!permit) { new_nodes_available = false; break; }  // (:222)
            add_node();
            if (eval(Neff + n_new - 1) != CAE_R_OK) break;  // (:238-240)
            place(Neff + n_new - 1);
          }
        }
        BP_PROF_END(6);
        BP_PROF_COUNT(11, placed);
        }  // !FM
        }  // !fast
      }
      pods_total += placed;
      if (!FM && tid == 0) p.sched[(size_t)t * p.E + g] = placed;
      if (warp == 0) bp_cp_async_wait();   // the next group's record has landed
      __syncthreads();
      ord_cur = ord_next;
      ord_next = ord_next2;
      if (batch && fm_stop) break;         // breakOnFailure: the pods behind stay unplaced (-1 in the trace)
    }
    if (batch) {
      // ---- end of the candidate: removable iff every pod was placed; keep it (persist) or undo it ----
      const bool removable = pods_total == sv(SIM_OWN_N) + sv(SIM_MOVED);
      if (removable && p.sim_persist) {
        if (tid == 0) {   // the pods now live where they were placed: append them there, in placement order
          p.sim_mv_head[sv(SIM_C)] = -1;
          for (int k = sv(SIM_SEG); k < sv(SIM_TRN); ++k) {
            const int q = p.sim_trace_pod[k], x = p.sim_trace_node[k];
            p.sim_mv_next[q] = -1;
            if (p.sim_mv_head[x] < 0) p.sim_mv_head[x] = q;
            else p.sim_mv_next[p.sim_mv_tail[x]] = q;
            p.sim_mv_tail[x] = q;
          }
          sv(SIM_NREM) += 1;
        }
      } else {
        for (int x = tid; x < N; x += TPB) {
#pragma unroll
          for (int a = 0; a < A; ++a) g_free[(size_t)a * Xg + x] = p.sim_bk_free[(size_t)a * N + x];
          g_slots[x] = p.sim_bk_slots[x];
          g_ports[x] = p.sim_bk_ports[x];
        }
        if (tid == 0) { S.log_n = sv(SIM_LOG0); p.sim_present[sv(SIM_C)] = 1; }
      }
      if (tid == 0) {
        if (fm_moved) sv(SIM_LI) = last_index;   // the runner's lastIndex survives the revert
        p.sim_result[sv(SIM_CAND) - 1] = removable ? 0 : 1;
        if (removable && ++sv(SIM_NREMOVABLE) == p.sim_max_removable) sv(SIM_CUT) = 1;   // unneededNodesLimit
      }
      __syncthreads();
    }
    if (!batch) break;
    }  // candidates
    if (p.prof && tid == 0) atomicAdd((unsigned long long*)&p.prof[7], (unsigned long long)(clock64() - prof_tmpl0));
    if constexpr (FM) {
      int over = 0, zero = 0;
      for (int c = tid; c < p.fm_nctrl; c += TPB) over += p.fm_ctrl_over[c] != 0;
      blk_sum_max<NW>(S, par, over, zero);
      if (batch && tid == 0 && !p.status[0]) p.sim_trace_off[p.sim_n] = sv(SIM_TRN);
      if (tid == 0) {
        if (batch) { last_index = sv(SIM_LI); fm_moved = true; }
        p.fm_out[0] = last_index; p.fm_out[1] = over; p.fm_out[2] = pods_total; p.fm_out[3] = fm_moved ? 1 : 0;
        if (S.overflow && p.status) atomicExch(p.status, 1);
      }
    } else if (tid == 0) {
      p.node_count[t] = nodes_with_pods;
      p.pod_count[t] = pods_total;
      if (p.last_index_out) p.last_index_out[t] = last_index;
      if (S.overflow && p.status) atomicExch(p.status, 1);
    }
  }
  if (tid == 0) hdr[1] = gver_ctr;
}

// The kernel is instantiated for 9 resource-dimension counts x {shared window, slab} + the filter pass: the file is compiled
// three times (-DBP_PART=0|1|2, A in {0,1,2} / {3,4,5} / {6,7,8}) so that build() can run the parts in parallel; the host
// side below lives in part 0.
#ifndef BP_PART
#define BP_PART 0
#endif
int bp_launch_part0(Engine* e, int A, int blocks_wanted, size_t smem, const BpParams& p, int* blocks_out, bool query_only, bool filter);
int bp_launch_part1(Engine* e, int A, int blocks_wanted, size_t smem, const BpParams& p, int* blocks_out, bool query_only, bool filter);
int bp_launch_part2(Engine* e, int A, int blocks_wanted, size_t smem, const BpParams& p, int* blocks_out, bool query_only, bool filter);

template <int A>
static int bp_launch_a(Engine* e, int blocks_wanted, size_t smem, const BpParams& p, int* blocks_out, bool query_only, bool filter) {
  if (filter) {
    binpack_kernel<A, 512, false, true><<<1, 512, 0, e->stream>>>(e->dobj, e->dyn, p);
    return 0;
  }
  auto kern = p.win ? binpack_kernel<A, 256, true, false> : binpack_kernel<A, 256, false, false>;
  CAE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  CAE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, smem));
  if (per_sm < 1) { set_error("binpack_kernel does not fit an SM"); return -1; }
  const int blocks = std::max(1, std::min(blocks_wanted, per_sm * e->sm_count));
  *blocks_out = blocks;
  if (query_only) return 0;
  kern<<<blocks, 256, smem, e->stream>>>(e->dobj, e->dyn, p);
  return 0;
}
#if BP_PART == 0
int bp_launch_part0(Engine* e, int A, int bw, size_t smem, const BpParams& p, int* bo, bool q, bool f) {
  return A == 0 ? bp_launch_a<0>(e, bw, smem, p, bo, q, f) : A == 1 ? bp_launch_a<1>(e, bw, smem, p, bo, q, f) : bp_launch_a<2>(e, bw, smem, p, bo, q, f);
}
#elif BP_PART == 1
int bp_launch_part1(Engine* e, int A, int bw, size_t smem, const BpParams& p, int* bo, bool q, bool f) {
  return A == 3 ? bp_launch_a<3>(e, bw, smem, p, bo, q, f) : A == 4 ? bp_launch_a<4>(e, bw, smem, p, bo, q, f) : bp_launch_a<5>(e, bw, smem, p, bo, q, f);
}
#else
int bp_launch_part2(Engine* e, int A, int bw, size_t smem, const BpParams& p, int* bo, bool q, bool f) {
  return A == 6 ? bp_launch_a<6>(e, bw, smem, p, bo, q, f) : A == 7 ? bp_launch_a<7>(e, bw, smem, p, bo, q, f) : bp_launch_a<8>(e, bw, smem, p, bo, q, f);
}
#endif

#if BP_PART == 0
// work order of the estimator blocks: templates by decreasing cost (pods in their schedulable groups), ties by index
__global__ void lpt_rank_kernel(const long long* __restrict__ cost, int t_begin, int nt, int32_t* __restrict__ perm) {
  __shared__ long long tile[256];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const long long mine = i < nt ? cost[t_begin + i] : 0;
  int rank = 0;
  for (int base = 0; base < nt; base += 256) {
    const int j = base + threadIdx.x;
    tile[threadIdx.x] = j < nt ? cost[t_begin + j] : LLONG_MIN;
    __syncthreads();
    const int lim = min(256, nt - base);
    for (int k = 0; k < lim; ++k) {
      const long long c = tile[k];
      rank += (c > mine) || (c == mine && base + k < i);
    }
    __syncthreads();
  }
  if (i < nt) perm[rank] = t_begin + i;
}

static int launch_binpack_any(Engine* e, int blocks_wanted, size_t smem, const BpParams& p, int* blocks_out, bool query_only, bool filter = false) {
  const int A = std::min(e->A, 8);
  if (A <= 2) return bp_launch_part0(e, A, blocks_wanted, smem, p, blocks_out, query_only, filter);
  if (A <= 5) return bp_launch_part1(e, A, blocks_wanted, smem, p, blocks_out, query_only, filter);
  return bp_launch_part2(e, A, blocks_wanted, smem, p, blocks_out, query_only, filter);
}

int launch_binpack(Engine* e) {
  const int nt = e->t_end - e->t_begin;
  if (nt <= 0) return 0;
  BpParams p{};
  p.E = e->E; p.T = e->T; p.N = e->N; p.U = e->U;
  p.has_dyn = e->has_dynamic ? 1 : 0;
  for (int a = 0; a < CAE_MAX_RES; ++a) p.act_dim[a] = e->act_dim[a];
  p.order = e->d_order; p.order_n = e->d_order_n; p.grec = e->d_grec; p.pre_code = e->d_pre_code; p.spec_sc = e->d_spec_sc; p.spec_dc = e->d_spec_dc;
  p.tmpl_free = e->d_tmpl_free; p.tmpl_slots = e->d_tmpl_slots; p.max_nodes = e->d_max_nodes;
  p.pc_of = e->d_pc_of; p.port_conf = e->d_port_conf; p.c_free = e->d_c_free; p.c_slots = e->d_c_slots;
  p.node_count = e->d_counts2; p.pod_count = e->d_counts2 + e->T; p.sched = e->d_sched;
  p.work_counter = e->d_work_counter; p.status = e->d_work_counter + 1;
  p.t_begin = e->t_begin; p.t_end = e->t_end;
  p.last_index_in = e->d_last_index_in; p.last_index_out = e->d_last_index_out;
  // node capacity of a simulation: the largest limiter cap, or (unlimited) one node per pod + 1
  // (every added node but possibly one holds >= 1 pod)
  const int cap = std::max(1, std::min(e->P + 1, e->pack_cap));
  p.cap = cap;
  const int A1 = std::max(e->A, 1);
  const int Neff = p.has_dyn ? e->N : 0;
  // shared window for the added nodes: per node A1 x int64 free + ports + slots + capacity + prefix + flag
  const size_t node_bytes = (size_t)A1 * 8 + 8 + 4 + 4 + 4 + 1;
  size_t smem = ((size_t)cap * node_bytes + 15) & ~(size_t)15;
  const size_t smem_limit = (size_t)e->smem_optin > 9216 ? (size_t)e->smem_optin - 9216 : 0;   // static part + reserve
  if (smem <= smem_limit) p.win = cap; else { p.win = 0; smem = 0; }
  const size_t Xg = (size_t)Neff + (p.win ? 0 : cap);
  int dmax = 1;
  for (int k = 0; k < e->dyn.K; ++k) dmax = std::max(dmax, e->dyn.Dc[k] + 1 + (e->dyn.is_host[k] ? cap : 0));
  p.dstride = p.has_dyn ? dmax : 1;
  p.log_cap = p.has_dyn ? (int)std::min<size_t>(4 * ((size_t)Neff + cap) + 1024, (size_t)1 << 24) : 1;
  size_t per_cta = 16 + Xg * ((size_t)A1 * 8 + 8 + 4 + 4 + 4 + 4) + (size_t)3 * DYN_MAX_Q * p.dstride * 4 + (size_t)p.log_cap * 12 + Xg;
  per_cta = (per_cta + 255) & ~(size_t)255;
  p.scratch_per_cta = per_cta;
  int blocks = 0;
  if (launch_binpack_any(e, nt, smem, p, &blocks, true)) return -1;
  const size_t budget = (size_t)24 << 30;  // keep the slabs within 24 GiB of the 180 GB HBM
  if (per_cta * blocks > budget) blocks = (int)std::max<size_t>(1, budget / per_cta);
  const size_t need = per_cta * blocks;
  const size_t sig = per_cta * 1000003u + Xg * 10007u + (size_t)p.dstride * 101u + (size_t)p.log_cap * 7u + (size_t)A1 + 0x9000000000ull;
  if (need > e->pack_scratch_bytes) {
    if (e->d_pack_scratch) cudaFree(e->d_pack_scratch);
    e->d_pack_scratch = nullptr;
    e->pack_scratch_bytes = 0;
    CAE_CUDA(cudaMalloc(&e->d_pack_scratch, need));
    e->pack_scratch_bytes = need;
    e->pack_layout_sig = 0;
  }
  if (sig != e->pack_layout_sig) {  // slot versions are only meaningful within one slab layout
    CAE_CUDA(cudaMemsetAsync(e->d_pack_scratch, 0, need, e->stream));
    e->pack_layout_sig = sig;
  }
  p.scratch = static_cast<unsigned char*>(e->d_pack_scratch);
  CAE_CUDA(cudaMemsetAsync(e->d_work_counter, 0, sizeof(int32_t) * 2, e->stream));
  // longest processing time first: the heaviest templates start first, the tail of the pass is made of light ones
  lpt_rank_kernel<<<(nt + 255) / 256, 256, 0, e->stream>>>(e->d_tmpl_cost, e->t_begin, nt, e->d_perm);
  e->stats.kernel_launches++;
  p.perm = e->d_perm;
  static const bool want_prof = getenv("CAE_PACK_PROF") != nullptr;
  long long* d_prof = nullptr;
  if (want_prof) {
    CAE_CUDA(cudaMalloc(&d_prof, sizeof(long long) * 16));
    CAE_CUDA(cudaMemsetAsync(d_prof, 0, sizeof(long long) * 16, e->stream));
    p.prof = d_prof;
  }
  int launched = 0;
  if (launch_binpack_any(e, blocks, smem, p, &launched, false)) return -1;
  e->stats.kernel_launches++;
  CAE_KERNEL_OK();
  if (want_prof) {
    long long h[16];
    CAE_CUDA(cudaMemcpyAsync(h, d_prof, sizeof(h), cudaMemcpyDeviceToHost, e->stream));
    CAE_CUDA(cudaStreamSynchronize(e->stream));
    cudaFree(d_prof);
    fprintf(stderr, "binpack prof: blocks=%d smem=%zu win=%d cycles{plain_rr=%lld plain_new=%lld dyn_setup=%lld fast=%lld genA=%lld genB=%lld template=%lld} "
            "counts{plain=%lld fast=%lld generic=%lld generic_pods=%lld genA_iters=%lld genB_iters=%lld cluster_caps=%lld cluster_phase=%lld}\n",
            launched, smem, p.win, h[0], h[1], h[2], h[4], h[5], h[6], h[7], h[8], h[9], h[10], h[11], h[12], h[13], h[14], h[15]);
  }
  return 0;
}

// ---- filter-out-schedulable pass -----------------------------------------------------------------------------------------
__global__ void run_rec_kernel(DevObjects o, DynTables d, int runs, const int32_t* __restrict__ run_off, const int32_t* __restrict__ pods,
                               int n_act, const int* __restrict__ act_dim, int has_dyn, const int32_t* __restrict__ spec_sc,
                               const int32_t* __restrict__ spec_dc, const int32_t* __restrict__ pc_of,
                               const unsigned long long* __restrict__ port_conf, GroupRec* __restrict__ out) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= runs) return;
  GroupRec g{};
  const int pb = run_off[r];
  g.n = run_off[r + 1] - pb;
  g.pad[0] = pb;
  const int spec = o.pend_spec[pods[pb]];
  g.spec = spec;
  g.sc = spec_sc[spec];
  g.dc = has_dyn ? spec_dc[spec] : 0;
  const int plist = o.ps_port_list[spec];
  const bool has_ports = o.port_off[plist + 1] > o.port_off[plist];
  g.pconf = has_ports ? port_conf[plist] : 0ull;
  g.pbit = has_ports ? (1ull << pc_of[plist]) : 0ull;
  bool feeds = false;   // runs are not groups: log every placement that some counter counts
  if (has_dyn) for (int q = 0; q < d.Q && !feeds; ++q) feeds = d.wmat[(size_t)q * d.S + spec] != 0;
  g.flags = (has_ports ? GREC_HAS_PORTS : 0u) | (feeds ? GREC_FEEDS : 0u) | (o.ps_hostname_spread[spec] ? GREC_HOST_SPREAD : 0u);
  for (int a = 0; a < n_act; ++a) {
    g.req[a] = o.ps_req[(size_t)spec * R + act_dim[a]];
    g.rinv[a] = g.req[a] > 0 ? __frcp_rn(__ll2float_rn(g.req[a])) : 0.f;
  }
  out[r] = g;
}

// HintingSimulator.TrySchedulePods on the cluster snapshot (one thread block).  `f` = device blob laid out by
// cae_filter_schedulable (api.cu); class marks and controller counters are zeroed there.
int launch_filter(Engine* e, const FilterLaunch& f) {
  BpParams p{};
  p.E = e->E; p.T = e->T; p.N = e->N; p.U = e->U;
  p.has_dyn = e->has_dynamic ? 1 : 0;
  for (int a = 0; a < CAE_MAX_RES; ++a) p.act_dim[a] = e->act_dim[a];
  p.pre_code = e->d_pre_code; p.spec_sc = e->d_spec_sc; p.spec_dc = e->d_spec_dc;
  p.pc_of = e->d_pc_of; p.port_conf = e->d_port_conf; p.c_free = e->d_c_free; p.c_slots = e->d_c_slots;
  p.work_counter = e->d_work_counter; p.status = e->d_work_counter + 1;
  p.t_begin = 0; p.t_end = 1; p.cap = 0; p.win = 0;
  p.fm_runs = f.runs; p.fm_last_index = f.last_index; p.fm_break = f.break_on_failure; p.fm_nctrl = f.nctrl;
  p.fm_pods = f.pods; p.fm_hint = f.hint; p.fm_class = f.cls; p.fm_class_ctrl = f.class_ctrl;
  p.fm_node_ok = f.node_ok; p.fm_assigned = f.assigned; p.fm_out = f.out;
  p.fm_ctrl_cnt = f.ctrl_cnt; p.fm_class_mark = f.class_mark; p.fm_ctrl_over = f.ctrl_over;
  const int A1 = std::max(e->A, 1);
  const size_t Xg = (size_t)e->N;
  int dmax = 1;
  for (int k = 0; k < e->dyn.K; ++k) dmax = std::max(dmax, e->dyn.Dc[k] + 2);
  p.dstride = p.has_dyn ? dmax : 1;
  // one entry per placement at most (batch: per placement of the kept simulations and the running one, <= the trace)
  p.log_cap = p.has_dyn ? f.n_pods + 1024 : 1;
  size_t per_cta = 16 + Xg * ((size_t)A1 * 8 + 8 + 4 + 4 + 4 + 4) + (size_t)3 * DYN_MAX_Q * p.dstride * 4 + (size_t)p.log_cap * 12 + Xg;
  per_cta = (per_cta + 255) & ~(size_t)255;
  p.scratch_per_cta = per_cta;
  const int n_rec = f.runs + (f.sim ? e->P : 0);   // batch: + one record per pending pod
  const size_t rec_bytes = ((size_t)std::max(n_rec, 1) * sizeof(GroupRec) + 255) & ~(size_t)255;
  const size_t need = per_cta + rec_bytes;
  const size_t sig = per_cta * 1000003u + Xg * 10007u + (size_t)p.dstride * 101u + (size_t)p.log_cap * 7u + (size_t)A1 + 0x7000000000ull;
  if (need > e->fm_scratch_bytes) {
    if (e->d_fm_scratch) cudaFree(e->d_fm_scratch);
    e->d_fm_scratch = nullptr;
    e->fm_scratch_bytes = 0;
    CAE_CUDA(cudaMalloc(&e->d_fm_scratch, need));
    e->fm_scratch_bytes = need;
    e->fm_layout_sig = 0;
  }
  if (sig != e->fm_layout_sig) {
    CAE_CUDA(cudaMemsetAsync(e->d_fm_scratch, 0, need, e->stream));
    e->fm_layout_sig = sig;
  }
  p.scratch = static_cast<unsigned char*>(e->d_fm_scratch);
  GroupRec* d_rec = reinterpret_cast<GroupRec*>(p.scratch + per_cta);
  p.grec = d_rec;
  CAE_CUDA(cudaMemsetAsync(e->d_work_counter, 0, sizeof(int32_t) * 2, e->stream));
  if (f.runs > 0) {
    run_rec_kernel<<<(f.runs + 127) / 128, 128, 0, e->stream>>>(e->dobj, e->dyn, f.runs, f.run_off, f.pods, e->A, e->d_act_dim, p.has_dyn,
                                                               e->d_spec_sc, e->d_spec_dc, e->d_pc_of, e->d_port_conf, d_rec);
    e->stats.kernel_launches++;
  }
  if (const SimLaunch* s = f.sim) {
    if (e->P > 0) {
      run_rec_kernel<<<(e->P + 127) / 128, 128, 0, e->stream>>>(e->dobj, e->dyn, e->P, s->iota, s->iota, e->A, e->d_act_dim, p.has_dyn,
                                                                e->d_spec_sc, e->d_spec_dc, e->d_pc_of, e->d_port_conf, d_rec + f.runs);
      e->stats.kernel_launches++;
    }
    p.sim_n = s->n; p.sim_persist = s->persist; p.sim_max_removable = s->max_removable; p.sim_trace_cap = s->trace_cap;
    p.sim_cand = s->cand; p.sim_pod_off = s->pod_off; p.sim_pods = s->pods; p.sim_run_off = s->cand_run_off;
    p.sim_rec_pod = d_rec + f.runs;
    p.sim_result = s->result; p.sim_trace_off = s->trace_off; p.sim_trace_pod = s->trace_pod; p.sim_trace_node = s->trace_node;
    p.sim_st = s->st; p.sim_present = s->present; p.sim_nok = s->nok; p.sim_seen = s->seen;
    p.sim_dest = f.node_ok;
    p.fm_node_ok = s->nok;
    p.sim_pos = s->pos; p.sim_at = s->at; p.sim_gone = s->gone;
    p.sim_mv_head = s->mv_head; p.sim_mv_tail = s->mv_tail; p.sim_mv_next = s->mv_next;
    p.sim_bk_free = s->bk_free; p.sim_bk_ports = s->bk_ports; p.sim_bk_slots = s->bk_slots;
  }
  { int unused = 0; if (launch_binpack_any(e, 1, 0, p, &unused, false, true)) return -1; }
  e->stats.kernel_launches++;
  CAE_KERNEL_OK();
  return 0;
}
#endif  // BP_PART == 0

}  // namespace cae
