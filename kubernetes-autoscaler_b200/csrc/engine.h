// engine.h — internal state of the scale-up simulation engine (host side).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <string>
#include <vector>

#include "../../include/caengine.h"
#include "dyn.cuh"
#include "tables.cuh"

namespace cae {

constexpr int FEAS_MAX_W = 4;
constexpr int FEAS_LUT_MAX_ROWS = 1024;     // threshold rows (68 KB of shared memory) above which the dense pass falls back to bit slices
constexpr int FEAS_TW = 16;                // template words per thread block of the dense pass; row pitch Twp is a multiple

void set_error(const std::string& msg);

// Everything the estimator needs to know about a pending pod group, gathered once per load so that a thread block
// fetches ONE contiguous record per group (cp.async, one group ahead) instead of chasing five dependent tables.
struct alignas(16) GroupRec {
  int32_t n, spec, sc, dc;            // pods, pod spec, static class, dynamic class (0 = plain)
  uint32_t flags;                     // GREC_*
  int32_t pad[3];
  unsigned long long pconf, pbit;     // host-port sets the pod collides with / the bit of its own set
  int64_t req[CAE_MAX_RES];           // request per ACTIVE resource dim
  float rinv[CAE_MAX_RES];            // 1 / req (0 when the dim is not requested)
};
static_assert(sizeof(GroupRec) == 144, "GroupRec is fetched as nine 16-byte chunks");
enum : uint32_t { GREC_HAS_PORTS = 1u, GREC_FEEDS = 2u, GREC_HOST_SPREAD = 4u };
constexpr int ORDER_NOT_ON_FRESH = 1 << 30;   // order entry flag: the group's static filters fail on the SANITIZED template

#define CAE_CUDA(expr)                                                                        \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      cae::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                     \
      return -1;                                                                              \
    }                                                                                         \
  } while (0)

#define CAE_KERNEL_OK()                                                                       \
  do {                                                                                        \
    cudaError_t _e = cudaGetLastError();                                                      \
    if (_e != cudaSuccess) {                                                                  \
      cae::set_error(std::string(__func__) + ": " + cudaGetErrorString(_e));                  \
      return -1;                                                                              \
    }                                                                                         \
  } while (0)

// Chunked bump allocator that persists across loads.  `mirrored` arenas pair every device chunk with a
// pinned host chunk at the same offsets so a whole load is ONE cudaMemcpyAsync per chunk.
struct Arena {
  struct Chunk { void* dev = nullptr; void* host = nullptr; size_t size = 0, used = 0, flushed = 0; };
  std::vector<Chunk> chunks;
  size_t cur = 0;
  size_t min_chunk = (size_t)32 << 20;
  bool mirrored = false;
  int alloc(void** dev, void** stage, size_t bytes);
  int flush(cudaStream_t st, int64_t* bytes);
  void reset();
  void release();
};

struct Engine {
  cae_config cfg{};
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr;
  Arena up;         // uploaded tables (pinned mirror), reset per load
  Arena scratch;    // device-only tables of the current load
  Engine() { up.mirrored = true; }
  DynTables dyn;    // PodTopologySpread / InterPodAffinity tables (dyn.cuh)
  const uint8_t* d_spec_used = nullptr;
  const int32_t* d_dc_ngroups = nullptr;
  int64_t* d_c_free = nullptr;            // [A][N] free capacity of the cluster nodes (fallback placements)
  int32_t* d_c_slots = nullptr;           // [N]
  int* d_act_dim = nullptr;               // [CAE_MAX_RES]
  std::vector<int32_t> h_spec_dc;
  bool h_dc_of_spec_valid = false;
  cae_stats stats{};
  bool loaded = false;

  // sizes of the current load
  int N = 0, T = 0, E = 0, P = 0, U = 0;  // U = N + 2T universe columns
  int A = 0;                              // active resource dims (some pending pod requests > 0)
  int act_dim[CAE_MAX_RES] = {0};
  int SC = 0, DC = 0;                     // static / dynamic classes
  int Tw = 0;                             // ceil(T/32)
  int Twp = 0;                            // Tw rounded up to whole FEAS_TW chunks: pitch of pre_ok / post_ok / rlut
  int p_begin = 0, p_end = 0;             // pod shard of this rank (feasibility)
  int t_begin = 0, t_end = 0;             // template shard of this rank (estimate)
  int Pl = 0, Plw = 0;                    // local pods, ceil(Pl/32)
  bool has_dynamic = false;               // any PTS / inter-pod affinity in the snapshot

  DevObjects dobj{};                      // device mirror of the object tables
  // derived device tables
  StaticClass* d_sclass = nullptr;        // [SC]
  uint8_t* d_pre_code = nullptr;          // [SC][U] static_code()
  uint32_t* d_pre_ok = nullptr;           // [SC][Twp] bit t: low nibble of pre_code[sc][N+t] == 0 and template has a pod slot
  int32_t* d_spec_sc = nullptr;           // [num_podspecs] static class of each spec
  int32_t* d_spec_dc = nullptr;           // [num_podspecs] dynamic class (0 = none)
  uint8_t* d_post_code = nullptr;         // [DC][T] PTS / IPA reason on the empty template (0 = ok)
  uint32_t* d_post_ok = nullptr;          // [DC][Twp]
  int W = 0;                              // 32-bit words of the packed rank encoding (feas.cu)
  uint32_t feas_guard[4] = {0, 0, 0, 0};  // guard-bit mask per word
  uint32_t* d_spec_w = nullptr;           // [num_podspecs][FEAS_MAX_W] packed request ranks
  uint32_t* d_pod_w = nullptr;            // [W][Pl] per pending pod
  uint16_t* d_pod_row = nullptr;          // [A][Pl] threshold-row id per active dim (LUT variant)
  uint32_t* d_tmpl_w = nullptr;           // [W][T] packed free-capacity ranks + guard bits
  int feas_B = 0;                         // bit slices of the free-capacity ranks (all fields)
  uint32_t feas_fstart = 0;               // bit b set: slice b is the most significant bit of a field
  uint8_t feas_sword[32] = {0}, feas_sshift[32] = {0};  // where bit b sits in the packed pod words
  uint32_t* d_tslice = nullptr;           // [ceil4(B)][Tw] bit-sliced template ranks
  // threshold bitmaps (feas.cu, LUT variant): row lut_base[a] + k, bit t = "a request of rank k in dim a fits template t"
  int lut_rows = 0;
  int lut_base[CAE_MAX_RES] = {0};
  uint8_t lut_word[CAE_MAX_RES] = {0}, lut_shift[CAE_MAX_RES] = {0};
  uint32_t lut_mask[CAE_MAX_RES] = {0};
  uint32_t* d_rlut = nullptr;             // [lut_rows][Twp]
  long long* d_tmpl_cost = nullptr;       // [T] pods in the schedulable groups of a template (order kernel)
  int32_t* d_perm = nullptr;              // [T] work order of the pack
  int k1_warps = 16;                      // warps per thread block of the LUT variant (CAE_K1_WARPS=8|16)
  bool force_bitslice = false;            // CAE_K1_BITSLICE=1: always take the bit-sliced comparator (tests)
  int32_t* d_pod_sc = nullptr;            // [P]
  int32_t* d_pod_dc = nullptr;            // [P]
  int64_t* d_tmpl_free = nullptr;         // [A][T] allocatable - DaemonSet requested
  int64_t* d_tmpl_free_all = nullptr;     // [R][T] same over all R dims (pack kernel)
  int32_t* d_tmpl_slots = nullptr;        // [T] allowed pods - DaemonSet pods
  int64_t* d_spec_req_t = nullptr;        // [num_podspecs][R] request (raw)
  // results kept on device
  uint32_t* d_fit_bits = nullptr;         // [T][Plw]
  uint8_t* d_reasons = nullptr;           // [T][Pl] (want_reasons)
  int32_t* d_fit_count = nullptr;         // [T]
  int32_t* d_fit_acc = nullptr;           // [T] self-cleaning accumulators of the dense pass
  int32_t* d_chunk_done = nullptr;        // [Twp / FEAS_TW] arrival counters per template chunk
  uint8_t* d_group_reason = nullptr;      // [T][E]
  bool group_reason_valid = false;
  int32_t* d_counts2 = nullptr;           // [2T] node_count | pod_count
  int32_t* d_sched = nullptr;             // [T][E]
  int32_t* d_order = nullptr;             // [T][E]
  int32_t* d_order_n = nullptr;           // [T]
  GroupRec* d_grec = nullptr;             // [E]
  double* d_score = nullptr;              // [T][E]
  int32_t* d_max_nodes = nullptr;         // [T]
  int32_t* d_last_index_buf = nullptr;    // [2T] lastIndex in | out (cae_estimate_all_ex)
  const int32_t* d_last_index_in = nullptr;   // set per call: NULL = every Estimate starts at 0
  int32_t* d_last_index_out = nullptr;
  int32_t* d_pc_of = nullptr;             // [num_port_lists] compact id of a pending pod's port list, -1 otherwise
  unsigned long long* d_port_conf = nullptr;  // [num_port_lists] conflict mask over compact ids
  int pack_cap = 1 << 30;                 // node capacity of a pack slab (from the limiter caps)
  // pack scratch
  void* d_pack_scratch = nullptr;
  size_t pack_scratch_bytes = 0;
  size_t pack_layout_sig = 0;
  // filter-out-schedulable pass (binpack.cu, FM): own slab + input blob
  void* d_fm_scratch = nullptr;
  size_t fm_scratch_bytes = 0, fm_layout_sig = 0;
  int32_t* d_fm_blob = nullptr;
  size_t fm_blob_words = 0;
  // fused histogram exchange over peer memory (feas.cu)
  static constexpr int PEER_MAX = 8, PEER_CAP = 1 << 16;
  int32_t* d_xbuf = nullptr;              // [2 parities][PEER_MAX][PEER_CAP] (count, step tag) slots + done counter, status
  int peer_world = 0;
  int32_t* peer_base[PEER_MAX] = {nullptr};
  int64_t peer_step = 0;
  int32_t* d_work_counter = nullptr;
  // host copies needed by host-side steps
  const int32_t *h_group_off = nullptr, *h_pend_spec = nullptr;   // host copy of the pending-pod rows: views into h_pending_stage
  std::vector<int32_t> h_group_spec;      // [E] spec of each group's pods (-1 = empty group)
  bool groups_homogeneous = true;         // every group holds pods of ONE spec (equivalence.BuildPodGroups guarantees it)
  std::vector<uint8_t> h_spec_pending;    // [num_podspecs] spec carried by a pending pod at the last full load
  int cap_P = 0, cap_E = 0, cap_Pl = 0;   // capacities of the resident per-pod / per-group buffers (cae_load_pending)
  int32_t* h_pending_stage = nullptr;     // pinned staging of pend_spec | group_off for the delta upload
  size_t pending_stage_words = 0;
  std::vector<int64_t> h_spec_req;        // [num_podspecs][R]
  std::vector<int64_t> h_cap_cpu, h_cap_mem;  // per template
  int num_podspecs = 0;
  int sm_count = 148;
  int smem_optin = 227 * 1024;             // opt-in shared memory per thread block
};

// kernels.cu
int launch_class_matrix(Engine* e);      // pre_code[SC][U]: needs only the object tables + the static classes
int launch_pre_ok_bits(Engine* e);       // pre_ok[SC][Twp]: needs pre_code and the templates' pod slots
int launch_post_bits(Engine* e);
int launch_dynamic_tables(Engine* e, const uint8_t* d_spec_used, const int32_t* d_dc_ngroups);
int launch_expand_pods(Engine* e);
int launch_port_conflicts(Engine* e, int num_port_lists);
int launch_feasibility(Engine* e, bool want_reasons);
int launch_group_feasibility(Engine* e);
int launch_order(Engine* e);
int launch_group_records(Engine* e);     // GroupRec[E] (after the class / counter tables of a load)
int launch_binpack(Engine* e);   // K3: block-per-template estimator (binpack.cu)
// cae_simulate_removals: the candidate loop of the filter pass (device pointers into the call's blob, see BpParams).
// Words of SimLaunch::st: the running candidate and what the candidate loop carries (kept in global memory: the filter
// instantiation of the kernel is at its register budget).  The caller zeroes them and sets SIM_LI to the raw lastIndex.
enum { SIM_RES, SIM_C, SIM_OWN0, SIM_OWN_N, SIM_MOVED, SIM_SEG, SIM_RUN0, SIM_RUNS_OWN, SIM_LOG0, SIM_NREM, SIM_TRN, SIM_LI,
       SIM_NREMOVABLE, SIM_CUT, SIM_NCUR, SIM_CAND, SIM_WORDS };
struct SimLaunch {
  int n, persist, max_removable, trace_cap;
  const int32_t *cand, *pod_off, *pods, *cand_run_off;
  const int32_t* iota;   // [P + 1] 0, 1, ..., P: run offsets and pods of the one-pod records
  int32_t *result, *trace_off, *trace_pod, *trace_node, *st;
  uint8_t *present, *nok, *seen;
  int32_t *pos, *at, *gone, *mv_head, *mv_tail, *mv_next, *bk_slots;
  int64_t* bk_free;
  unsigned long long* bk_ports;
};
struct FilterLaunch {
  int runs, n_pods, last_index, break_on_failure, nctrl;
  const int32_t *run_off, *pods, *hint, *cls, *class_ctrl;
  const uint8_t* node_ok;
  int32_t *assigned, *out, *ctrl_cnt;
  uint8_t *class_mark, *ctrl_over;
  const SimLaunch* sim;   // NULL = one pass (cae_filter_schedulable)
};
int launch_filter(Engine* e, const FilterLaunch& f);
int launch_price(Engine* e, const cae_price_inputs& in_dev, const int32_t* d_node_count, const int32_t* d_sched, const int32_t* d_order,
                 double* d_score);
int launch_expander(Engine* e, const int32_t* chain, int chain_len, const int32_t* d_node_count,
                    const int32_t* d_pod_count, const int32_t* d_sched, uint8_t* d_mask, double* d_waste);

}  // namespace cae
