// api.cu — C ABI of libcaengine.so (include/caengine.h) and the host-side flattener.
//
// cae_load turns the interned object tables into the engine's device layout:
//   * every table is uploaded verbatim (DevObjects) — selectors, tolerations, label sets are
//     evaluated ON THE GPU, the host never runs a predicate;
//   * pod specs are interned into "static classes" (tolerations, node affinity/selector, nodeName,
//     host ports) so the plugins whose verdict does not depend on the pod's size are evaluated once
//     per (class, node) by class_matrix_kernel and re-used by every pod of the class;
//   * per-pod request planes [A][P] (A = resource dims any pending pod asks for) and per-template
//     free-capacity planes [A][T] are laid out SoA for coalesced int64 loads in the dense pass.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <tuple>
#include <unordered_map>

#include "engine.h"

namespace cae {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }

// ---- arenas: chunked bump allocators that persist across loads (no cudaMalloc on the hot path) ----
int Arena::alloc(void** dev, void** stage, size_t bytes) {
  bytes = (std::max<size_t>(bytes, 16) + 255) & ~(size_t)255;
  for (;;) {
    if (cur < chunks.size() && chunks[cur].used + bytes <= chunks[cur].size) break;
    if (cur + 1 < chunks.size()) { ++cur; continue; }
    Chunk c;
    c.size = std::max(bytes, min_chunk);
    if (cudaMalloc(&c.dev, c.size) != cudaSuccess) { set_error("cudaMalloc failed"); return -1; }
    if (mirrored && cudaHostAlloc(&c.host, c.size, cudaHostAllocDefault) != cudaSuccess) { set_error("cudaHostAlloc failed"); return -1; }
    chunks.push_back(c);
    cur = chunks.size() - 1;
  }
  Chunk& c = chunks[cur];
  *dev = static_cast<char*>(c.dev) + c.used;
  if (stage) *stage = mirrored ? static_cast<char*>(c.host) + c.used : nullptr;
  c.used += bytes;
  return 0;
}
void Arena::reset() { for (auto& c : chunks) c.used = c.flushed = 0; cur = 0; }
void Arena::release() {
  for (auto& c : chunks) { cudaFree(c.dev); if (c.host) cudaFreeHost(c.host); }
  chunks.clear();
  cur = 0;
}
int Arena::flush(cudaStream_t st, int64_t* bytes) {
  for (auto& c : chunks)   // incremental: only what was staged since the last flush
    if (c.used > c.flushed) {
      if (cudaMemcpyAsync(static_cast<char*>(c.dev) + c.flushed, static_cast<char*>(c.host) + c.flushed, c.used - c.flushed,
                          cudaMemcpyHostToDevice, st) != cudaSuccess) { set_error("H2D failed"); return -1; }
      if (bytes) *bytes += (int64_t)(c.used - c.flushed);
      c.flushed = c.used;
    }
  return 0;
}

template <class T>
static int upload(Engine* e, const T* host, size_t n, const T** dev) {
  void *p = nullptr, *h = nullptr;
  if (e->up.alloc(&p, &h, n * sizeof(T))) return -1;
  if (n) memcpy(h, host, n * sizeof(T));
  *dev = static_cast<const T*>(p);
  return 0;
}
template <class T>
static int upload_mut(Engine* e, const std::vector<T>& v, T** dev) {
  const T* p = nullptr;
  if (upload(e, v.data(), v.size(), &p)) return -1;
  *dev = const_cast<T*>(p);
  return 0;
}
template <class T>
static int dev_alloc(Engine* e, T** dev, size_t n, bool zero = false) {
  void* p = nullptr;
  if (e->scratch.alloc(&p, nullptr, n * sizeof(T))) return -1;
  if (zero && n) {
    cudaError_t err = cudaMemsetAsync(p, 0, n * sizeof(T), e->stream);
    if (err != cudaSuccess) { set_error(std::string("memset: ") + cudaGetErrorString(err)); return -1; }
  }
  *dev = static_cast<T*>(p);
  return 0;
}

#define UP(field, count)                                                           \
  if (upload(e, o->field, (size_t)(count), &e->dobj.field)) return -1

static bool host_label(const cae_objects* o, int ls, int key, int* val) {
  for (int i = o->ls_off[ls]; i < o->ls_off[ls + 1]; ++i)
    if (o->ls_key[i] == key) { *val = o->ls_val[i]; return true; }
  return false;
}

// Interning for the pod-state dependent plugins (dyn.cuh): topology keys -> compact ids, label values
// -> domain indices, pod specs -> dynamic classes, and the list of counters each class needs.
// Structure only; every match / count is computed on the device (dyn_kernels.cu).
static int build_dynamic(Engine* e, const cae_objects* o, const std::vector<uint8_t>& spec_pending,
                         const std::vector<int32_t>& spec_sc, std::vector<int32_t>& spec_dc) {
  DynTables& d = e->dyn;
  d = DynTables();
  const int N = e->N, T = e->T, NT = N + T, S = o->num_podspecs;
  d.S = S;
  auto nonempty = [&](const int32_t* off, int l) { return off[l + 1] > off[l]; };
  std::vector<uint8_t> spec_used(spec_pending);
  for (int i = 0; i < o->node_pod_off[NT]; ++i) spec_used[o->node_pod_spec[i]] = 1;
  bool any = false;
  std::vector<int> keys;
  auto add_key = [&](int key) { if (std::find(keys.begin(), keys.end(), key) == keys.end()) keys.push_back(key); };
  std::vector<int> exist_keys;  // topology keys of anti-affinity terms held by any pod in the snapshot
  for (int s = 0; s < S; ++s) {
    if (!spec_used[s]) continue;
    int al = o->ps_anti_list[s];
    for (int t = o->aff_off[al]; t < o->aff_off[al + 1]; ++t) {
      any = true;
      add_key(o->aterm_key[t]);
      if (std::find(exist_keys.begin(), exist_keys.end(), o->aterm_key[t]) == exist_keys.end()) exist_keys.push_back(o->aterm_key[t]);
    }
    if (!spec_pending[s]) continue;
    int pl = o->ps_pts_list[s], fl = o->ps_aff_list[s];
    for (int c = o->pts_off[pl]; c < o->pts_off[pl + 1]; ++c) { any = true; add_key(o->pts_key[c]); }
    for (int t = o->aff_off[fl]; t < o->aff_off[fl + 1]; ++t) { any = true; add_key(o->aterm_key[t]); }
  }
  e->has_dynamic = any;
  if (!any) return 0;
  if ((int)keys.size() > DYN_MAX_KEYS) { set_error("more than 8 distinct topology keys"); return 1; }
  d.K = (int)keys.size();
  std::vector<int32_t> dom((size_t)d.K * NT, -1);
  for (int k = 0; k < d.K; ++k) {
    d.key_id[k] = keys[k];
    d.is_host[k] = keys[k] == o->hostname_key;
    std::map<int, int> ids;
    for (int row = 0; row < NT; ++row) {
      if (row == N) d.Dc[k] = (int)ids.size();
      int v;
      if (!host_label(o, o->node_labelset[row], keys[k], &v)) continue;
      auto it = ids.find(v);
      if (it == ids.end()) it = ids.emplace(v, (int)ids.size()).first;
      dom[(size_t)k * NT + row] = it->second;
    }
    if (T == 0) d.Dc[k] = (int)ids.size();
    d.D[k] = (int)ids.size();
  }
  auto kidx = [&](int key) { return (int)(std::find(keys.begin(), keys.end(), key) - keys.begin()); };
  // dynamic classes
  std::map<std::tuple<int, int, int, int, int, int>, int> dc_ids;
  std::vector<int32_t> dc_spec(1, 0), dc_sc(1, 0), dc_q_off(1, 0), dc_ngroups(1, 0);
  std::vector<uint8_t> q_kind;
  std::vector<int32_t> q_k, q_dc, q_p0, q_base_off(1, 0);
  dc_q_off.push_back(0);
  for (int s = 0; s < S; ++s) {
    if (!spec_pending[s]) continue;
    int pl = o->ps_pts_list[s], fl = o->ps_aff_list[s], al = o->ps_anti_list[s];
    if (!nonempty(o->pts_off, pl) && !nonempty(o->aff_off, fl) && !nonempty(o->aff_off, al) && exist_keys.empty()) continue;
    auto key = std::make_tuple(o->ps_namespace[s], o->ps_labelset[s], pl, fl, al, spec_sc[s]);
    auto it = dc_ids.find(key);
    if (it == dc_ids.end()) {
      int dc = (int)dc_spec.size();
      it = dc_ids.emplace(key, dc).first;
      dc_spec.push_back(s);
      dc_sc.push_back(spec_sc[s]);
      dc_ngroups.push_back(0);
      auto add_q = [&](int kind, int k, int p0) {
        q_kind.push_back((uint8_t)kind); q_k.push_back(k); q_dc.push_back(dc); q_p0.push_back(p0);
        q_base_off.push_back(q_base_off.back() + d.Dc[k]);
      };
      for (int c = o->pts_off[pl]; c < o->pts_off[pl + 1]; ++c) add_q(Q_PTS, kidx(o->pts_key[c]), c);
      for (int t = o->aff_off[fl]; t < o->aff_off[fl + 1]; ++t) add_q(Q_AFF, kidx(o->aterm_key[t]), t);
      for (int t = o->aff_off[al]; t < o->aff_off[al + 1]; ++t) add_q(Q_ANTI, kidx(o->aterm_key[t]), t);
      for (int key2 : exist_keys) add_q(Q_EXIST, kidx(key2), -1);
      if ((int)q_kind.size() - dc_q_off.back() > DYN_MAX_Q) { set_error("a pod needs more than 12 topology counters"); return 1; }
      dc_q_off.push_back((int)q_kind.size());
    }
    spec_dc[s] = it->second;
  }
  for (int g = 0; g < o->num_groups; ++g)
    if (o->group_off[g + 1] > o->group_off[g]) dc_ngroups[spec_dc[o->pend_spec[o->group_off[g]]]]++;
  d.DC = (int)dc_spec.size();
  d.Q = (int)q_kind.size();
  e->DC = d.DC;
  const int32_t* p32 = nullptr; const uint8_t* p8 = nullptr;
#define UPV(vec, field) { if (upload(e, (vec).data(), (vec).size(), &field)) return -1; }
  UPV(dom, d.dom); UPV(dc_spec, d.dc_spec); UPV(dc_sc, d.dc_sc); UPV(dc_q_off, d.dc_q_off); UPV(q_kind, d.q_kind);
  UPV(q_k, d.q_k); UPV(q_dc, d.q_dc); UPV(q_p0, d.q_p0); UPV(q_base_off, d.q_base_off);
  UPV(spec_used, p8); e->d_spec_used = p8;
  UPV(dc_ngroups, p32); e->d_dc_ngroups = p32;
#undef UPV
  const size_t Q = std::max(d.Q, 1), pool = std::max(q_base_off.back(), 1);
  if (dev_alloc(e, &d.wmat, Q * S) || dev_alloc(e, &d.q_self, Q) || dev_alloc(e, &d.q_wown, Q) || dev_alloc(e, &d.q_active, Q) ||
      dev_alloc(e, &d.dc_aff_self, (size_t)d.DC) || dev_alloc(e, &d.dc_active, (size_t)d.DC) || dev_alloc(e, &d.elig, Q * e->U) ||
      dev_alloc(e, &d.base_cnt, pool, true) || dev_alloc(e, &d.base_pres, pool, true) || dev_alloc(e, &d.base_tot, Q, true) ||
      dev_alloc(e, &d.ds_w, Q * std::max(T, 1)) || dev_alloc(e, &d.st_min1, Q) || dev_alloc(e, &d.st_arg1, Q) ||
      dev_alloc(e, &d.st_min2, Q) || dev_alloc(e, &d.st_ndom, Q) || dev_alloc(e, &d.st_nmin, Q) || dev_alloc(e, &d.q_nfeed, Q, true) ||
      dev_alloc(e, &d.group_feeds, (size_t)std::max(e->E, 1), true) || dev_alloc(e, &d.qrec, Q))
    return -1;
  e->h_dc_of_spec_valid = true;
  return 0;
}

struct LoadTimer {   // CAE_LOAD_TIMING=1: host wall clock of the phases of cae_load on stderr
  bool on;
  std::chrono::steady_clock::time_point t0;
  std::string out;
  LoadTimer() : on(getenv("CAE_LOAD_TIMING") != nullptr), t0(std::chrono::steady_clock::now()) {}
  void mark(const char* what) {
    if (!on) return;
    auto t1 = std::chrono::steady_clock::now();
    char buf[96];
    snprintf(buf, sizeof(buf), " %s=%.1fus", what, std::chrono::duration<double, std::micro>(t1 - t0).count());
    out += buf;
    t0 = t1;
  }
  ~LoadTimer() { if (on) fprintf(stderr, "cae_load:%s\n", out.c_str()); }
};

// Host copy of the pending-pod rows in pinned memory (source of the H2D copy of cae_load_pending, read by the filter pass),
// the spec of every group and whether the groups are homogeneous.  `check_pending`: refuse specs that were not pending at
// the last full load (returns 2).
static int stage_pending(Engine* e, int P, const int32_t* pend_spec, int E, const int32_t* group_off, bool check_pending) {
  const size_t words = (size_t)P + E + 1;
  if (words > e->pending_stage_words) {
    if (e->h_pending_stage) cudaFreeHost(e->h_pending_stage);
    e->h_pending_stage = nullptr;
    e->pending_stage_words = 0;
    const size_t cap_words = std::max(words, (size_t)e->cap_P + e->cap_E + 1);
    CAE_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&e->h_pending_stage), cap_words * 4, cudaHostAllocDefault));
    e->pending_stage_words = cap_words;
  }
  const int S = e->num_podspecs;
  // one pass per group: the exemplar's spec must have been pending at the last full load, the other pods must equal it
  std::vector<int32_t> gspec(E, -1);
  bool homog = true;
  for (int g = 0; g < E; ++g) {
    const int b = group_off[g], en = group_off[g + 1];
    if (en <= b) continue;
    const int s0 = pend_spec[b];
    if (check_pending && (s0 < 0 || s0 >= S || !e->h_spec_pending[s0])) { set_error("cae_load_pending: a pod spec that was not pending at the last cae_load"); return 2; }
    gspec[g] = s0;
    int diff = 0;
    for (int p = b + 1; p < en; ++p) diff |= pend_spec[p] ^ s0;
    homog &= diff == 0;
  }
  if (!homog && check_pending)   // heterogeneous groups (only the filter pass accepts them): every pod's spec is checked
    for (int p = 0; p < P; ++p) {
      const int s = pend_spec[p];
      if (s < 0 || s >= S || !e->h_spec_pending[s]) { set_error("cae_load_pending: a pod spec that was not pending at the last cae_load"); return 2; }
    }
  if (P) memcpy(e->h_pending_stage, pend_spec, sizeof(int32_t) * P);
  memcpy(e->h_pending_stage + P, group_off, sizeof(int32_t) * (E + 1));
  e->h_pend_spec = e->h_pending_stage;
  e->h_group_off = e->h_pending_stage + P;
  e->h_group_spec.swap(gspec);
  e->groups_homogeneous = homog;
  return 0;
}

static int do_load(Engine* e, const cae_objects* o) {
  LoadTimer lt;
  if (o->abi_version != CAE_ABI_VERSION) { set_error("cae_objects.abi_version mismatch"); return -2; }
  if (o->num_res < 3 || o->num_res > CAE_MAX_RES) { set_error("num_res out of range"); return 1; }
  e->up.reset();
  e->scratch.reset();
  e->loaded = false;
  e->group_reason_valid = false;
  e->stats.h2d_bytes = 0;
  const int N = o->num_cluster_nodes, T = o->num_templates, NT = N + T;
  e->N = N; e->T = T; e->U = N + 2 * T; e->E = o->num_groups; e->P = o->num_pending;
  e->Tw = (T + 31) / 32;
  e->Twp = (e->Tw + FEAS_TW - 1) / FEAS_TW * FEAS_TW;
  e->num_podspecs = o->num_podspecs;
  const int W = std::max(1, e->cfg.world_size), rk = e->cfg.rank;
  e->p_begin = (int)((int64_t)e->P * rk / W);
  e->p_end = (int)((int64_t)e->P * (rk + 1) / W);
  e->p_begin = (e->p_begin / 32) * 32;  // word-aligned shards so bit rows concatenate
  if (rk + 1 < W) e->p_end = (e->p_end / 32) * 32;
  if (e->cfg.flags & CAE_CFG_PODS_PRESHARDED) { e->p_begin = 0; e->p_end = e->P; }   // the caller uploaded its own pod shard only
  e->Pl = e->p_end - e->p_begin;
  e->Plw = (e->Pl + 31) / 32;
  e->t_begin = (int)((int64_t)T * rk / W);
  e->t_end = (int)((int64_t)T * (rk + 1) / W);

  cudaEventRecord(e->ev0, e->stream);
  DevObjects& d = e->dobj;
  d.num_res = o->num_res; d.num_values = o->num_values; d.hostname_key = o->hostname_key;
  d.unschedulable_taint_key = o->unschedulable_taint_key; d.N = N; d.T = T;
  UP(value_is_int, o->num_values); UP(value_int, o->num_values);
  UP(ns_labelset, o->num_namespaces); UP(ns_exists, o->num_namespaces);
  UP(ls_off, o->num_labelsets + 1); UP(ls_key, o->ls_off[o->num_labelsets]); UP(ls_val, o->ls_off[o->num_labelsets]);
  UP(req_key, o->num_reqs); UP(req_op, o->num_reqs); UP(req_val_off, o->num_reqs + 1);
  UP(req_vals, o->num_reqs ? o->req_val_off[o->num_reqs] : 0);
  UP(sel_kind, o->num_selectors); UP(sel_req_off, o->num_selectors + 1);
  UP(naff_nodesel, o->num_naff); UP(naff_has_required, o->num_naff); UP(naff_term_off, o->num_naff + 1);
  UP(term_expr_sel, o->num_naff_terms); UP(term_field_off, o->num_naff_terms + 1);
  { int nf = o->term_field_off[o->num_naff_terms]; UP(field_op, nf); UP(field_node_name, nf); }
  { int n = o->tol_off[o->num_tol_lists]; UP(tol_off, o->num_tol_lists + 1); UP(tol_key, n); UP(tol_op, n); UP(tol_val, n); UP(tol_effect, n); }
  { int n = o->taint_off[o->num_taint_lists]; UP(taint_off, o->num_taint_lists + 1); UP(taint_key, n); UP(taint_val, n); UP(taint_effect, n); }
  { int n = o->port_off[o->num_port_lists]; UP(port_off, o->num_port_lists + 1); UP(port_ip, n); UP(port_proto, n); UP(port_num, n); }
  { int n = o->pts_off[o->num_pts_lists]; UP(pts_off, o->num_pts_lists + 1); UP(pts_max_skew, n); UP(pts_key, n); UP(pts_selector, n);
    UP(pts_min_domains, n); UP(pts_node_affinity_policy, n); UP(pts_node_taints_policy, n); }
  { int n = o->num_aterms; UP(aff_off, o->num_aff_lists + 1); UP(aterm_selector, n); UP(aterm_key, n); UP(aterm_ns_off, n + 1);
    UP(aterm_ns, o->aterm_ns_off[n]); UP(aterm_ns_selector, n); }
  { int n = o->num_podspecs; UP(ps_namespace, n); UP(ps_labelset, n); UP(ps_req, (size_t)n * R); UP(ps_tol_list, n); UP(ps_naff, n);
    UP(ps_node_name, n); UP(ps_port_list, n); UP(ps_pts_list, n); UP(ps_aff_list, n); UP(ps_anti_list, n); UP(ps_terminating, n);
    UP(ps_hostname_spread, n); }
  UP(node_name, NT); UP(node_labelset, NT); UP(node_taint_list, NT); UP(node_unschedulable, NT);
  UP(node_alloc, (size_t)NT * R); UP(node_allowed_pods, NT); UP(node_cap_cpu, NT); UP(node_cap_mem, NT);
  UP(node_has_alloc_cpu, NT); UP(node_has_alloc_mem, NT);
  UP(node_pod_off, NT + 1); UP(node_pod_spec, o->node_pod_off[NT]);
  UP(group_off, o->num_groups + 1); UP(pend_spec, o->num_pending);

  // ---- host-side interning of pod specs into classes (no predicate is evaluated here) ----
  const int S = o->num_podspecs;
  std::vector<uint8_t> spec_pending(S, 0);
  for (int p = 0, prev = -1; p < o->num_pending; ++p)   // pods of a group are adjacent and share a spec: touch the flag on changes only
    if (o->pend_spec[p] != prev) { prev = o->pend_spec[p]; spec_pending[prev] = 1; }
  struct Key4 { int a, b, c, d; bool operator==(const Key4& k) const { return a == k.a && b == k.b && c == k.c && d == k.d; } };
  struct Key4Hash {
    size_t operator()(const Key4& k) const {
      uint64_t h = (uint64_t)(uint32_t)k.a * 0x9E3779B97F4A7C15ull;
      h = (h ^ (uint32_t)k.b) * 0xBF58476D1CE4E5B9ull;
      h = (h ^ (uint32_t)k.c) * 0x94D049BB133111EBull;
      h = (h ^ (uint32_t)k.d) * 0x9E3779B97F4A7C15ull;
      return (size_t)(h ^ (h >> 29));
    }
  };
  std::unordered_map<Key4, int, Key4Hash> sc_ids;
  sc_ids.reserve((size_t)S * 2);
  std::vector<StaticClass> sclass;
  sclass.reserve(S);
  std::vector<int32_t> spec_sc(S, 0), spec_dc(S, 0);
  for (int s = 0; s < S; ++s) {
    if (!spec_pending[s]) continue;
    const Key4 key{o->ps_tol_list[s], o->ps_naff[s], o->ps_node_name[s], o->ps_port_list[s]};
    auto ins = sc_ids.emplace(key, (int)sclass.size());   // ids in order of first appearance
    if (ins.second) sclass.push_back({key.a, key.b, key.c, key.d});
    spec_sc[s] = ins.first->second;
  }
  // host-port lists of pending pods get compact ids (one bit each in a node's used-port mask)
  std::vector<int32_t> pc_of(o->num_port_lists, -1);
  int npc = 0;
  for (int s = 0; s < S; ++s) {
    int pl = o->ps_port_list[s];
    if (!spec_pending[s] || o->port_off[pl + 1] == o->port_off[pl] || pc_of[pl] >= 0) continue;
    if (npc == 64) { set_error("more than 64 distinct host-port sets among pending pods"); return 1; }
    pc_of[pl] = npc++;
  }
  if (sclass.empty()) sclass.push_back({0, -1, -1, 0});
  e->SC = (int)sclass.size();
  e->DC = 1;  // class 0: no topology-spread / inter-pod-affinity involvement
  e->h_dc_of_spec_valid = false;
  // The object tables and the static classes are complete: ship them and start the class matrix now, so that the
  // device works while the host goes on interning (dynamic classes, rank encoding).
  if (upload_mut(e, sclass, &e->d_sclass) || upload_mut(e, pc_of, &e->d_pc_of) || dev_alloc(e, &e->d_pre_code, (size_t)e->SC * e->U) ||
      dev_alloc(e, &e->d_port_conf, (size_t)std::max(o->num_port_lists, 1)))
    return -1;
  if (e->up.flush(e->stream, &e->stats.h2d_bytes)) return -1;
  if (launch_port_conflicts(e, o->num_port_lists)) return -1;
  if (launch_class_matrix(e)) return -1;
  lt.mark("stage+classes");
  { int rc = build_dynamic(e, o, spec_pending, spec_sc, spec_dc); if (rc) return rc; }
  lt.mark("build_dynamic");

  // active resource dims + free capacity of templates and cluster nodes
  e->A = 0;
  for (int r = 0; r < R; ++r) {
    bool used = false;
    for (int s = 0; s < S && !used; ++s) used = spec_pending[s] && o->ps_req[(size_t)s * R + r] > 0;
    if (used) e->act_dim[e->A++] = r;
  }
  const int A1 = std::max(e->A, 1);
  // order-preserving rank encoding of the request / free-capacity operands (feas.cu)
  std::vector<std::vector<int64_t>> rvals(e->A);
  for (int a = 0; a < e->A; ++a) {
    for (int s = 0; s < S; ++s) if (spec_pending[s] && o->ps_req[(size_t)s * R + e->act_dim[a]] > 0) rvals[a].push_back(o->ps_req[(size_t)s * R + e->act_dim[a]]);
    std::sort(rvals[a].begin(), rvals[a].end());
    rvals[a].erase(std::unique(rvals[a].begin(), rvals[a].end()), rvals[a].end());
  }
  int f_word[CAE_MAX_RES], f_shift[CAE_MAX_RES], f_bits[CAE_MAX_RES];
  e->W = 0;
  for (int w = 0; w < FEAS_MAX_W; ++w) e->feas_guard[w] = 0;
  { int w = 0, shift = 0;
    for (int a = 0; a < e->A; ++a) {
      int bits = 1;
      while ((1ll << bits) <= (long long)rvals[a].size()) ++bits;   // ranks 0..D need `bits` bits
      bits += 1;                                                     // + guard bit
      if (shift + bits > 32) { ++w; shift = 0; }
      if (w >= FEAS_MAX_W || bits > 32) { set_error("resource request cardinality too large for the rank encoding"); return 1; }
      f_word[a] = w; f_shift[a] = shift; f_bits[a] = bits;
      e->feas_guard[w] |= 1u << (shift + bits - 1);
      shift += bits;
      e->W = w + 1;
    } }
  std::vector<uint32_t> spec_w((size_t)S * FEAS_MAX_W, 0), tmpl_w((size_t)std::max(e->W, 1) * std::max(T, 1), 0);
  for (int s = 0; s < S; ++s) {
    if (!spec_pending[s]) continue;
    for (int a = 0; a < e->A; ++a) {
      int64_t v = o->ps_req[(size_t)s * R + e->act_dim[a]];
      uint32_t rank = v > 0 ? (uint32_t)(std::lower_bound(rvals[a].begin(), rvals[a].end(), v) - rvals[a].begin()) + 1 : 0;
      spec_w[(size_t)s * FEAS_MAX_W + f_word[a]] |= rank << f_shift[a];
    }
  }
  std::vector<int64_t> free_all((size_t)R * T), free_act((size_t)A1 * T), cfree((size_t)A1 * std::max(N, 1));
  std::vector<int32_t> slots(T), cslots(std::max(N, 1));
  for (int row = 0; row < NT; ++row) {
    int64_t reqd[R] = {0};
    int npods = o->node_pod_off[row + 1] - o->node_pod_off[row];
    for (int i = o->node_pod_off[row]; i < o->node_pod_off[row + 1]; ++i)
      for (int r = 0; r < R; ++r) reqd[r] += o->ps_req[(size_t)o->node_pod_spec[i] * R + r];
    if (row >= N) {
      int t = row - N;
      for (int r = 0; r < R; ++r) free_all[(size_t)r * T + t] = o->node_alloc[(size_t)row * R + r] - reqd[r];
      for (int a = 0; a < e->A; ++a) free_act[(size_t)a * T + t] = free_all[(size_t)e->act_dim[a] * T + t];
      slots[t] = o->node_allowed_pods[row] - npods;
      for (int a = 0; a < e->A; ++a) {
        int64_t f = free_act[(size_t)a * T + t];
        uint32_t rank = (uint32_t)(std::upper_bound(rvals[a].begin(), rvals[a].end(), f) - rvals[a].begin());
        tmpl_w[(size_t)f_word[a] * T + t] |= (rank | (1u << (f_bits[a] - 1))) << f_shift[a];
      }
    } else {   // cluster nodes: run state of the hostname-spread fallback (K3) and of the filter-out-schedulable pass
      for (int a = 0; a < e->A; ++a) cfree[(size_t)a * N + row] = o->node_alloc[(size_t)row * R + e->act_dim[a]] - reqd[e->act_dim[a]];
      cslots[row] = o->node_allowed_pods[row] - npods;
    }
  }
  // bit-sliced free-capacity ranks for the dense pass (feas.cu): slice b, word tw holds bit b of the rank
  // of templates tw*32 .. tw*32+31; slices run MSB-first inside a field, fields concatenated
  e->feas_B = 0;
  e->feas_fstart = 0;
  for (int a = 0; a < e->A; ++a) {
    const int nb = f_bits[a] - 1;
    for (int i = nb - 1; i >= 0; --i) {
      if (e->feas_B >= 32) { set_error("resource request cardinality too large for the bit-sliced encoding"); return 1; }
      e->feas_sword[e->feas_B] = (uint8_t)f_word[a];
      e->feas_sshift[e->feas_B] = (uint8_t)(f_shift[a] + i);
      if (i == nb - 1) e->feas_fstart |= 1u << e->feas_B;
      ++e->feas_B;
    }
  }
  // threshold bitmaps for the LUT variant of the dense pass: one row per (dim, request rank)
  e->lut_rows = 0;
  for (int a = 0; a < e->A; ++a) {
    e->lut_base[a] = e->lut_rows;
    e->lut_rows += (int)rvals[a].size() + 1;
    e->lut_word[a] = (uint8_t)f_word[a];
    e->lut_shift[a] = (uint8_t)f_shift[a];
    e->lut_mask[a] = (1u << (f_bits[a] - 1)) - 1u;
  }
  e->d_tslice = nullptr;
  if (e->force_bitslice || e->lut_rows > FEAS_LUT_MAX_ROWS) {   // only the fallback variant of the dense pass reads the slices
    const int Bpad = std::max(4, (e->feas_B + 3) / 4 * 4);
    std::vector<uint32_t> tslice((size_t)Bpad * std::max(e->Tw, 1), 0);
    for (int b = 0; b < e->feas_B; ++b)
      for (int t = 0; t < T; ++t)
        tslice[(size_t)b * e->Tw + t / 32] |= ((tmpl_w[(size_t)e->feas_sword[b] * T + t] >> e->feas_sshift[b]) & 1u) << (t % 32);
    if (upload_mut(e, tslice, &e->d_tslice)) return -1;
  }
  {
    std::vector<uint32_t> rlut((size_t)std::max(e->lut_rows, 1) * std::max(e->Twp, 1), 0);
    for (int a = 0; a < e->A; ++a)
      for (int t = 0; t < T; ++t) {
        const uint32_t rank_free = (tmpl_w[(size_t)f_word[a] * T + t] >> f_shift[a]) & e->lut_mask[a];
        for (uint32_t k = 0; k <= rank_free; ++k) rlut[(size_t)(e->lut_base[a] + k) * e->Twp + t / 32] |= 1u << (t % 32);
      }
    if (upload_mut(e, rlut, &e->d_rlut)) return -1;
  }
  if (upload_mut(e, spec_sc, &e->d_spec_sc) || upload_mut(e, slots, &e->d_tmpl_slots) ||
      upload_mut(e, free_all, &e->d_tmpl_free_all) || upload_mut(e, free_act, &e->d_tmpl_free) || upload_mut(e, cfree, &e->d_c_free) ||
      upload_mut(e, cslots, &e->d_c_slots) || upload_mut(e, spec_w, &e->d_spec_w) || upload_mut(e, tmpl_w, &e->d_tmpl_w) || upload_mut(e, spec_dc, &e->d_spec_dc))
    return -1;

  lt.mark("ranks+tables");
  if (dev_alloc(e, &e->d_pre_ok, (size_t)e->SC * std::max(e->Twp, 1)) ||
      dev_alloc(e, &e->d_post_code, (size_t)e->DC * std::max(T, 1), true) || dev_alloc(e, &e->d_post_ok, (size_t)e->DC * std::max(e->Twp, 1)) ||
      dev_alloc(e, &e->d_pod_w, (size_t)std::max(e->W, 1) * std::max(e->Pl, 1)) || dev_alloc(e, &e->d_pod_row, (size_t)std::max(e->A, 1) * std::max(e->Pl, 1)) || dev_alloc(e, &e->d_pod_sc, (size_t)std::max(e->Pl, 1)) ||
      dev_alloc(e, &e->d_pod_dc, (size_t)std::max(e->Pl, 1)) || dev_alloc(e, &e->d_fit_bits, (size_t)std::max(T, 1) * std::max(e->Plw, 1)) ||
      dev_alloc(e, &e->d_fit_count, (size_t)std::max(T, 1), true) || dev_alloc(e, &e->d_fit_acc, (size_t)std::max(T, 1), true) ||
      dev_alloc(e, &e->d_chunk_done, (size_t)std::max(e->Twp / FEAS_TW, 1), true) || dev_alloc(e, &e->d_group_reason, (size_t)std::max(T, 1) * std::max(e->E, 1)) ||
      dev_alloc(e, &e->d_counts2, (size_t)2 * std::max(T, 1), true) || dev_alloc(e, &e->d_sched, (size_t)std::max(T, 1) * std::max(e->E, 1), true) ||
      dev_alloc(e, &e->d_order, (size_t)std::max(T, 1) * std::max(e->E, 1)) || dev_alloc(e, &e->d_grec, (size_t)std::max(e->E, 1)) || dev_alloc(e, &e->d_order_n, (size_t)std::max(T, 1), true) ||
      dev_alloc(e, &e->d_max_nodes, (size_t)std::max(T, 1), true) || dev_alloc(e, &e->d_last_index_buf, (size_t)2 * std::max(T, 1), true) || dev_alloc(e, &e->d_tmpl_cost, (size_t)std::max(T, 1), true) ||
      dev_alloc(e, &e->d_perm, (size_t)std::max(T, 1)) || dev_alloc(e, &e->d_work_counter, 4, true) ||
      dev_alloc(e, &e->d_act_dim, CAE_MAX_RES))
    return -1;
  e->d_score = nullptr;
  e->d_reasons = nullptr;
  if (e->cfg.want_reasons && dev_alloc(e, &e->d_reasons, (size_t)std::max(T, 1) * std::max(e->Pl, 1))) return -1;

  // host copies for host-side steps (homogeneity check) and for the per-tick delta (cae_load_pending)
  e->h_spec_pending = spec_pending;
  e->cap_P = e->P; e->cap_E = e->E; e->cap_Pl = e->Pl;
  { int rc = stage_pending(e, e->P, o->pend_spec, e->E, o->group_off, false); if (rc) return rc; }

  lt.mark("dev_alloc+memsets");
  if (e->up.flush(e->stream, &e->stats.h2d_bytes)) return -1;   // ONE pinned H2D copy per arena chunk
  CAE_CUDA(cudaMemcpyAsync(e->d_act_dim, e->act_dim, sizeof(int) * CAE_MAX_RES, cudaMemcpyHostToDevice, e->stream));
  if (launch_pre_ok_bits(e)) return -1;
  if (e->has_dynamic) {
    if (launch_dynamic_tables(e, e->d_spec_used, e->d_dc_ngroups)) return -1;
    // classes none of whose counters can ever be non-zero are plain: fold them back into class 0
    std::vector<uint8_t> act(e->dyn.DC);
    CAE_CUDA(cudaMemcpyAsync(act.data(), e->dyn.dc_active, act.size(), cudaMemcpyDeviceToHost, e->stream));
    CAE_CUDA(cudaStreamSynchronize(e->stream));
    bool changed = false;
    for (int s = 0; s < S; ++s) if (spec_dc[s] && !act[spec_dc[s]]) { spec_dc[s] = 0; changed = true; }
    if (changed) CAE_CUDA(cudaMemcpyAsync(e->d_spec_dc, spec_dc.data(), sizeof(int32_t) * S, cudaMemcpyHostToDevice, e->stream));
    e->h_spec_dc = spec_dc;
    CAE_CUDA(cudaStreamSynchronize(e->stream));
  }
  if (launch_post_bits(e)) return -1;
  if (launch_expand_pods(e)) return -1;
  if (launch_group_records(e)) return -1;
  cudaEventRecord(e->ev1, e->stream);
  lt.mark("launches");
  CAE_CUDA(cudaStreamSynchronize(e->stream));
  lt.mark("sync");
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev0, e->ev1);
  e->stats.h2d_ms = ms;
  e->loaded = true;
  return 0;
}

}  // namespace cae

using cae::Engine;

// The expander filter chain is a sequential scan over <= T options in option order
// (expander/factory/chain.go:36-45) — it keeps the reference's order-dependent quirks
// (waste.go:58-65: equality tested before the nil/less-than branch).
static int32_t run_expander_chain(const int32_t* chain, int32_t chain_len, int T, const int32_t* node_count,
                                  const int32_t* pod_count, const double* waste, uint8_t* best_mask,
                                  const double* price = nullptr, const uint8_t* price_error = nullptr,
                                  const int32_t* priority = nullptr) {
  std::vector<int> opts;
  for (int t = 0; t < T; ++t) if (node_count[t] > 0) opts.push_back(t);
  for (int c = 0; c < chain_len; ++c) {
    std::vector<int> best;
    if (chain[c] == CAE_EXP_LEAST_WASTE) {
      double least = 0.0;
      for (int t : opts) {
        double w = waste[t];
        if (w == least) best.push_back(t);
        if (best.empty() || w < least) { least = w; best.assign(1, t); }
      }
    } else if (chain[c] == CAE_EXP_MOST_PODS) {
      int mx = 0;
      for (int t : opts) {
        if (pod_count[t] == mx) { best.push_back(t); continue; }
        if (pod_count[t] > mx) { mx = pod_count[t]; best.assign(1, t); }
      }
    } else if (chain[c] == CAE_EXP_LEAST_NODES) {
      int least = INT32_MAX;
      for (int t : opts) {
        if (node_count[t] == 0) continue;
        if (node_count[t] == least) { best.push_back(t); continue; }
        if (node_count[t] < least) { least = node_count[t]; best.assign(1, t); }
      }
    } else if (chain[c] == CAE_EXP_PRICE) {   // expander/price/price.go:166-173
      if (!price) { cae::set_error("price filter without price scores"); return -2; }
      double best_score = 0.0;
      for (int t : opts) {
        if (price_error && price_error[t]) continue;
        if (best.empty() || best_score == price[t]) { best.push_back(t); best_score = price[t]; }
        else if (best_score > price[t]) { best.assign(1, t); best_score = price[t]; }
      }
    } else if (chain[c] == CAE_EXP_PRIORITY) {   // expander/priority/priority.go:119-165
      if (!priority) { cae::set_error("priority filter without priorities"); return -2; }
      int max_prio = -1;
      for (int t : opts) {
        if (priority[t] < 0 || priority[t] < max_prio) continue;   // not in the configuration / lower priority
        if (priority[t] > max_prio) { max_prio = priority[t]; best.clear(); }
        best.push_back(t);
      }
      if (best.empty()) best = opts;   // "no priorities info found for any of the expansion options. No options filtered."
    } else { cae::set_error("unknown expander filter"); return 1; }
    opts.swap(best);
    if (opts.size() == 1) break;
  }
  if (best_mask) {
    std::fill(best_mask, best_mask + T, 0);
    for (int t : opts) best_mask[t] = 1;
  }
  return 0;
}

extern "C" {

const char* cae_last_error(void) { return cae::g_err.c_str(); }
const char* cae_version(void) { return "caengine/0.1 sm_100a"; }

int32_t cae_create(const cae_config* cfg, cae_engine** out) {
  if (!cfg || !out) return -2;
  if (cfg->abi_version != CAE_ABI_VERSION) { cae::set_error("cae_config.abi_version mismatch"); return -2; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cae::set_error("no CUDA device: the engine has no CPU fallback");
    return -1;
  }
  if (cfg->flags & CAE_CFG_GATES_REPORTED) {
    const int32_t g = cfg->feature_gates;
    if (!(g & CAE_GATE_NODE_INCLUSION_POLICY_IN_PTS) || (g & CAE_GATE_TAINT_TOLERATION_COMPARISON_OPERATORS) || (g & CAE_GATE_DRA_EXTENDED_RESOURCE)) {
      cae::set_error("feature gates differ from the ones the engine implements (NodeInclusionPolicyInPodTopologySpread on, "
                     "TaintTolerationComparisonOperators off, DRAExtendedResource off)");
      return 1;
    }
  }
  Engine* e = new Engine();
  e->cfg = *cfg;
  if (e->cfg.world_size < 1) e->cfg.world_size = 1;
  if (cudaSetDevice(cfg->device) != cudaSuccess) { cae::set_error("cudaSetDevice failed"); delete e; return -1; }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, cfg->device) == cudaSuccess) { e->sm_count = prop.multiProcessorCount; e->smem_optin = (int)prop.sharedMemPerBlockOptin; }
  if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) { cae::set_error("stream create failed"); delete e; return -1; }
  cudaEventCreate(&e->ev0);
  cudaEventCreate(&e->ev1);
  { const char* v = getenv("CAE_K1_BITSLICE"); e->force_bitslice = v && v[0] == '1'; }
  { const char* v = getenv("CAE_K1_WARPS"); if (v && atoi(v) == 8) e->k1_warps = 8; }
  *out = reinterpret_cast<cae_engine*>(e);
  return 0;
}

void cae_destroy(cae_engine* h) {
  if (!h) return;
  Engine* e = reinterpret_cast<Engine*>(h);
  cudaSetDevice(e->cfg.device);
  e->up.release();
  e->scratch.release();
  if (e->d_pack_scratch) cudaFree(e->d_pack_scratch);
  if (e->d_fm_scratch) cudaFree(e->d_fm_scratch);
  if (e->d_fm_blob) cudaFree(e->d_fm_blob);
  if (e->h_pending_stage) cudaFreeHost(e->h_pending_stage);
  if (e->ev2) { cudaEventDestroy(e->ev2); cudaEventDestroy(e->ev3); }
  if (e->ev0) cudaEventDestroy(e->ev0);
  if (e->ev1) cudaEventDestroy(e->ev1);
  if (e->stream) cudaStreamDestroy(e->stream);
  delete e;
}

int32_t cae_load(cae_engine* h, const cae_objects* objs) {
  if (!h || !objs) return -2;
  Engine* e = reinterpret_cast<Engine*>(h);
  cudaSetDevice(e->cfg.device);
  return cae::do_load(e, objs);
}

int32_t cae_load_pending(cae_engine* h, int32_t num_pending, const int32_t* pend_spec, int32_t num_groups, const int32_t* group_off) {
  Engine* e = reinterpret_cast<Engine*>(h);
  if (!e || !e->loaded) { cae::set_error("cae_load_pending before cae_load"); return -2; }
  if (num_pending < 0 || num_groups < 0 || (num_pending && !pend_spec) || !group_off) { cae::set_error("cae_load_pending: bad arguments"); return -2; }
  cudaSetDevice(e->cfg.device);
  const int P = num_pending, E = num_groups;
  // shard of this rank under the same rule as cae_load
  const int W = std::max(1, e->cfg.world_size), rk = e->cfg.rank;
  int pb = (int)((int64_t)P * rk / W), pe = (int)((int64_t)P * (rk + 1) / W);
  pb = (pb / 32) * 32;
  if (rk + 1 < W) pe = (pe / 32) * 32;
  if (e->cfg.flags & CAE_CFG_PODS_PRESHARDED) { pb = 0; pe = P; }
  const int Pl = pe - pb;
  if (P > e->cap_P || E > e->cap_E || Pl > e->cap_Pl) { cae::set_error("cae_load_pending: more pods / groups than the resident buffers hold"); return 2; }
  if (group_off[0] != 0 || group_off[E] != P) { cae::set_error("cae_load_pending: group_off does not cover the pending pods"); return -2; }
  if (e->has_dynamic) {   // the topology counters know which GROUPS feed them: the group -> spec sequence must be the resident one
    bool same = E == e->E;
    for (int g = 0; g < E && same; ++g) {
      const int s_new = group_off[g + 1] > group_off[g] ? pend_spec[group_off[g]] : -1;
      same = s_new == e->h_group_spec[g];
    }
    if (!same) { cae::set_error("cae_load_pending: the group -> spec sequence changed under topology counters"); return 2; }
  }
  // wait for the previous delta's copies before the pinned rows are overwritten (normally long finished)
  CAE_CUDA(cudaStreamSynchronize(e->stream));
  { int rc = cae::stage_pending(e, P, pend_spec, E, group_off, true); if (rc) return rc; }
  const size_t words = (size_t)P + E + 1;
  if (P) CAE_CUDA(cudaMemcpyAsync(const_cast<int32_t*>(e->dobj.pend_spec), e->h_pend_spec, sizeof(int32_t) * P, cudaMemcpyHostToDevice, e->stream));
  CAE_CUDA(cudaMemcpyAsync(const_cast<int32_t*>(e->dobj.group_off), e->h_group_off, sizeof(int32_t) * (E + 1), cudaMemcpyHostToDevice, e->stream));
  e->stats.h2d_bytes = (int64_t)words * 4;
  e->P = P; e->E = E; e->p_begin = pb; e->p_end = pe; e->Pl = Pl; e->Plw = (Pl + 31) / 32;
  e->group_reason_valid = false;
  if (cae::launch_expand_pods(e)) return -1;
  if (cae::launch_group_records(e)) return -1;
  // no synchronize: the stream orders the copies and the two kernels before whatever the caller launches next
  return 0;
}

int32_t cae_feasibility(cae_engine* h, uint32_t* fit_bits, uint8_t* reasons, int32_t* fit_count) {
  Engine* e = reinterpret_cast<Engine*>(h);
  if (!e || !e->loaded) { cae::set_error("cae_feasibility before cae_load"); return -2; }
  cudaSetDevice(e->cfg.device);
  bool want_r = e->cfg.want_reasons && e->d_reasons;
  cudaEventRecord(e->ev0, e->stream);
  if (cae::launch_feasibility(e, want_r)) return -1;
  cudaEventRecord(e->ev1, e->stream);
  e->stats.d2h_bytes = 0;
  if (!e->ev2) { cudaEventCreate(&e->ev2); cudaEventCreate(&e->ev3); }
  cudaEvent_t c0 = e->ev2, c1 = e->ev3;
  cudaEventRecord(c0, e->stream);
  if (fit_bits && e->T && e->Plw) {
    CAE_CUDA(cudaMemcpyAsync(fit_bits, e->d_fit_bits, sizeof(uint32_t) * (size_t)e->T * e->Plw, cudaMemcpyDeviceToHost, e->stream));
    e->stats.d2h_bytes += sizeof(uint32_t) * (size_t)e->T * e->Plw;
  }
  if (reasons && want_r && e->T && e->Pl) {
    CAE_CUDA(cudaMemcpyAsync(reasons, e->d_reasons, (size_t)e->T * e->Pl, cudaMemcpyDeviceToHost, e->stream));
    e->stats.d2h_bytes += (size_t)e->T * e->Pl;
  }
  if (fit_count && e->T) {
    CAE_CUDA(cudaMemcpyAsync(fit_count, e->d_fit_count, sizeof(int32_t) * e->T, cudaMemcpyDeviceToHost, e->stream));
    e->stats.d2h_bytes += sizeof(int32_t) * e->T;
  }
  cudaEventRecord(c1, e->stream);
  int32_t peer_status = 0;
  if (e->peer_world > 1)
    CAE_CUDA(cudaMemcpyAsync(&peer_status, e->d_xbuf + (size_t)4 * Engine::PEER_MAX * Engine::PEER_CAP + 9, sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
  CAE_CUDA(cudaStreamSynchronize(e->stream));
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev0, e->ev1);
  e->stats.feasibility_ms = ms;
  cudaEventElapsedTime(&ms, c0, c1);
  e->stats.d2h_ms = ms;
  e->stats.evals = (int64_t)e->Pl * e->T;
  if (peer_status) { cae::set_error("peer exchange timed out: a rank did not contribute its histogram"); return -1; }
  return 0;
}

int32_t cae_feasibility_groups(cae_engine* h, uint8_t* reasons) {
  Engine* e = reinterpret_cast<Engine*>(h);
  if (!e || !e->loaded) { cae::set_error("cae_feasibility_groups before cae_load"); return -2; }
  cudaSetDevice(e->cfg.device);
  if (cae::launch_group_feasibility(e)) return -1;
  if (reasons && e->T && e->E)
    CAE_CUDA(cudaMemcpyAsync(reasons, e->d_group_reason, (size_t)e->T * e->E, cudaMemcpyDeviceToHost, e->stream));
  CAE_CUDA(cudaStreamSynchronize(e->stream));
  return 0;
}

int32_t cae_estimate_all(cae_engine* h, const int32_t* max_nodes, int32_t* node_count, int32_t* pod_count,
                         int32_t* sched_count, int32_t* order) {
  return cae_estimate_all_ex(h, max_nodes, nullptr, node_count, pod_count, sched_count, order, nullptr);
}

int32_t cae_estimate_all_ex(cae_engine* h, const int32_t* max_nodes, const int32_t* last_index_in, int32_t* node_count,
                            int32_t* pod_count, int32_t* sched_count, int32_t* order, int32_t* last_index_out) {
  Engine* e = reinterpret_cast<Engine*>(h);
  if (!e || !e->loaded) { cae::set_error("cae_estimate_all before cae_load"); return -2; }
  cudaSetDevice(e->cfg.device);
  // groups must be homogeneous (equivalence.BuildPodGroups guarantees it: core/scaleup/equivalence/groups.go:40-104); checked at load
  if (!e->groups_homogeneous) { cae::set_error("pod group with non-equivalent pods"); return 1; }
  const int T = e->T, E = e->E;
  if (T == 0) return 0;
  e->pack_cap = 1;
  for (int t = e->t_begin; t < e->t_end; ++t) {
    int m = max_nodes ? max_nodes[t] : 0;
    e->pack_cap = std::max(e->pack_cap, m > 0 ? m : (m == 0 ? e->P + 1 : 1));
  }
  e->d_last_index_in = nullptr;
  e->d_last_index_out = last_index_out ? e->d_last_index_buf + T : nullptr;
  if (last_index_in) {
    for (int t = 0; t < T; ++t) if (last_index_in[t] < 0) { cae::set_error("cae_estimate_all_ex: negative lastIndex"); return -2; }
    CAE_CUDA(cudaMemcpyAsync(e->d_last_index_buf, last_index_in, sizeof(int32_t) * T, cudaMemcpyHostToDevice, e->stream));
    e->d_last_index_in = e->d_last_index_buf;
  }
  if (last_index_out) CAE_CUDA(cudaMemsetAsync(e->d_last_index_buf + T, 0, sizeof(int32_t) * T, e->stream));
  if (max_nodes) CAE_CUDA(cudaMemcpyAsync(e->d_max_nodes, max_nodes, sizeof(int32_t) * T, cudaMemcpyHostToDevice, e->stream));
  else CAE_CUDA(cudaMemsetAsync(e->d_max_nodes, 0, sizeof(int32_t) * T, e->stream));
  CAE_CUDA(cudaMemsetAsync(e->d_counts2, 0, sizeof(int32_t) * 2 * T, e->stream));
  CAE_CUDA(cudaMemsetAsync(e->d_sched, 0, sizeof(int32_t) * (size_t)T * std::max(E, 1), e->stream));
  CAE_CUDA(cudaMemsetAsync(e->d_order, 0xff, sizeof(int32_t) * (size_t)T * std::max(E, 1), e->stream));
  cudaEventRecord(e->ev0, e->stream);
  if (!e->group_reason_valid && cae::launch_group_feasibility(e)) return -1;
  int rc = cae::launch_order(e);
  if (rc) return rc;
  rc = cae::launch_binpack(e);
  if (rc) return rc;
  cudaEventRecord(e->ev1, e->stream);
  int32_t pack_status = 0;
  CAE_CUDA(cudaMemcpyAsync(&pack_status, e->d_work_counter + 1, sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
  std::vector<int32_t> order_n_host(T);
  CAE_CUDA(cudaMemcpyAsync(order_n_host.data(), e->d_order_n, sizeof(int32_t) * T, cudaMemcpyDeviceToHost, e->stream));
  if (node_count) CAE_CUDA(cudaMemcpyAsync(node_count, e->d_counts2, sizeof(int32_t) * T, cudaMemcpyDeviceToHost, e->stream));
  if (pod_count) CAE_CUDA(cudaMemcpyAsync(pod_count, e->d_counts2 + T, sizeof(int32_t) * T, cudaMemcpyDeviceToHost, e->stream));
  if (sched_count && E) CAE_CUDA(cudaMemcpyAsync(sched_count, e->d_sched, sizeof(int32_t) * (size_t)T * E, cudaMemcpyDeviceToHost, e->stream));
  if (order && E) CAE_CUDA(cudaMemcpyAsync(order, e->d_order, sizeof(int32_t) * (size_t)T * E, cudaMemcpyDeviceToHost, e->stream));
  if (last_index_out) CAE_CUDA(cudaMemcpyAsync(last_index_out, e->d_last_index_buf + T, sizeof(int32_t) * T, cudaMemcpyDeviceToHost, e->stream));
  CAE_CUDA(cudaStreamSynchronize(e->stream));
  {
    int64_t steps = 0;
    for (int t = e->t_begin; t < e->t_end; ++t) steps += order_n_host[t];
    e->stats.estimate_group_steps = steps;
  }
  if (order && E)   // the device rows carry a flag bit per entry (ORDER_NOT_ON_FRESH); padding stays -1
    for (size_t i = 0, nn = (size_t)T * E; i < nn; ++i) if (order[i] >= 0) order[i] &= ~cae::ORDER_NOT_ON_FRESH;
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev0, e->ev1);
  e->stats.estimate_ms = ms;
  if (pack_status) { cae::set_error("placement log overflow (cross-group topology counters)"); return 1; }
  return 0;
}

int32_t cae_expander_best(cae_engine* h, const int32_t* chain, int32_t chain_len, const int32_t* node_count,
                          const int32_t* pod_count, const int32_t* sched_count, uint8_t* best_mask, double* waste_score) {
  Engine* e = reinterpret_cast<Engine*>(h);
  if (!e || !e->loaded) { cae::set_error("cae_expander_best before cae_load"); return -2; }
  cudaSetDevice(e->cfg.device);
  const int T = e->T, E = e->E;
  if (T == 0) return 0;
  // scores on the device: from the caller's (all-reduced) option table, or — sched_count == NULL —
  // straight from the device-resident result of the last cae_estimate_all (single-shard fast path)
  int32_t *d_nc = nullptr, *d_sched = nullptr;
  double* d_waste = nullptr;
  std::vector<double> waste(T);
  if (sched_count == nullptr) {
    void* pw = nullptr;
    if (e->scratch.alloc(&pw, nullptr, sizeof(double) * T)) return -1;
    d_waste = static_cast<double*>(pw);
    cudaEventRecord(e->ev0, e->stream);
    if (cae::launch_expander(e, chain, chain_len, e->d_counts2, nullptr, e->d_sched, nullptr, d_waste)) return -1;
    cudaEventRecord(e->ev1, e->stream);
    CAE_CUDA(cudaMemcpyAsync(waste.data(), d_waste, sizeof(double) * T, cudaMemcpyDeviceToHost, e->stream));
    CAE_CUDA(cudaStreamSynchronize(e->stream));
  } else {
    CAE_CUDA(cudaMalloc(&d_nc, sizeof(int32_t) * T));
    CAE_CUDA(cudaMalloc(&d_sched, sizeof(int32_t) * (size_t)T * std::max(E, 1)));
    CAE_CUDA(cudaMalloc(&d_waste, sizeof(double) * T));
    CAE_CUDA(cudaMemcpyAsync(d_nc, node_count, sizeof(int32_t) * T, cudaMemcpyHostToDevice, e->stream));
    if (E) CAE_CUDA(cudaMemcpyAsync(d_sched, sched_count, sizeof(int32_t) * (size_t)T * E, cudaMemcpyHostToDevice, e->stream));
    cudaEventRecord(e->ev0, e->stream);
    if (cae::launch_expander(e, chain, chain_len, d_nc, nullptr, d_sched, nullptr, d_waste)) return -1;
    cudaEventRecord(e->ev1, e->stream);
    CAE_CUDA(cudaMemcpyAsync(waste.data(), d_waste, sizeof(double) * T, cudaMemcpyDeviceToHost, e->stream));
    CAE_CUDA(cudaStreamSynchronize(e->stream));
    cudaFree(d_nc); cudaFree(d_sched); cudaFree(d_waste);
  }
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev0, e->ev1);
  e->stats.expander_ms = ms;
  if (waste_score) std::copy(waste.begin(), waste.end(), waste_score);
  return run_expander_chain(chain, chain_len, T, node_count, pod_count, waste.data(), best_mask);
}

int32_t cae_waste_scores(cae_engine* h, double* waste_score) {
  Engine* e = reinterpret_cast<Engine*>(h);
  if (!e || !e->loaded || !waste_score) { cae::set_error("cae_waste_scores before cae_load"); return -2; }
  cudaSetDevice(e->cfg.device);
  const int T = e->T;
  if (T == 0) return 0;
  void* pw = nullptr;
  if (e->scratch.alloc(&pw, nullptr, sizeof(double) * T)) return -1;
  const int32_t chain0 = CAE_EXP_LEAST_WASTE;
  if (cae::launch_expander(e, &chain0, 1, e->d_counts2, nullptr, e->d_sched, nullptr, static_cast<double*>(pw))) return -1;
  CAE_CUDA(cudaMemcpyAsync(waste_score, pw, sizeof(double) * T, cudaMemcpyDeviceToHost, e->stream));
  CAE_CUDA(cudaStreamSynchronize(e->stream));
  for (int t = 0; t < T; ++t)
    if (t < e->t_begin || t >= e->t_end) waste_score[t] = 0.0;   // rows of other ranks: x + 0.0 == x, a sum all-reduce assembles the vector
  return 0;
}

int32_t cae_expander_chain(const int32_t* chain, int32_t chain_len, int32_t num_templates, const int32_t* node_count,
                           const int32_t* pod_count, const double* waste_score, uint8_t* best_mask) {
  if (!chain || !node_count || !pod_count || !waste_score || num_templates < 0) return -2;
  return run_expander_chain(chain, chain_len, num_templates, node_count, pod_count, waste_score, best_mask);
}

int32_t cae_price_scores(cae_engine* h, const cae_price_inputs* in, const int32_t* node_count, const int32_t* sched_count,
                         const int32_t* order, double* score) {
  Engine* e = reinterpret_cast<Engine*>(h);
  if (!e || !e->loaded || !in || !score || !in->node_price || !in->pod_price) { cae::set_error("cae_price_scores: bad arguments"); return -2; }
  if ((node_count == nullptr) != (sched_count == nullptr) || (node_count == nullptr) != (order == nullptr)) {
    cae::set_error("cae_price_scores: node_count, sched_count and order must be given together");
    return -2;
  }
  cudaSetDevice(e->cfg.device);
  const int T = e->T, E = std::max(e->E, 1), S = e->num_podspecs;
  if (T == 0) return 0;
  // one staging blob: node_price | pod_price | unfitness | score, then the byte vectors
  const size_t nd = (size_t)T + S + (in->unfitness ? T : 0) + T;
  double* d_f = nullptr;
  uint8_t* d_b = nullptr;
  CAE_CUDA(cudaMalloc(&d_f, nd * sizeof(double)));
  CAE_CUDA(cudaMalloc(&d_b, (size_t)3 * T));
  cae_price_inputs dev = *in;
  size_t off = 0;
  CAE_CUDA(cudaMemcpyAsync(d_f + off, in->node_price, sizeof(double) * T, cudaMemcpyHostToDevice, e->stream)); dev.node_price = d_f + off; off += T;
  CAE_CUDA(cudaMemcpyAsync(d_f + off, in->pod_price, sizeof(double) * S, cudaMemcpyHostToDevice, e->stream)); dev.pod_price = d_f + off; off += S;
  if (in->unfitness) { CAE_CUDA(cudaMemcpyAsync(d_f + off, in->unfitness, sizeof(double) * T, cudaMemcpyHostToDevice, e->stream)); dev.unfitness = d_f + off; off += T; }
  double* d_score = d_f + off;
  dev.has_gpu = dev.exists = dev.price_error = nullptr;
  if (in->has_gpu) { CAE_CUDA(cudaMemcpyAsync(d_b, in->has_gpu, T, cudaMemcpyHostToDevice, e->stream)); dev.has_gpu = d_b; }
  if (in->exists) { CAE_CUDA(cudaMemcpyAsync(d_b + T, in->exists, T, cudaMemcpyHostToDevice, e->stream)); dev.exists = d_b + T; }
  int32_t *d_nc = e->d_counts2, *d_sched = e->d_sched, *d_order = e->d_order, *d_tmp = nullptr;
  if (node_count) {
    CAE_CUDA(cudaMalloc(&d_tmp, sizeof(int32_t) * ((size_t)T + (size_t)2 * T * E)));
    d_nc = d_tmp; d_sched = d_tmp + T; d_order = d_sched + (size_t)T * E;
    CAE_CUDA(cudaMemcpyAsync(d_nc, node_count, sizeof(int32_t) * T, cudaMemcpyHostToDevice, e->stream));
    CAE_CUDA(cudaMemcpyAsync(d_sched, sched_count, sizeof(int32_t) * (size_t)T * E, cudaMemcpyHostToDevice, e->stream));
    CAE_CUDA(cudaMemcpyAsync(d_order, order, sizeof(int32_t) * (size_t)T * E, cudaMemcpyHostToDevice, e->stream));
  }
  // with caller-supplied rows every template is scored; the device-resident result only holds this rank's shard
  const int tb = e->t_begin, te = e->t_end;
  if (node_count) { e->t_begin = 0; e->t_end = T; }
  const int rc = cae::launch_price(e, dev, d_nc, d_sched, d_order, d_score);
  e->t_begin = tb; e->t_end = te;
  if (rc) return rc;
  CAE_CUDA(cudaMemcpyAsync(score, d_score, sizeof(double) * T, cudaMemcpyDeviceToHost, e->stream));
  CAE_CUDA(cudaStreamSynchronize(e->stream));
  cudaFree(d_f); cudaFree(d_b);
  if (d_tmp) cudaFree(d_tmp);
  return 0;
}

int32_t cae_expander_chain_ex(const int32_t* chain, int32_t chain_len, int32_t num_templates, const int32_t* node_count,
                              const int32_t* pod_count, const double* waste_score, const double* price_score,
                              const uint8_t* price_error, const int32_t* priority, uint8_t* best_mask) {
  if (!chain || !node_count || !pod_count || num_templates < 0) return -2;
  for (int c = 0; c < chain_len; ++c)
    if (chain[c] == CAE_EXP_LEAST_WASTE && !waste_score) { cae::set_error("least-waste filter without waste scores"); return -2; }
  return run_expander_chain(chain, chain_len, num_templates, node_count, pod_count, waste_score, best_mask, price_score, price_error, priority);
}

int32_t cae_get_stats(cae_engine* h, cae_stats* out) {
  if (!h || !out) return -2;
  *out = reinterpret_cast<Engine*>(h)->stats;
  return 0;
}

void* cae_device_buffer(cae_engine* h, int32_t which, size_t* bytes) {
  Engine* e = reinterpret_cast<Engine*>(h);
  if (!e || !e->loaded) return nullptr;
  if (which == 0) { if (bytes) *bytes = sizeof(int32_t) * e->T; return e->d_fit_count; }
  if (which == 1) { if (bytes) *bytes = sizeof(int32_t) * 2 * e->T; return e->d_counts2; }
  return nullptr;
}

int32_t cae_filter_schedulable(cae_engine* h, const int32_t* pod_order, int32_t n_pods, const int32_t* hint_node,
                               const int32_t* sim_class, const int32_t* class_ctrl, int32_t n_classes, const uint8_t* node_ok,
                               int32_t last_index_in, int32_t break_on_failure, int32_t* assigned_node,
                               int32_t* last_index_out, int32_t* overflowing_controllers) {
  Engine* e = reinterpret_cast<Engine*>(h);
  if (!e || !e->loaded) { cae::set_error("cae_filter_schedulable before cae_load"); return -2; }
  if (n_pods < 0 || (n_pods > 0 && !pod_order) || !assigned_node || (sim_class && n_classes > 0 && !class_ctrl)) {
    cae::set_error("cae_filter_schedulable: bad arguments");
    return -2;
  }
  cudaSetDevice(e->cfg.device);
  const int P = e->P, N = e->N;
  // plugin_runner.go:81 scans from (lastIndex + i) % len: a lastIndex left by a longer node list wraps, and stays as it is
  // until a scan places a pod (:123)
  const int32_t last_index_raw = last_index_in;
  last_index_in = N > 0 ? (int32_t)((((int64_t)last_index_in % N) + N) % N) : 0;
  // runs: consecutive pods of the order with the same spec and similarity class and no hint
  std::vector<int32_t> run_off;
  for (int k = 0; k < n_pods; ++k) {
    const int pod = pod_order[k];
    if (pod < 0 || pod >= P) { cae::set_error("cae_filter_schedulable: pod index out of range"); return -2; }
    bool start = k == 0;
    if (!start) {
      const int prev = pod_order[k - 1];
      start = e->h_pend_spec[pod] != e->h_pend_spec[prev] || (hint_node && (hint_node[pod] >= 0 || hint_node[prev] >= 0)) ||
              (sim_class && sim_class[pod] != sim_class[prev]);
    }
    if (start) run_off.push_back(k);
  }
  run_off.push_back(n_pods);
  const int runs = (int)run_off.size() - 1;
  int nctrl = 0;
  if (!sim_class) n_classes = 0;
  for (int c = 0; c < n_classes; ++c) {
    if (class_ctrl[c] < 0) { cae::set_error("cae_filter_schedulable: negative controller id"); return -2; }
    nctrl = std::max(nctrl, class_ctrl[c] + 1);
  }
  if (sim_class)
    for (int i = 0; i < P; ++i)
      if (sim_class[i] >= n_classes) { cae::set_error("cae_filter_schedulable: similarity class out of range"); return -2; }
  // one blob: run_off | pods | hint | class | class_ctrl | assigned | out[4] | ctrl_cnt | node_ok, class_mark, ctrl_over (bytes)
  auto words = [](size_t bytes) { return (bytes + 3) / 4; };
  size_t off = 0;
  const size_t o_run = off; off += runs + 1;
  const size_t o_pods = off; off += std::max(n_pods, 1);
  const size_t o_hint = off; off += hint_node ? P : 0;
  const size_t o_cls = off; off += sim_class ? P : 0;
  const size_t o_cc = off; off += std::max(n_classes, 1);
  const size_t o_in_end = off;
  const size_t o_nodeok = off; off += node_ok ? words(N) : 0;
  const size_t o_in_end2 = off;
  const size_t o_asg = off; off += std::max(P, 1);
  const size_t o_out = off; off += 4;
  const size_t o_cnt = off; off += std::max(nctrl, 1);
  const size_t o_mark = off; off += words(std::max(n_classes, 1));
  const size_t o_over = off; off += words(std::max(nctrl, 1));
  (void)o_in_end;
  if (off > e->fm_blob_words) {
    if (e->d_fm_blob) cudaFree(e->d_fm_blob);
    e->d_fm_blob = nullptr;
    e->fm_blob_words = 0;
    CAE_CUDA(cudaMalloc(&e->d_fm_blob, off * 4));
    e->fm_blob_words = off;
  }
  std::vector<int32_t> hostblob(o_in_end2, 0);
  std::copy(run_off.begin(), run_off.end(), hostblob.begin() + o_run);
  if (n_pods) std::copy(pod_order, pod_order + n_pods, hostblob.begin() + o_pods);
  if (hint_node) std::copy(hint_node, hint_node + P, hostblob.begin() + o_hint);
  if (sim_class) std::copy(sim_class, sim_class + P, hostblob.begin() + o_cls);
  if (n_classes) std::copy(class_ctrl, class_ctrl + n_classes, hostblob.begin() + o_cc);
  if (node_ok && N) memcpy(hostblob.data() + o_nodeok, node_ok, N);
  CAE_CUDA(cudaMemcpyAsync(e->d_fm_blob, hostblob.data(), o_in_end2 * 4, cudaMemcpyHostToDevice, e->stream));
  CAE_CUDA(cudaMemsetAsync(e->d_fm_blob + o_asg, 0xFF, (size_t)std::max(P, 1) * 4, e->stream));   // -1 = stays unschedulable
  CAE_CUDA(cudaMemsetAsync(e->d_fm_blob + o_out, 0, (off - o_out) * 4, e->stream));
  cae::FilterLaunch f{};
  f.runs = runs; f.n_pods = n_pods; f.last_index = last_index_in; f.break_on_failure = break_on_failure ? 1 : 0; f.nctrl = nctrl;
  f.run_off = e->d_fm_blob + o_run; f.pods = e->d_fm_blob + o_pods;
  f.hint = hint_node ? e->d_fm_blob + o_hint : nullptr;
  f.cls = sim_class ? e->d_fm_blob + o_cls : nullptr;
  f.class_ctrl = e->d_fm_blob + o_cc;
  f.node_ok = node_ok ? reinterpret_cast<const uint8_t*>(e->d_fm_blob + o_nodeok) : nullptr;
  f.assigned = e->d_fm_blob + o_asg; f.out = e->d_fm_blob + o_out; f.ctrl_cnt = e->d_fm_blob + o_cnt;
  f.class_mark = reinterpret_cast<uint8_t*>(e->d_fm_blob + o_mark);
  f.ctrl_over = reinterpret_cast<uint8_t*>(e->d_fm_blob + o_over);
  cudaEventRecord(e->ev0, e->stream);
  if (runs > 0 && cae::launch_filter(e, f)) return -1;
  cudaEventRecord(e->ev1, e->stream);
  int32_t out[4] = {last_index_raw, 0, 0, 0}, status = 0;
  if (P) CAE_CUDA(cudaMemcpyAsync(assigned_node, e->d_fm_blob + o_asg, (size_t)P * 4, cudaMemcpyDeviceToHost, e->stream));
  if (runs > 0) {
    CAE_CUDA(cudaMemcpyAsync(out, e->d_fm_blob + o_out, sizeof(out), cudaMemcpyDeviceToHost, e->stream));
    CAE_CUDA(cudaMemcpyAsync(&status, e->d_work_counter + 1, sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
  }
  CAE_CUDA(cudaStreamSynchronize(e->stream));
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev0, e->ev1);
  e->stats.estimate_ms = ms;
  if (status) { cae::set_error("placement log overflow in the filter pass"); return 1; }
  if (last_index_out) *last_index_out = out[3] ? out[0] : last_index_raw;
  if (overflowing_controllers) *overflowing_controllers = out[1];
  return 0;
}

int32_t cae_simulate_removals(cae_engine* h, int32_t n_cand, const int32_t* cand_node, const int32_t* cand_pod_off,
                              const int32_t* cand_pods, const int32_t* hint_node, const uint8_t* node_ok, int32_t persist,
                              int32_t max_removable, int32_t last_index_in, int32_t* result, int32_t trace_cap, int32_t* trace_off,
                              int32_t* trace_pod, int32_t* trace_node, int32_t* last_index_out) {
  Engine* e = reinterpret_cast<Engine*>(h);
  if (!e || !e->loaded) { cae::set_error("cae_simulate_removals before cae_load"); return -2; }
  auto bad = [](const char* what) { cae::set_error(std::string("cae_simulate_removals: ") + what); return -2; };
  if (n_cand < 0 || trace_cap < 0 || max_removable < 0 || last_index_in < 0 || !trace_off || !last_index_out ||
      (n_cand > 0 && (!cand_node || !cand_pod_off || !result)) || (trace_cap > 0 && (!trace_pod || !trace_node)))
    return bad("bad arguments");
  cudaSetDevice(e->cfg.device);
  const int P = e->P, N = e->N;
  if (n_cand == 0) { trace_off[0] = 0; *last_index_out = last_index_in; return 0; }
  if (cand_pod_off[0] != 0) return bad("cand_pod_off[0] must be 0");
  for (int c = 0; c < n_cand; ++c) {
    if (cand_node[c] < 0 || cand_node[c] >= N) return bad("candidate node index out of range");
    if (cand_pod_off[c + 1] < cand_pod_off[c]) return bad("cand_pod_off is not monotone");
  }
  const int n_pods = cand_pod_off[n_cand];
  if (n_pods > 0 && !cand_pods) return bad("bad arguments");
  std::vector<uint8_t> listed(std::max(P, 1), 0);
  for (int k = 0; k < n_pods; ++k) {
    const int pod = cand_pods[k];
    if (pod < 0 || pod >= P) return bad("pod index out of range");
    if (listed[pod]) return bad("a pod is listed under two candidates");
    listed[pod] = 1;
  }
  if (hint_node)
    for (int i = 0; i < P; ++i)
      if (hint_node[i] < -1 || hint_node[i] >= N) return bad("hinted node out of range");
  // runs of each candidate's own pods: consecutive pods of one spec and no hint (a hinted pod is a run of its own)
  std::vector<int32_t> run_off, cand_run_off(n_cand + 1);
  for (int c = 0; c < n_cand; ++c) {
    cand_run_off[c] = (int32_t)run_off.size();
    for (int k = cand_pod_off[c]; k < cand_pod_off[c + 1]; ++k) {
      const int pod = cand_pods[k];
      bool start = k == cand_pod_off[c];
      if (!start) {
        const int prev = cand_pods[k - 1];
        start = e->h_pend_spec[pod] != e->h_pend_spec[prev] || (hint_node && (hint_node[pod] >= 0 || hint_node[prev] >= 0));
      }
      if (start) run_off.push_back(k);
    }
  }
  const int runs = (int)run_off.size();
  cand_run_off[n_cand] = runs;
  run_off.push_back(n_pods);
  // one blob, in 4-byte words; inputs first (one upload), then outputs and work arrays
  auto words = [](size_t bytes) { return (bytes + 3) / 4; };
  auto even = [](size_t w) { return (w + 1) & ~(size_t)1; };   // 8-byte alignment for the int64 / uint64 arrays
  const int A1 = std::max(e->A, 1);
  size_t off = 0;
  const size_t o_st = off; off += cae::SIM_WORDS;
  const size_t o_cand = off; off += n_cand;
  const size_t o_poff = off; off += n_cand + 1;
  const size_t o_pods = off; off += std::max(n_pods, 1);
  const size_t o_run = off; off += runs + 1;
  const size_t o_crun = off; off += n_cand + 1;
  const size_t o_iota = off; off += P + 1;
  const size_t o_hint = off; off += hint_node ? P : 0;
  const size_t o_nodeok = off; off += node_ok ? words(N) : 0;
  const size_t o_in_end = off;
  const size_t o_res = off; off += n_cand;
  const size_t o_toff = off; off += n_cand + 1;
  const size_t o_tpod = off; off += std::max(trace_cap, 1);
  const size_t o_tnode = off; off += std::max(trace_cap, 1);
  const size_t o_out = off; off += 4;
  const size_t o_pos = off; off += N;
  const size_t o_at = off; off += N;
  const size_t o_gone = off; off += n_cand;
  const size_t o_mvt = off; off += N;
  const size_t o_mvn = off; off += std::max(P, 1);
  const size_t o_bksl = off; off += N;
  const size_t o_zero = off;   // zeroed: seen, nok
  const size_t o_seen = off; off += words(N);
  const size_t o_nok = off; off += words(N);
  const size_t o_ones = off;   // 0x01 bytes: present
  const size_t o_pres = off; off += words(N);
  const size_t o_mvh = off; off += N;   // 0xFF: -1
  off = even(off);
  const size_t o_bkp = off; off += (size_t)2 * N;
  const size_t o_bkf = off; off += (size_t)2 * A1 * N;
  if (off > e->fm_blob_words) {
    if (e->d_fm_blob) cudaFree(e->d_fm_blob);
    e->d_fm_blob = nullptr;
    e->fm_blob_words = 0;
    CAE_CUDA(cudaMalloc(&e->d_fm_blob, off * 4));
    e->fm_blob_words = off;
  }
  std::vector<int32_t> hostblob(o_in_end, 0);
  hostblob[o_st + cae::SIM_LI] = last_index_in;
  std::copy(cand_node, cand_node + n_cand, hostblob.begin() + o_cand);
  std::copy(cand_pod_off, cand_pod_off + n_cand + 1, hostblob.begin() + o_poff);
  if (n_pods) std::copy(cand_pods, cand_pods + n_pods, hostblob.begin() + o_pods);
  std::copy(run_off.begin(), run_off.end(), hostblob.begin() + o_run);
  std::copy(cand_run_off.begin(), cand_run_off.end(), hostblob.begin() + o_crun);
  for (int i = 0; i <= P; ++i) hostblob[o_iota + i] = i;
  if (hint_node) std::copy(hint_node, hint_node + P, hostblob.begin() + o_hint);
  if (node_ok && N) memcpy(hostblob.data() + o_nodeok, node_ok, N);
  int32_t* blob = e->d_fm_blob;
  CAE_CUDA(cudaMemcpyAsync(blob, hostblob.data(), o_in_end * 4, cudaMemcpyHostToDevice, e->stream));
  CAE_CUDA(cudaMemsetAsync(blob + o_zero, 0, (o_ones - o_zero) * 4, e->stream));
  CAE_CUDA(cudaMemsetAsync(blob + o_ones, 0x01, (o_mvh - o_ones) * 4, e->stream));
  CAE_CUDA(cudaMemsetAsync(blob + o_mvh, 0xFF, (size_t)N * 4, e->stream));
  CAE_CUDA(cudaMemsetAsync(blob + o_out, 0, 4 * 4, e->stream));
  cae::SimLaunch s{};
  s.n = n_cand; s.persist = persist ? 1 : 0; s.max_removable = max_removable; s.trace_cap = trace_cap;
  s.cand = blob + o_cand; s.pod_off = blob + o_poff; s.pods = blob + o_pods; s.cand_run_off = blob + o_crun; s.iota = blob + o_iota;
  s.result = blob + o_res; s.trace_off = blob + o_toff; s.trace_pod = blob + o_tpod; s.trace_node = blob + o_tnode; s.st = blob + o_st;
  s.present = reinterpret_cast<uint8_t*>(blob + o_pres); s.nok = reinterpret_cast<uint8_t*>(blob + o_nok);
  s.seen = reinterpret_cast<uint8_t*>(blob + o_seen);
  s.pos = blob + o_pos; s.at = blob + o_at; s.gone = blob + o_gone;
  s.mv_head = blob + o_mvh; s.mv_tail = blob + o_mvt; s.mv_next = blob + o_mvn; s.bk_slots = blob + o_bksl;
  s.bk_free = reinterpret_cast<int64_t*>(blob + o_bkf); s.bk_ports = reinterpret_cast<unsigned long long*>(blob + o_bkp);
  cae::FilterLaunch f{};
  f.runs = runs; f.n_pods = trace_cap; f.last_index = last_index_in; f.break_on_failure = 1; f.nctrl = 0;
  f.run_off = blob + o_run; f.pods = blob + o_pods;
  f.hint = hint_node ? blob + o_hint : nullptr;
  f.cls = nullptr; f.class_ctrl = blob + o_cand;   // no similarity classes: with breakOnFailure a mark never changes a result
  f.node_ok = node_ok ? reinterpret_cast<const uint8_t*>(blob + o_nodeok) : nullptr;
  f.assigned = nullptr; f.out = blob + o_out; f.ctrl_cnt = nullptr; f.class_mark = nullptr; f.ctrl_over = nullptr;
  f.sim = &s;
  cudaEventRecord(e->ev0, e->stream);
  if (cae::launch_filter(e, f)) return -1;
  cudaEventRecord(e->ev1, e->stream);
  int32_t out[4] = {0, 0, 0, 0}, status = 0;
  CAE_CUDA(cudaMemcpyAsync(result, blob + o_res, (size_t)n_cand * 4, cudaMemcpyDeviceToHost, e->stream));
  CAE_CUDA(cudaMemcpyAsync(trace_off, blob + o_toff, (size_t)(n_cand + 1) * 4, cudaMemcpyDeviceToHost, e->stream));
  CAE_CUDA(cudaMemcpyAsync(out, blob + o_out, sizeof(out), cudaMemcpyDeviceToHost, e->stream));
  CAE_CUDA(cudaMemcpyAsync(&status, e->d_work_counter + 1, sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
  CAE_CUDA(cudaStreamSynchronize(e->stream));
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev0, e->ev1);
  e->stats.estimate_ms = ms;
  if (status == 2) { cae::set_error("cae_simulate_removals: the trace needs more than trace_cap entries"); return 1; }
  if (status) { cae::set_error("placement log overflow in the filter pass"); return 1; }
  const int tr_n = trace_off[n_cand];
  if (tr_n > 0) {
    CAE_CUDA(cudaMemcpyAsync(trace_pod, blob + o_tpod, (size_t)tr_n * 4, cudaMemcpyDeviceToHost, e->stream));
    CAE_CUDA(cudaMemcpyAsync(trace_node, blob + o_tnode, (size_t)tr_n * 4, cudaMemcpyDeviceToHost, e->stream));
    CAE_CUDA(cudaStreamSynchronize(e->stream));
  }
  *last_index_out = out[0];
  return 0;
}

void* cae_stream(cae_engine* h) {
  Engine* e = reinterpret_cast<Engine*>(h);
  return e ? reinterpret_cast<void*>(e->stream) : nullptr;
}

static int ensure_xbuf(Engine* e) {
  if (e->d_xbuf) return 0;
  const size_t n = (size_t)4 * Engine::PEER_MAX * Engine::PEER_CAP + 16;   // [2 parities][PEER_MAX][PEER_CAP] (count, tag) slots + counters (feas.cu)
  CAE_CUDA(cudaMalloc(&e->d_xbuf, n * sizeof(int32_t)));
  CAE_CUDA(cudaMemset(e->d_xbuf, 0, n * sizeof(int32_t)));
  return 0;
}

int32_t cae_peer_handle(cae_engine* h, void* handle) {
  Engine* e = reinterpret_cast<Engine*>(h);
  if (!e || !handle) return -2;
  cudaSetDevice(e->cfg.device);
  if (ensure_xbuf(e)) return -1;
  static_assert(sizeof(cudaIpcMemHandle_t) == CAE_PEER_HANDLE_BYTES, "IPC handle size");
  cudaIpcMemHandle_t hd;
  CAE_CUDA(cudaIpcGetMemHandle(&hd, e->d_xbuf));
  memcpy(handle, &hd, sizeof(hd));
  return 0;
}

int32_t cae_peer_attach(cae_engine* h, const void* handles, int32_t world) {
  Engine* e = reinterpret_cast<Engine*>(h);
  if (!e || !handles) return -2;
  if (world < 1 || world > Engine::PEER_MAX || world != e->cfg.world_size) { cae::set_error("cae_peer_attach: bad world size"); return -2; }
  cudaSetDevice(e->cfg.device);
  if (ensure_xbuf(e)) return -1;
  for (int r = 0; r < world; ++r) {
    if (r == e->cfg.rank) { e->peer_base[r] = e->d_xbuf; continue; }
    cudaIpcMemHandle_t hd;
    memcpy(&hd, static_cast<const char*>(handles) + (size_t)r * CAE_PEER_HANDLE_BYTES, sizeof(hd));
    void* p = nullptr;
    CAE_CUDA(cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess));
    e->peer_base[r] = static_cast<int32_t*>(p);
  }
  e->peer_world = world;
  return 0;
}

void* cae_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 16, cudaHostAllocDefault) != cudaSuccess) return nullptr;
  return p;
}
void cae_host_free(void* p) { if (p) cudaFreeHost(p); }

}  // extern "C"
