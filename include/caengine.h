/*
 * caengine.h — C ABI of libcaengine.so, the B200-native scale-up simulation engine.
 *
 * This is the drop-in boundary for ONE hot path of the Cluster Autoscaler (reference
 * openshift/kubernetes-autoscaler, CA 1.35): pending pods x node-group templates through the
 * scheduler-framework Filter plugins, the first-fit-decreasing pack of BinpackingNodeEstimator and
 * the expander's option scoring.  The reference has no FFI of its own (100 % Go); every entry point
 * below names the Go interface/function it stands in for, and INTEGRATION.md shows the cgo stub a
 * maintainer would add on the reference side.
 *
 * Conventions
 *   - extern "C", plain pointers + lengths, caller-owned host buffers, no torch / C++ types.
 *   - every string of the Kubernetes object world (label keys/values, taint keys, namespaces, node
 *     names, host IPs, resource names) is interned by the caller into dense int32 ids; id spaces
 *     are per kind.  -1 means "absent/empty" wherever a field is optional.
 *   - all lists are CSR: xxx_off[n+1] offsets into flat arrays.  List id 0 of every list table is
 *     the empty list by convention (so a zero-initialised spec has no tolerations, ports, ...).
 *   - status codes: 0 ok; >0 "unsupported input, use the stock Go path" (never a guess);
 *     <0 fatal (CUDA / internal).  cae_last_error() returns a thread-local message.
 */
#ifndef CAENGINE_H_
#define CAENGINE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CAE_ABI_VERSION 1

/* Resource dimensions of a request / allocatable vector.
 * Mirrors framework.Resource (vendor/k8s.io/kubernetes/pkg/scheduler/framework/types.go:870-986):
 * MilliCPU, Memory, EphemeralStorage are fixed slots, ScalarResources are interned into 3..7. */
#define CAE_MAX_RES 8
#define CAE_RES_CPU 0 /* milli-cores  (Quantity.MilliValue) */
#define CAE_RES_MEM 1 /* bytes        (Quantity.Value)      */
#define CAE_RES_EPH 2 /* bytes                               */

/* label-selector requirement operators (apimachinery/pkg/labels/selector.go:247-294) */
enum cae_req_op {
  CAE_OP_IN = 0, /* also Equals / DoubleEquals */
  CAE_OP_NOT_IN = 1,
  CAE_OP_EXISTS = 2,
  CAE_OP_DOES_NOT_EXIST = 3,
  CAE_OP_GT = 4,
  CAE_OP_LT = 5
};

/* selector kinds: metav1.LabelSelectorAsSelector(nil) == Nothing, {} == Everything
 * (apimachinery/pkg/apis/meta/v1/helpers.go:36-42) */
enum cae_sel_kind { CAE_SEL_NOTHING = 0, CAE_SEL_REQS = 1 /* AND of reqs; zero reqs = Everything */ };

/* toleration operators (vendor/k8s.io/api/core/v1/toleration.go:52-77) */
enum cae_tol_op { CAE_TOL_EQUAL = 0 /* "" or Equal */, CAE_TOL_EXISTS = 1, CAE_TOL_LT = 2, CAE_TOL_GT = 3, CAE_TOL_INVALID = 4 };

/* taint effects; 0 is only legal on a toleration (empty effect = matches all) */
enum cae_effect { CAE_EFFECT_NONE = 0, CAE_EFFECT_NO_SCHEDULE = 1, CAE_EFFECT_PREFER_NO_SCHEDULE = 2, CAE_EFFECT_NO_EXECUTE = 3 };

enum cae_proto { CAE_PROTO_TCP = 0 /* "" or TCP */, CAE_PROTO_UDP = 1, CAE_PROTO_SCTP = 2 };

/* v1.NodeInclusionPolicy */
enum cae_inclusion { CAE_POLICY_IGNORE = 0, CAE_POLICY_HONOR = 1 };

/* First failing plugin in the default Filter order
 * (vendor/k8s.io/kubernetes/pkg/scheduler/apis/config/v1/default_plugins.go:34-52), as reported by
 * SchedulerPluginRunner.RunFiltersOnNode (simulator/clustersnapshot/predicate/plugin_runner.go:131-166).
 * The estimator branches on CAE_R_PTS_SKEW (binpacking_estimator.go:186,269-276). */
enum cae_reason {
  CAE_R_OK = 0,
  CAE_R_PREFILTER_NODEAFFINITY = 1, /* PreFilter failed (conflicting metadata.name terms) or PreFilterResult excluded the node */
  CAE_R_NODE_UNSCHEDULABLE = 2,
  CAE_R_NODE_NAME = 3,
  CAE_R_TAINT = 4,
  CAE_R_NODE_AFFINITY = 5,
  CAE_R_NODE_PORTS = 6,
  CAE_R_FIT = 7, /* NodeResourcesFit: too many pods and/or insufficient <resource> */
  CAE_R_PTS_MISSING_LABEL = 8, /* ErrReasonNodeLabelNotMatch */
  CAE_R_PTS_SKEW = 9,          /* ErrReasonConstraintsNotMatch */
  CAE_R_IPA_AFFINITY = 10,
  CAE_R_IPA_ANTI_AFFINITY = 11,
  CAE_R_IPA_EXISTING_ANTI_AFFINITY = 12
};

/* ------------------------------------------------------------------------------------------------
 * cae_objects — the cluster snapshot + pending pods + templates as interned columnar tables.
 * This is what the Go shim builds once per tick from ClusterSnapshot.ListNodeInfos(), the
 * []*equivalence.PodGroup of ScaleUp (core/scaleup/orchestrator/orchestrator.go:105) and the
 * per-node-group template NodeInfos (orchestrator.go:87 `nodeInfos`).
 * ---------------------------------------------------------------------------------------------- */
typedef struct cae_objects {
  int32_t abi_version; /* CAE_ABI_VERSION */
  int32_t num_res;     /* resource dims in use, 3..CAE_MAX_RES */

  /* value dictionary side table: decimal int64 parse of each label value (for Gt/Lt) */
  int32_t num_values;
  const uint8_t* value_is_int; /* [num_values] strconv.ParseInt(v,10,64) succeeded */
  const int64_t* value_int;    /* [num_values] */

  int32_t hostname_key; /* key id of "kubernetes.io/hostname", -1 if it never occurs */
  int32_t unschedulable_taint_key; /* key id of "node.kubernetes.io/unschedulable", -1 if it never occurs */

  /* namespaces: Namespace objects known to the lister (interpodaffinity/plugin.go:144-157) */
  int32_t num_namespaces;
  const int32_t* ns_labelset; /* [num_namespaces] label set of the Namespace object (0 if none) */
  const uint8_t* ns_exists;   /* [num_namespaces] the Namespace object exists in the lister */

  /* label sets (node labels, pod labels, namespace labels); pairs sorted by key id; set 0 = {} */
  int32_t num_labelsets;
  const int32_t* ls_off; /* [num_labelsets+1] */
  const int32_t* ls_key;
  const int32_t* ls_val;

  /* requirement pool shared by all selectors */
  int32_t num_reqs;
  const int32_t* req_key;     /* [num_reqs] */
  const int32_t* req_op;      /* [num_reqs] enum cae_req_op */
  const int32_t* req_val_off; /* [num_reqs+1] */
  const int32_t* req_vals;    /* value ids */

  /* label selectors: selector s = AND of reqs [sel_req_off[s], sel_req_off[s+1]) */
  int32_t num_selectors;
  const int32_t* sel_kind;    /* [num_selectors] enum cae_sel_kind */
  const int32_t* sel_req_off; /* [num_selectors+1] */

  /* required node affinity + nodeSelector of a pod
   * (component-helpers/scheduling/corev1/nodeaffinity/nodeaffinity.go:286-334) */
  int32_t num_naff;
  const int32_t* naff_nodesel;      /* [num_naff] selector id of spec.nodeSelector, -1 if empty */
  const uint8_t* naff_has_required; /* [num_naff] nodeAffinity.requiredDuringScheduling... != nil */
  const int32_t* naff_term_off;     /* [num_naff+1] -> terms, INCLUDING empty terms (they select nothing, :60-66) */
  int32_t num_naff_terms;
  const int32_t* term_expr_sel;  /* [num_naff_terms] selector over node labels, -1 if no matchExpressions */
  const int32_t* term_field_off; /* [num_naff_terms+1] -> matchFields on metadata.name */
  const int32_t* field_op;       /* CAE_OP_IN / CAE_OP_NOT_IN, exactly one value each */
  const int32_t* field_node_name; /* node-name id */

  /* toleration lists */
  int32_t num_tol_lists;
  const int32_t* tol_off; /* [num_tol_lists+1] */
  const int32_t* tol_key; /* -1 = empty key */
  const int32_t* tol_op;  /* enum cae_tol_op */
  const int32_t* tol_val; /* value id, -1 = "" */
  const int32_t* tol_effect;

  /* taint lists (all effects; the engine applies DoNotScheduleTaintsFilterFunc itself) */
  int32_t num_taint_lists;
  const int32_t* taint_off;
  const int32_t* taint_key;
  const int32_t* taint_val; /* -1 = "" */
  const int32_t* taint_effect;

  /* host-port lists: util.GetHostPorts(pod) (kubernetes/pkg/scheduler/util/utils.go:183) */
  int32_t num_port_lists;
  const int32_t* port_off;
  const int32_t* port_ip;    /* ip id; id 0 MUST be "0.0.0.0" (also used for "") */
  const int32_t* port_proto; /* enum cae_proto */
  const int32_t* port_num;   /* > 0 */

  /* DoNotSchedule topology spread constraint lists (podtopologyspread/common.go:87-129);
   * matchLabelKeys already merged into the selector by the caller (common.go:96-106) */
  int32_t num_pts_lists;
  const int32_t* pts_off;
  const int32_t* pts_max_skew;
  const int32_t* pts_key;
  const int32_t* pts_selector;
  const int32_t* pts_min_domains;          /* nil -> 1 */
  const int32_t* pts_node_affinity_policy; /* nil -> CAE_POLICY_HONOR */
  const int32_t* pts_node_taints_policy;   /* nil -> CAE_POLICY_IGNORE */

  /* required pod (anti)affinity term lists (kube-scheduler/framework/types.go:377-444) */
  int32_t num_aff_lists;
  const int32_t* aff_off;
  const int32_t* aterm_selector;
  const int32_t* aterm_key;        /* topology key */
  const int32_t* aterm_ns_off;     /* [num_aterms+1] explicit namespaces (own ns already defaulted in, :436-444) */
  const int32_t* aterm_ns;
  const int32_t* aterm_ns_selector; /* selector id over namespace labels; CAE_SEL_NOTHING selector if nil */
  int32_t num_aterms;

  /* pod specs: everything about a pod the Filter plugins read.  Request = PodRequests with
   * pod-level resources + overhead (component-helpers/resource/helpers.go:149-285), done by caller. */
  int32_t num_podspecs;
  const int32_t* ps_namespace;
  const int32_t* ps_labelset;
  const int64_t* ps_req; /* [num_podspecs * CAE_MAX_RES] */
  const int32_t* ps_tol_list;
  const int32_t* ps_naff;      /* -1: no nodeSelector and no required node affinity */
  const int32_t* ps_node_name; /* spec.nodeName id, -1 if empty */
  const int32_t* ps_port_list;
  const int32_t* ps_pts_list;
  const int32_t* ps_aff_list;  /* required pod affinity terms */
  const int32_t* ps_anti_list; /* required pod anti-affinity terms */
  const uint8_t* ps_terminating; /* DeletionTimestamp != nil */
  const uint8_t* ps_hostname_spread; /* isPodUsingHostNameTopologyKey (estimator/binpacking_estimator.go:280-292):
                                        ANY topologySpreadConstraint (also ScheduleAnyway) uses kubernetes.io/hostname */

  /* nodes: cluster nodes [0, num_cluster_nodes) in snapshot list order, then the node-group
   * templates [num_cluster_nodes, num_cluster_nodes + num_templates) */
  int32_t num_cluster_nodes;
  int32_t num_templates;
  const int32_t* node_name;
  const int32_t* node_labelset;
  const int32_t* node_taint_list;
  const uint8_t* node_unschedulable;
  const int64_t* node_alloc;        /* [nodes * CAE_MAX_RES] Status.Allocatable */
  const int32_t* node_allowed_pods; /* Allocatable["pods"], 0 if absent (types.go:920-921) */
  const int64_t* node_cap_cpu;      /* Status.Capacity cpu milli  (expander/waste/waste.go:86) */
  const int64_t* node_cap_mem;      /* Status.Capacity memory */
  const uint8_t* node_has_alloc_cpu; /* Allocatable has a cpu entry (decreasing_pod_orderer.go:77) */
  const uint8_t* node_has_alloc_mem;
  /* pods already on each node: resident pods for cluster nodes, DaemonSet/mirror pods for templates */
  const int32_t* node_pod_off; /* [nodes+1] */
  const int32_t* node_pod_spec;

  /* pending pods, grouped: group g = pods [group_off[g], group_off[g+1]) in Estimate order */
  int32_t num_groups;
  int32_t num_pending;
  const int32_t* group_off;
  const int32_t* pend_spec; /* [num_pending] podspec id */
} cae_objects;

/* ------------------------------------------------------------------------------------------------
 * Engine
 * ---------------------------------------------------------------------------------------------- */
typedef struct cae_engine cae_engine;

/* cae_config.flags */
#define CAE_CFG_PODS_PRESHARDED 1   /* world_size > 1: cae_objects holds ONLY this rank's pending pods (the caller sliced
                                       pend_spec / group_off); the dense pass covers all of them, the histogram exchange
                                       still runs over world_size ranks */
#define CAE_CFG_GATES_REPORTED 2    /* feature_gates is filled in; cae_create answers status 1 when a gate the engine
                                       hard-codes differs (the caller must then use the stock path) */
/* cae_config.feature_gates: the scheduler feature gates the path reads (vendor/k8s.io/kubernetes/pkg/scheduler/framework/
   plugins/feature/feature.go:27-52, read process-globally at plugin construction).  The engine implements:
   NodeInclusionPolicyInPodTopologySpread ON (podtopologyspread/common.go:43-58), TaintTolerationComparisonOperators OFF
   (Lt/Gt tolerations, api/core/v1/toleration.go:52-77), DRAExtendedResource OFF (noderesources/fit.go:208);
   MatchLabelKeysInPodTopologySpread is resolved by the caller when it builds the selectors (either value is accepted). */
#define CAE_GATE_NODE_INCLUSION_POLICY_IN_PTS 1
#define CAE_GATE_TAINT_TOLERATION_COMPARISON_OPERATORS 2
#define CAE_GATE_DRA_EXTENDED_RESOURCE 4
#define CAE_GATE_MATCH_LABEL_KEYS_IN_PTS 8

typedef struct cae_config {
  int32_t abi_version;
  int32_t device;          /* CUDA device ordinal */
  int32_t rank;            /* this process' shard index (pods for feasibility, templates for estimate) */
  int32_t world_size;      /* number of shards */
  int32_t want_reasons;    /* also produce the dense reason matrix in cae_feasibility */
  int32_t flags;           /* CAE_CFG_* */
  int32_t feature_gates;   /* CAE_GATE_* as utilfeature.DefaultFeatureGate reports them on the Go side (with CAE_CFG_GATES_REPORTED) */
  int32_t reserved[9];
} cae_config;

typedef struct cae_stats {
  int64_t evals;            /* pod x template predicate evaluations of the last cae_feasibility */
  double feasibility_ms;    /* device time of the feasibility pass (CUDA events) */
  double estimate_ms;       /* device time of order + pack */
  double expander_ms;
  double h2d_ms, d2h_ms;
  int64_t h2d_bytes, d2h_bytes;
  int64_t kernel_launches;  /* kernels launched by the engine since creation */
  int64_t estimate_group_steps; /* (template, schedulable group) pairs the last cae_estimate_all walked on this rank */
  int64_t reserved[7];
} cae_stats;

/* Replaces: estimator.NewBinpackingNodeEstimator / EstimatorBuilder (estimator/estimator.go:59-75). */
int32_t cae_create(const cae_config* cfg, cae_engine** out);
void cae_destroy(cae_engine* e);
const char* cae_last_error(void);
const char* cae_version(void);

/* Replaces: ClusterSnapshot.SetClusterState + TemplateNodeInfoRegistry (static_autoscaler.go:371-379)
 * as seen by the path.  Flattens the objects into SoA device buffers: interns pod/nodes into
 * classes, compiles selectors, uploads.  Must be called once per tick before the calls below.
 * The engine keeps no pointer into `objs` after return. */
int32_t cae_load(cae_engine* e, const cae_objects* objs);

/* Dense feasibility matrix: every pending pod (not just exemplars) x every template, on the forked
 * snapshot with only that template node added.
 * Replaces: ScaleUpOrchestrator.SchedulablePodGroups (orchestrator.go:603-638) ->
 *           PredicateSnapshot.CheckPredicates (predicate_snapshot.go:244) -> RunFiltersOnNode.
 *   fit_bits  [T][ceil(Plocal/32)] uint32, bit p%32 of word p/32 set iff pod p fits template t
 *             (template-major: one warp ballot = one word).  May be NULL.
 *   reasons   [T][Plocal] uint8 enum cae_reason, only if cfg.want_reasons.  May be NULL.
 *   fit_count [T] int32 number of local pods that fit template t (caller all-reduces over shards).
 * Plocal = pods of this shard (block partition of [0,P) over world_size). */
/* The per-tick delta: new pending-pod rows against the snapshot that is already resident.
 * Replaces: the part of DeltaSnapshotStore.SetClusterState / Fork-Commit (simulator/clustersnapshot/store/delta.go:499-588)
 * that changes between two scale-up loops when nodes, templates and the set of pod specs are unchanged — the list of
 * pending pods and their grouping.  Everything derived from the object world (interned tables, class matrices, rank
 * dictionaries, topology counters) stays in HBM; only pend_spec[num_pending] and group_off[num_groups + 1] travel
 * (4 B per pod), the per-pod rows and group records are re-derived on the device.
 * Status 2 = the delta does not apply (a pod spec that was not pending at the last cae_load, more pods / groups than the
 * resident buffers hold, or — with topology-spread / inter-pod-affinity counters in the snapshot — a different
 * group -> spec sequence): call cae_load with the full snapshot instead.  Nothing is changed in that case. */
int32_t cae_load_pending(cae_engine* e, int32_t num_pending, const int32_t* pend_spec, int32_t num_groups, const int32_t* group_off);

int32_t cae_feasibility(cae_engine* e, uint32_t* fit_bits, uint8_t* reasons, int32_t* fit_count);

/* Exemplar feasibility, what the orchestrator itself asks: group exemplar x template.
 *   reasons [T][E] uint8 */
int32_t cae_feasibility_groups(cae_engine* e, uint8_t* reasons);

/* Bin-packing estimate for every template at once.
 * Replaces: BinpackingNodeEstimator.Estimate (estimator/binpacking_estimator.go:97-139) called per
 * node group from ComputeExpansionOption (orchestrator.go:462-520), incl. DecreasingPodOrderer.Order
 * (decreasing_pod_orderer.go:46-88) and the node-count part of thresholdBasedEstimationLimiter
 * (threshold_based_limiter.go:34-69).
 *   max_nodes   [T] limiter result per template: <0 no node may be added, 0 unlimited, >0 cap.
 *   node_count  [T] len(newNodesWithPods)
 *   pod_count   [T] len(scheduledPods)
 *   sched_count [T][E] pods of group g scheduled on template t — always a prefix of the group,
 *               so with `order` this is the reference's scheduledPods list.  May be NULL.
 *   order       [T][E] group ids in processing order, -1 padded (groups not feasible are absent).
 *               May be NULL.
 * Only templates of this shard (block partition of [0,T)) are computed; other rows are zero so a
 * sum all-reduce over shards assembles the result. */
int32_t cae_estimate_all(cae_engine* e, const int32_t* max_nodes, int32_t* node_count,
                         int32_t* pod_count, int32_t* sched_count, int32_t* order);
/* The same with SchedulerPluginRunner.lastIndex (simulator/clustersnapshot/predicate/plugin_runner.go:34,81,123) carried per
 * template: last_index_in[t] (>= 0, NULL = 0) is the runner's value when the Estimate of template t starts — it may be RAW,
 * i.e. left by a longer node list: the reference uses it modulo the current list length until a scan places a pod —
 * last_index_out[t] its value when that Estimate returns (it survives the snapshot's Revert).  cae_estimate_all starts every
 * Estimate at 0, which makes the node groups independent; a caller that wants ONE long-lived runner across node groups
 * (SURVEY App. A.11) chains the calls: out[t] of one call is in[t+1] of the next. */
int32_t cae_estimate_all_ex(cae_engine* e, const int32_t* max_nodes, const int32_t* last_index_in, int32_t* node_count,
                            int32_t* pod_count, int32_t* sched_count, int32_t* order, int32_t* last_index_out);

/* Expander filters over the options produced by cae_estimate_all (one option per template with
 * node_count > 0).  Replaces: expander.Filter.BestOptions for least-waste / most-pods / least-nodes
 * (expander/waste/waste.go:37-73, mostpods/mostpods.go:33-54, leastnodes/leastnodes.go:35-61) and
 * the chain (expander/factory/chain.go:36-45) up to, not including, the random fallback. */
enum cae_expander { CAE_EXP_LEAST_WASTE = 0, CAE_EXP_MOST_PODS = 1, CAE_EXP_LEAST_NODES = 2, CAE_EXP_PRICE = 3, CAE_EXP_PRIORITY = 4 };
int32_t cae_expander_best(cae_engine* e, const int32_t* chain, int32_t chain_len,
                          const int32_t* node_count, const int32_t* pod_count,
                          const int32_t* sched_count, /* [T][E]; NULL = use the device-resident result of
                                                         the last cae_estimate_all (single shard) */
                          uint8_t* best_mask /* [T] 1 = in the surviving option set */,
                          double* waste_score /* [T], may be NULL */);

/* The step BEFORE the scale-up path: filterOutSchedulablePodListProcessor.filterOutSchedulableByPacking ->
 * HintingSimulator.TrySchedulePods on the cluster snapshot (cluster-autoscaler/core/podlistprocessor/
 * filter_out_schedulable.go:96-126, simulator/scheduling/hinting_simulator.go:53-135), including the
 * SimilarPodsScheduling shortcut (simulator/scheduling/similar_pods.go:59-112).  Pending pods that fit on the free
 * capacity of EXISTING nodes are placed there, one by one in `pod_order`, and do not need a scale-up.
 *   pod_order [n_pods]     pending-pod indices in processing order: the caller's priority sort (Go's sort.Slice is
 *                          unstable, so the order among equal priorities is the caller's); fastest when identical
 *                          pods are adjacent
 *   hint_node [num_pending] cluster node hinted for a pod (Hints.Get), -1 = none; NULL = no hints
 *   sim_class [num_pending] id of (controller UID, labels, spec) for pods owned by a non-DaemonSet controller, -1
 *                          otherwise; NULL = none.  class_ctrl [n_classes] = controller id (>= 0) of a class
 *   node_ok [N]            isNodeAcceptable, NULL = scheduling.ScheduleAnywhere
 *   last_index_in          SchedulerPluginRunner.lastIndex before the call (0 for a fresh runner)
 * Outputs: assigned_node [num_pending] = cluster node index, -1 = stays unschedulable (also for pods not in
 * pod_order); the runner's lastIndex afterwards; SimilarPodsScheduling.OverflowingControllerCount().
 * Uses the tables of the last cae_load (its templates are ignored); does not change the estimator's results. */
int32_t cae_filter_schedulable(cae_engine* e, const int32_t* pod_order, int32_t n_pods, const int32_t* hint_node,
                               const int32_t* sim_class, const int32_t* class_ctrl, int32_t n_classes, const uint8_t* node_ok,
                               int32_t last_index_in, int32_t break_on_failure, int32_t* assigned_node,
                               int32_t* last_index_out, int32_t* overflowing_controllers);

/* The scale-down consumer of the same pass, batched: the planner's loop over the unneeded-node candidates of a tick
 * (categorizeNodes, core/scaledown/planner/planner.go) calling RemovalSimulator.SimulateNodeRemoval (simulator/cluster.go:126-217)
 * for each one in turn, on ONE snapshot, in one call.  Candidate c leaves the snapshot (its residents, DaemonSet pods
 * included, stop counting for topology spread / inter-pod affinity), its pods are tried by HintingSimulator.TrySchedulePods
 * with breakOnFailure on the remaining nodes (findPlaceFor, :184-217), and it is removable iff every pod is placed.
 *   cand_node [n_cand]         cluster node index of each candidate, in the planner's order
 *   cand_pod_off [n_cand+1], cand_pods   pending-pod indices of each candidate's pods to move (GetPodsToMove), in order; the
 *                              pending rows of the last cae_load are these pods with nodeName cleared (its templates are ignored);
 *                              a pod may be listed under one candidate only
 *   hint_node [num_pending]    Hints.Get of each pod as a cluster node index, -1 = none; NULL = no hints.  A hint naming a
 *                              node out of the snapshot is ignored, like a hint naming a deleted node (hinting_simulator.go:88-91)
 *   node_ok [N]                the destination map (nodes the pods may go to), NULL = every node
 *   persist                    persistSuccessfulSimulations: a removable candidate stays removed and its pods stay where they
 *                              were placed for the rest of the call (withForkedSnapshot Commit, :169-182); pods placed on a later
 *                              candidate are then part of ITS pods to move, after its own, in placement order.  Any other
 *                              simulation is reverted.  The loaded snapshot itself never changes.
 *   max_removable              unneededNodesLimit: once that many candidates are removable the rest are not simulated; 0 = no limit
 *   last_index_in              SchedulerPluginRunner.lastIndex before the loop (raw, >= 0); ONE runner serves every simulation
 * Outputs: result [n_cand] 0 removable, 1 NoPlaceToMovePods, 2 NoNodeInfo (removed by an earlier persisted simulation, or
 * listed twice), -1 not simulated (after max_removable).  The trace: trace_off [n_cand+1] into trace_pod / trace_node
 * [trace_cap]: for every simulated candidate the exact pod list TrySchedulePods received (NodeToBeRemoved.PodsToReschedule)
 * and the node each pod went to, -1 = not placed or not tried after the first failure; the caller sets its hints from it.
 * last_index_out: the runner's lastIndex after the loop.
 * Status 1: the trace needs more than trace_cap entries (the message names it; a trace never needs more than
 * n_cand x num_pending) or the placement log overflowed; -2: malformed input.  No other engine result changes. */
int32_t cae_simulate_removals(cae_engine* e, int32_t n_cand, const int32_t* cand_node, const int32_t* cand_pod_off,
                              const int32_t* cand_pods, const int32_t* hint_node, const uint8_t* node_ok, int32_t persist,
                              int32_t max_removable, int32_t last_index_in, int32_t* result, int32_t trace_cap, int32_t* trace_off,
                              int32_t* trace_pod, int32_t* trace_node, int32_t* last_index_out);

/* The two halves of cae_expander_best for templates sharded over ranks (no [T][E] matrix ever leaves a GPU):
 * cae_waste_scores returns the least-waste score (expander/waste/waste.go:44-72) of this rank's template shard from
 * the device-resident result of the last cae_estimate_all, 0.0 for the rows of other ranks, so that a SUM all-reduce of
 * double[T] assembles the vector bit-exactly; cae_expander_chain runs the filter chain on the host from the all-reduced
 * node_count | pod_count and that vector (no engine state is read). */
int32_t cae_waste_scores(cae_engine* e, double* waste_score /* [T] */);
int32_t cae_expander_chain(const int32_t* chain, int32_t chain_len, int32_t num_templates, const int32_t* node_count,
                           const int32_t* pod_count, const double* waste_score, uint8_t* best_mask /* [T] */);

/* Price expander (expander/price/price.go:90-183).  The cloud provider's PricingModel and the preferred-node provider
 * stay on the Go side; the shim evaluates them once per tick into plain vectors, the engine computes the option score
 *   score = suppressedUnfitness x (NodePrice x nodeCount + stabilization) / (sum of PodPrice + stabilization)  [x 2 if !Exist()]
 * in float64 exactly as Go evaluates it on amd64 (no fused multiply-add; the pod prices are ADDED ONE POD AT A TIME in
 * scheduling order, price.go:128-135; math.Tanh restated from Go's pure-Go tanh.go / exp.go, price.go:146).
 *   node_price [T]            pricingModel.NodePrice(template node, now, now + 1h)
 *   pod_price [num_podspecs]  pricingModel.PodPrice of a pod of that spec (pods of a group are equivalent)
 *   unfitness [T] or NULL     NodeUnfitness(preferredNode, node); NULL = SimpleNodeUnfitness (preferred.go:87-92) from
 *                             preferred_cpu_milli and the template's cpu capacity
 *   has_gpu [T]               gpu.NodeHasGpu(GPULabel, node): unfitness is overridden by 1000 (price.go:150-153)
 *   exists [T]                NodeGroup.Exist(); a group yet to be created costs x 2 (price.go:157-159)
 *   price_error [T] or NULL   NodePrice / PodPrice returned an error: the option is skipped (price.go:120,130) */
typedef struct cae_price_inputs {
  const double* node_price;
  const double* pod_price;
  const double* unfitness;
  const uint8_t* has_gpu;
  const uint8_t* exists;
  const uint8_t* price_error;
  double stabilization_price;
  int64_t preferred_cpu_milli;
} cae_price_inputs;
/* score [T] of every option (0.0 where node_count == 0).  node_count / sched_count / order as returned by
 * cae_estimate_all; all three NULL = score the device-resident result of the last cae_estimate_all (rows of other ranks
 * come back 0.0, so a sum all-reduce assembles the vector like cae_waste_scores). */
int32_t cae_price_scores(cae_engine* e, const cae_price_inputs* in, const int32_t* node_count, const int32_t* sched_count,
                         const int32_t* order, double* score);
/* The filter chain over assembled vectors, with the price and priority filters:
 *   price_score / price_error  from cae_price_scores / cae_price_inputs (needed when the chain holds CAE_EXP_PRICE)
 *   priority [T]               highest priority of the ConfigMap whose regexp list matches the node group id, < 0 = the id
 *                              matches no entry (expander/priority/priority.go:119-165; the regexps are the shim's) */
int32_t cae_expander_chain_ex(const int32_t* chain, int32_t chain_len, int32_t num_templates, const int32_t* node_count,
                              const int32_t* pod_count, const double* waste_score, const double* price_score,
                              const uint8_t* price_error, const int32_t* priority, uint8_t* best_mask /* [T] */);

int32_t cae_get_stats(cae_engine* e, cae_stats* out);

/* Raw device pointers of the engine's result buffers, for zero-copy collectives (torch.distributed
 * / NCCL on the caller's side): 0 = fit_count int32[T], 1 = node_count|pod_count int32[2T]. */
void* cae_device_buffer(cae_engine* e, int32_t which, size_t* bytes);

/* The CUDA stream (cudaStream_t) every launch and copy of this engine is ordered on, for callers that order
 * their own device work with it (a collective on the result buffers, an L2 flush in a benchmark). */
void* cae_stream(cae_engine* e);

/* Fused histogram exchange for the multi-GPU dense pass (one process per GPU, one node).  Each engine owns
 * an exchange buffer in its HBM; after cae_peer_attach the LAST thread block of every cae_feasibility
 * launch writes the rank's per-template fit counts into its slot of every rank's buffer over NVLink (stores
 * to CUDA-IPC mapped peer memory), signals arrival, waits for all ranks and publishes the summed histogram
 * as fit_count — inside the same kernel, no collective launch.  Equivalent to all_reduce(sum, int32[T]).
 * Every rank must call cae_feasibility the same number of times; a rank that never arrives makes the others
 * fail with status < 0 after ~2 s instead of hanging.
 *   cae_peer_handle: writes the 64-byte CUDA IPC handle of this engine's exchange buffer.
 *   cae_peer_attach: handles of all ranks in rank order (world * 64 bytes). */
#define CAE_PEER_HANDLE_BYTES 64
int32_t cae_peer_handle(cae_engine* e, void* handle);
int32_t cae_peer_attach(cae_engine* e, const void* handles, int32_t world);

/* Page-locked host memory for the caller's large input / output buffers (fit_bits, reasons): copies
 * to and from pinned memory run at full PCIe speed and asynchronously. */
void* cae_host_alloc(size_t bytes);
void cae_host_free(void* p);

#ifdef __cplusplus
}
#endif
#endif /* CAENGINE_H_ */
