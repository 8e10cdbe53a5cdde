"""Host-side mirror of the scale-down consumer of the same primitive (SURVEY §8f rank 3):
``RemovalSimulator.SimulateNodeRemoval`` / ``findPlaceFor`` (``cluster-autoscaler/simulator/cluster.go:126-217``).

``findPlaceFor`` is ``HintingSimulator.TrySchedulePods(snapshot without the node, its pods, isCandidateNode,
breakOnFailure=true)`` — exactly what ``cae_filter_schedulable`` runs on the GPU — so this file is bookkeeping only:
take the node out of the snapshot, clear ``spec.nodeName`` of the pods to move, ask the simulator, and (optionally)
persist a successful simulation into the snapshot.  Which pods must move (``GetPodsToMove``: drainability rules, PDBs)
is outside §8; the default here is every pod that is not DaemonSet-owned, or the caller passes the list.

``SimulateNodeRemovals`` is the planner's loop over the candidates of a tick in ONE engine call (``cae_simulate_removals``):
one encoding of the cluster, the candidates simulated in order on the GPU, the hints / lastIndex / committed snapshot
rebuilt here from the returned trace.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from .encode import encode
from .engine import Engine
from .estimator import shared_engine
from .objects import Namespace, Node, NodeInfo, Pod
from .podlistprocessor import HintingSimulator, HintKeyFromPod, Hints
from .podutil import build_pod_groups

# simulator/cluster.go:55-95
NoReason, NoPlaceToMovePods, NoNodeInfo = "NoReason", "NoPlaceToMovePods", "NoNodeInfo"


@dataclass
class NodeToBeRemoved:
    """simulator/cluster.go:41-51."""
    node: Node
    pods_to_reschedule: List[Pod] = field(default_factory=list)
    daemonset_pods: List[Pod] = field(default_factory=list)


@dataclass
class UnremovableNode:
    """simulator/cluster.go:53-58."""
    node: Node
    reason: str


class RemovalSimulator:
    def __init__(self, cluster_snapshot: List[NodeInfo], persistSuccessfulSimulations: bool = False,
                 engine: Optional[Engine] = None, schedulingSimulator: Optional[HintingSimulator] = None) -> None:
        self.cluster = cluster_snapshot          # mutated only when a successful simulation is persisted
        self.canPersist = persistSuccessfulSimulations
        self.schedulingSimulator = schedulingSimulator or HintingSimulator(engine)

    def SimulateNodeRemoval(self, nodeName: str, destinationMap: Dict[str, bool], pods_to_move: Optional[Sequence[Pod]] = None,
                            namespaces: Sequence[Namespace] = ()) -> Tuple[Optional[NodeToBeRemoved], Optional[UnremovableNode]]:
        """Exactly one of the two results is set (cluster.go:126-167)."""
        ni = next((n for n in self.cluster if n.node.name == nodeName), None)
        if ni is None:
            return None, UnremovableNode(Node(name=nodeName), NoNodeInfo)
        daemonset = [p for p in ni.pods if p.owner_kind == "DaemonSet"]
        to_move = list(pods_to_move) if pods_to_move is not None else [p for p in ni.pods if p.owner_kind != "DaemonSet"]
        placements = self._findPlaceFor(ni, to_move, destinationMap, namespaces)
        if placements is None:
            return None, UnremovableNode(ni.node, NoPlaceToMovePods)
        if self.canPersist:                       # withForkedSnapshot: Commit (cluster.go:169-182)
            self.cluster.remove(ni)
            by_name = {n.node.name: n for n in self.cluster}
            for pod, node_name in placements:
                by_name[node_name].pods.append(pod)
        return NodeToBeRemoved(ni.node, to_move, daemonset), None

    def _findPlaceFor(self, removed: NodeInfo, pods: Sequence[Pod], nodes: Dict[str, bool], namespaces):
        """cluster.go:184-217: the node leaves the snapshot first so that it does not take part in topology spreading."""
        removed_name = removed.node.name
        snapshot = [n for n in self.cluster if n is not removed]
        newpods = []
        for p in pods:
            q = p.clone()
            q.node_name = ""
            newpods.append(q)
        if not newpods:
            return []
        statuses, _ = self.schedulingSimulator.TrySchedulePods(
            snapshot, newpods, lambda ni: ni.node.name != removed_name and bool(nodes.get(ni.node.name)), True, namespaces)
        if len(statuses) != len(newpods):
            return None                           # "can reschedule only %d out of %d pods"
        return [(s.pod, s.node_name) for s in statuses]

    def SimulateNodeRemovals(self, candidates: Sequence[str], destinationMap: Dict[str, bool],
                             pods_to_move: Optional[Dict[str, Sequence[Pod]]] = None, namespaces: Sequence[Namespace] = (),
                             max_removable: int = 0) -> List[Tuple[Optional[NodeToBeRemoved], Optional[UnremovableNode]]]:
        """The planner's loop (categorizeNodes, core/scaledown/planner/planner.go) of SimulateNodeRemoval over `candidates`,
        in order, in ONE engine call (cae_simulate_removals): the same pairs, hints, lastIndex and (with persist) committed
        snapshot as calling SimulateNodeRemoval(name, destinationMap) for each name in turn, except that a name listed twice
        gets NoNodeInfo.  max_removable (unneededNodesLimit, 0 = none): once that many are removable the rest are not
        simulated and come back as (None, None).  pods_to_move maps a name to that node's own pods to move (default: its
        non-DaemonSet pods); pods a persisted simulation placed on a later candidate are moved with it, after its own."""
        x = prepare_removals(self.cluster, candidates, destinationMap, self.schedulingSimulator.hints, pods_to_move, namespaces)
        eng = self.schedulingSimulator.engine or shared_engine()
        if x.cand_node:
            eng.load(x.enc)
            result, toff, tpod, tnode, li = eng.simulate_removals(x.cand_node, x.cand_pod_off, x.cand_pods, x.hint, x.node_ok,
                                                                  self.canPersist, max_removable, self.schedulingSimulator.last_index)
        else:
            result, toff, tpod, tnode, li = [], [0], [], [], self.schedulingSimulator.last_index
        return self._apply_removals(x, result, toff, tpod, tnode, li, max_removable)

    def _apply_removals(self, x: "RemovalInputs", result, trace_off, trace_pod, trace_node, last_index: int,
                        max_removable: int = 0) -> List[Tuple[Optional[NodeToBeRemoved], Optional[UnremovableNode]]]:
        """Turns the engine's answer into what the sequential loop returns and leaves behind: the pairs, the hints of every
        placement (failed simulations included), lastIndex and, with persist, the committed snapshot."""
        hints = self.schedulingSimulator.hints
        out: List[Tuple[Optional[NodeToBeRemoved], Optional[UnremovableNode]]] = []
        removable = 0
        for k, name in enumerate(x.names):
            j = x.engine_pos[k]
            if max_removable and removable >= max_removable:
                out.append((None, None))                  # not simulated
                continue
            if j < 0:                                     # not in the snapshot
                out.append((None, UnremovableNode(Node(name=name), NoNodeInfo)))
                continue
            r = int(result[j])
            ni = x.cluster[x.cand_node[j]]
            if r == -1:
                out.append((None, None))
                continue
            if r == 2:
                out.append((None, UnremovableNode(Node(name=name), NoNodeInfo)))
                continue
            seg = range(int(trace_off[j]), int(trace_off[j + 1]))
            pods = [x.clones[int(trace_pod[i])] for i in seg]
            placed = []
            for i in seg:
                node = int(trace_node[i])
                if node >= 0:
                    hints.Set(HintKeyFromPod(x.clones[int(trace_pod[i])]), x.cluster[node].node.name)
                    placed.append((x.clones[int(trace_pod[i])], x.cluster[node].node.name))
            if r == 1:
                out.append((None, UnremovableNode(ni.node, NoPlaceToMovePods)))
                continue
            removable += 1
            own = set(id(p) for p in x.own_pods[j])
            to_move = [x.originals[int(trace_pod[i])] if id(x.originals[int(trace_pod[i])]) in own else pods[n]
                       for n, i in enumerate(seg)]
            if self.canPersist:                           # withForkedSnapshot: Commit (cluster.go:169-182)
                self.cluster.remove(ni)
                by_name = {n.node.name: n for n in self.cluster}
                for pod, node_name in placed:
                    by_name[node_name].pods.append(pod.clone())
            out.append((NodeToBeRemoved(ni.node, to_move, [p for p in ni.pods if p.owner_kind == "DaemonSet"]), None))
        self.schedulingSimulator.last_index = last_index
        return out

    def DropOldHints(self) -> None:
        self.schedulingSimulator.DropOldHints()


@dataclass
class RemovalInputs:
    """What cae_simulate_removals takes, built from objects (the Go shim builds the same from the planner's candidates)."""
    enc: object
    cluster: List[NodeInfo]            # the snapshot as loaded (node index = position)
    names: List[str]                   # the candidates as asked
    engine_pos: List[int]              # candidate k -> its row in cand_node, -1 = not in the snapshot (NoNodeInfo on the host)
    cand_node: List[int]
    cand_pod_off: List[int]
    cand_pods: List[int]
    own_pods: List[List[Pod]]          # per engine candidate: the node's own pods to move
    originals: List[Pod]               # pending-pod index -> the pod as the caller holds it
    clones: List[Pod]                  # pending-pod index -> the clone with nodeName cleared that is tried
    hint: Optional[np.ndarray]
    node_ok: Optional[np.ndarray]


def prepare_removals(cluster_snapshot: Sequence[NodeInfo], candidates: Sequence[str], destinationMap: Dict[str, bool],
                     hints: Optional[Hints] = None, pods_to_move: Optional[Dict[str, Sequence[Pod]]] = None,
                     namespaces: Sequence[Namespace] = ()) -> RemovalInputs:
    """One encoding for the whole loop: the cluster as it is, pending rows = every candidate's own pods to move (clones with
    nodeName cleared), the candidates as node indices in CSR form.  A name not in the snapshot stays on the host (NoNodeInfo);
    a name listed again goes to the engine with no pods (the engine answers NoNodeInfo)."""
    cluster = list(cluster_snapshot)
    node_index = {ni.node.name: i for i, ni in enumerate(cluster)}
    names = list(candidates)
    engine_pos, cand_node, own_pods, seen = [], [], [], set()
    for name in names:
        i = node_index.get(name)
        if i is None:
            engine_pos.append(-1)
            continue
        engine_pos.append(len(cand_node))
        cand_node.append(i)
        if name in seen:
            own_pods.append([])
            continue
        seen.add(name)
        ni = cluster[i]
        if pods_to_move is not None and name in pods_to_move:
            own = list(pods_to_move[name])
            if any(p.owner_kind == "DaemonSet" for p in own):
                raise ValueError("pods_to_move of %s holds a DaemonSet pod: DaemonSet pods are not moved" % name)
        else:
            own = [p for p in ni.pods if p.owner_kind != "DaemonSet"]
        own_pods.append(own)
    originals = [p for own in own_pods for p in own]
    clones = []
    for p in originals:
        q = p.clone()
        q.node_name = ""
        clones.append(q)
    groups = build_pod_groups(clones)
    enc = encode(cluster, [], groups, namespaces)
    row: Dict[int, int] = {}
    k = 0
    for g in groups:
        for p in g.pods:
            row[id(p)] = k
            k += 1
    by_row_orig: List[Optional[Pod]] = [None] * len(clones)
    by_row_clone: List[Optional[Pod]] = [None] * len(clones)
    cand_pod_off, cand_pods = [0], []
    n = 0
    for own in own_pods:
        for _ in own:
            r = row[id(clones[n])]
            by_row_orig[r], by_row_clone[r] = originals[n], clones[n]
            cand_pods.append(r)
            n += 1
        cand_pod_off.append(len(cand_pods))
    hint = np.full(enc.P, -1, np.int32)
    if hints is not None:
        for r, p in enumerate(by_row_clone):
            h = hints.Get(HintKeyFromPod(p))
            if h is not None and h in node_index:
                hint[r] = node_index[h]
    ok = np.array([1 if destinationMap.get(ni.node.name) else 0 for ni in cluster], np.uint8)
    return RemovalInputs(enc, cluster, names, engine_pos, cand_node, cand_pod_off, cand_pods, own_pods, by_row_orig, by_row_clone,
                         hint if (hint >= 0).any() else None, None if ok.all() else ok)


NewRemovalSimulator = RemovalSimulator
