"""Python binding of the engine's C ABI (``include/caengine.h``) — what the cgo shim does in Go.

There is no CPU path here: if ``libcaengine.so`` or a CUDA device is missing every call raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np

from . import capi
from .encode import EncodedObjects


class EngineError(RuntimeError):
    pass


class EngineUnsupported(EngineError):
    """Status > 0: the input uses something the engine refuses; the caller must use the stock path."""


class PinnedArray:
    """numpy view over page-locked memory from cae_host_alloc."""

    def __init__(self, lib, shape, dtype) -> None:
        self._lib = lib
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        self._ptr = lib.cae_host_alloc(max(self.nbytes, 16))
        if not self._ptr:
            raise EngineError("cae_host_alloc failed")
        buf = (C.c_uint8 * max(self.nbytes, 1)).from_address(self._ptr)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def close(self) -> None:
        if self._ptr:
            self.array = None
            self._lib.cae_host_free(self._ptr)
            self._ptr = None

    def __del__(self) -> None:
        try:
            self.close()
        except Exception:
            pass


def shard_pods(P: int, rank: int, world_size: int) -> Tuple[int, int]:
    """Block partition of the pending pods for the dense pass; shard starts are multiples of 32 so the
    template-major bit rows of the ranks concatenate word by word (must match do_load in csrc/api.cu)."""
    b = (P * rank // world_size) // 32 * 32
    e = P * (rank + 1) // world_size
    if rank + 1 < world_size:
        e = e // 32 * 32
    return b, e


def shard_templates(T: int, rank: int, world_size: int) -> Tuple[int, int]:
    """Block partition of the templates for the pack: rows of other ranks stay zero, so a sum
    all-reduce of node_count|pod_count assembles the result."""
    return T * rank // world_size, T * (rank + 1) // world_size


class Engine:
    def __init__(self, device: int = 0, rank: int = 0, world_size: int = 1, want_reasons: bool = False,
                 pods_presharded: bool = False, feature_gates: Optional[int] = None) -> None:
        self.lib = capi.load_engine_lib()
        self.lib.cae_host_alloc.argtypes = [C.c_size_t]
        self.lib.cae_host_alloc.restype = C.c_void_p
        self.lib.cae_host_free.argtypes = [C.c_void_p]
        self.lib.cae_host_free.restype = None
        cfg = capi.cae_config()
        cfg.abi_version = capi.CONST["CAE_ABI_VERSION"]
        cfg.device, cfg.rank, cfg.world_size, cfg.want_reasons = device, rank, world_size, int(want_reasons)
        self.rank, self.world_size, self.want_reasons = rank, world_size, want_reasons
        self.pods_presharded = pods_presharded
        # the scheduler feature gates as the Go side would report them; default = the values the engine implements
        gates = capi.CONST["CAE_GATE_NODE_INCLUSION_POLICY_IN_PTS"] | capi.CONST["CAE_GATE_MATCH_LABEL_KEYS_IN_PTS"] \
            if feature_gates is None else int(feature_gates)
        cfg.flags = capi.CONST["CAE_CFG_GATES_REPORTED"] | (capi.CONST["CAE_CFG_PODS_PRESHARDED"] if pods_presharded else 0)
        cfg.feature_gates = gates
        h = C.c_void_p()
        self._check(self.lib.cae_create(C.byref(cfg), C.byref(h)))
        self.h = h
        self.enc: Optional[EncodedObjects] = None
        self._pinned = {}

    # ---- plumbing ---------------------------------------------------------------------------
    def _check(self, rc: int) -> None:
        if rc == 0:
            return
        msg = (self.lib.cae_last_error() or b"").decode()
        if rc > 0:
            raise EngineUnsupported(msg)
        raise EngineError("caengine status %d: %s" % (rc, msg))

    def close(self) -> None:
        if getattr(self, "h", None):
            for p in self._pinned.values():
                p.close()
            self._pinned = {}
            self.lib.cae_destroy(self.h)
            self.h = None

    def __del__(self) -> None:
        try:
            self.close()
        except Exception:
            pass

    def _pin(self, name: str, shape, dtype) -> np.ndarray:
        cur = self._pinned.get(name)
        if cur is None or cur.array.shape != tuple(shape) or cur.array.dtype != np.dtype(dtype):
            if cur is not None:
                cur.close()
            cur = PinnedArray(self.lib, tuple(shape), dtype)
            self._pinned[name] = cur
        return cur.array

    # ---- shards -------------------------------------------------------------------------------
    def pod_shard(self, P: int) -> Tuple[int, int]:
        if self.pods_presharded:   # the loaded objects hold this rank's pods only
            return 0, P
        return shard_pods(P, self.rank, self.world_size)

    def template_shard(self, T: int) -> Tuple[int, int]:
        return shard_templates(T, self.rank, self.world_size)

    # ---- API ------------------------------------------------------------------------------------
    def load(self, enc: EncodedObjects) -> None:
        self.enc = enc
        self._check(self.lib.cae_load(self.h, enc.ptr()))

    def load_pending(self, enc: EncodedObjects) -> bool:
        """The per-tick delta (cae_load_pending): only the pending-pod rows of `enc` travel; nodes, templates and pod specs
        must be the ones of the last load().  Returns False when the engine answers "use a full load" (status 2)."""
        a = enc.arrays
        rc = self.lib.cae_load_pending(self.h, enc.P, a["pend_spec"].ctypes.data_as(C.c_void_p), enc.E,
                                       a["group_off"].ctypes.data_as(C.c_void_p))
        if rc == 2:
            return False
        self._check(rc)
        self.enc = enc
        return True

    def feasibility(self, want_bits: bool = True):
        """Dense pods x templates pass. Returns (fit_bits [T][ceil(Pl/32)] uint32 | None,
        reasons [T][Pl] uint8 | None, fit_count [T] int32) for this rank's pod shard."""
        enc = self.enc
        pb, pe = self.pod_shard(enc.P)
        Pl, T = pe - pb, enc.T
        bits = self._pin("bits", (T, (Pl + 31) // 32), np.uint32) if want_bits else None
        reasons = self._pin("reasons", (T, Pl), np.uint8) if self.want_reasons else None
        count = self._pin("count", (T,), np.int32)
        self._check(self.lib.cae_feasibility(
            self.h, bits.ctypes.data_as(C.c_void_p) if bits is not None else None,
            reasons.ctypes.data_as(C.c_void_p) if reasons is not None else None,
            count.ctypes.data_as(C.c_void_p)))
        return bits, reasons, count

    def feasibility_groups(self) -> np.ndarray:
        enc = self.enc
        out = np.zeros((enc.T, enc.E), np.uint8)
        self._check(self.lib.cae_feasibility_groups(self.h, out.ctypes.data_as(C.c_void_p)))
        return out

    def estimate_all_li(self, max_nodes, last_index_in):
        """cae_estimate_all_ex: Estimate of every template with the plugin runner's lastIndex carried in per template.
        Returns node_count, pod_count, sched, order, last_index_out."""
        enc = self.enc
        T, E = enc.T, enc.E
        mn = None if max_nodes is None else np.ascontiguousarray(max_nodes, np.int32)
        li = np.ascontiguousarray(last_index_in, np.int32)
        nc, pc = np.zeros(T, np.int32), np.zeros(T, np.int32)
        sched, order = np.zeros((T, E), np.int32), np.zeros((T, E), np.int32)
        lo = np.zeros(T, np.int32)
        vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        self._check(self.lib.cae_estimate_all_ex(self.h, vp(mn), vp(li), vp(nc), vp(pc), vp(sched), vp(order), vp(lo)))
        return nc, pc, sched, order, lo

    def estimate_all(self, max_nodes: Optional[Sequence[int]] = None, want_sched: bool = True, copy: bool = True):
        """Returns node_count[T], pod_count[T], sched_count[T][E], order[T][E] (rows outside this
        rank's template shard are zero / -1).  Outputs land in pinned buffers; copy=False returns
        views that the next call overwrites; want_sched=False skips the two [T][E] matrices."""
        enc = self.enc
        T, E = enc.T, enc.E
        mn = None if max_nodes is None else np.ascontiguousarray(max_nodes, np.int32)
        node_count = self._pin("node_count", (T,), np.int32)
        pod_count = self._pin("pod_count", (T,), np.int32)
        sched = self._pin("sched", (T, E), np.int32) if want_sched else None
        order = self._pin("order", (T, E), np.int32) if want_sched else None
        vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        self._check(self.lib.cae_estimate_all(self.h, vp(mn), vp(node_count), vp(pod_count), vp(sched), vp(order)))
        if copy:
            return (node_count.copy(), pod_count.copy(), None if sched is None else sched.copy(),
                    None if order is None else order.copy())
        return node_count, pod_count, sched, order

    def expander_best(self, chain: Sequence[int], node_count, pod_count, sched=None):
        """sched=None scores the device-resident result of the last estimate_all (single shard)."""
        enc = self.enc
        ch = np.asarray(chain, np.int32)
        nc = np.ascontiguousarray(node_count, np.int32)
        pc = np.ascontiguousarray(pod_count, np.int32)
        sc = None if sched is None else np.ascontiguousarray(sched, np.int32)
        mask = np.zeros(enc.T, np.uint8)
        waste = np.zeros(enc.T, np.float64)
        vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        self._check(self.lib.cae_expander_best(self.h, vp(ch), len(ch), vp(nc), vp(pc), vp(sc), vp(mask), vp(waste)))
        return mask, waste

    def waste_scores(self) -> np.ndarray:
        """Least-waste score of this rank's template shard from the device-resident result of the last estimate_all
        (0.0 for the rows of other ranks: a sum all-reduce of float64[T] assembles the vector)."""
        waste = np.zeros(self.enc.T, np.float64)
        self._check(self.lib.cae_waste_scores(self.h, waste.ctypes.data_as(C.c_void_p)))
        return waste

    def price_scores(self, node_price, pod_price, stabilization_price: float, preferred_cpu_milli: int = 0, unfitness=None,
                     has_gpu=None, exists=None, node_count=None, sched=None, order=None) -> np.ndarray:
        """Price expander score per option (expander/price/price.go).  node_count/sched/order None = the device-resident
        result of the last estimate_all."""
        T = self.enc.T
        keep = []

        def arr(a, dt):
            if a is None:
                return None
            a = np.ascontiguousarray(a, dt)
            keep.append(a)
            return a
        pin = capi.cae_price_inputs()
        f64p, u8p = C.POINTER(C.c_double), C.POINTER(C.c_uint8)
        pin.node_price = arr(node_price, np.float64).ctypes.data_as(f64p)
        pin.pod_price = arr(pod_price, np.float64).ctypes.data_as(f64p)
        u = arr(unfitness, np.float64)
        pin.unfitness = u.ctypes.data_as(f64p) if u is not None else None
        g = arr(has_gpu, np.uint8)
        pin.has_gpu = g.ctypes.data_as(u8p) if g is not None else None
        x = arr(exists, np.uint8)
        pin.exists = x.ctypes.data_as(u8p) if x is not None else None
        pin.price_error = None
        pin.stabilization_price = float(stabilization_price)
        pin.preferred_cpu_milli = int(preferred_cpu_milli)
        score = np.zeros(T, np.float64)
        vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        self._check(self.lib.cae_price_scores(self.h, C.byref(pin), vp(arr(node_count, np.int32)), vp(arr(sched, np.int32)),
                                              vp(arr(order, np.int32)), vp(score)))
        return score

    def filter_schedulable(self, pod_order: Sequence[int], hint_node=None, sim_class=None, class_ctrl=None, node_ok=None,
                           last_index: int = 0, break_on_failure: bool = False):
        """HintingSimulator.TrySchedulePods on the cluster snapshot of the last load.  Returns (assigned[P] cluster node
        index or -1, lastIndex afterwards, overflowing controller count)."""
        enc = self.enc
        order = np.ascontiguousarray(pod_order, np.int32)
        hn = None if hint_node is None else np.ascontiguousarray(hint_node, np.int32)
        sc = None if sim_class is None else np.ascontiguousarray(sim_class, np.int32)
        cc = None if class_ctrl is None else np.ascontiguousarray(class_ctrl, np.int32)
        ok = None if node_ok is None else np.ascontiguousarray(node_ok, np.uint8)
        assigned = np.full(max(enc.P, 1), -1, np.int32)
        li, ov = np.zeros(1, np.int32), np.zeros(1, np.int32)
        vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        self._check(self.lib.cae_filter_schedulable(self.h, vp(order), len(order), vp(hn), vp(sc), vp(cc),
                                                    0 if cc is None else len(cc), vp(ok), int(last_index), int(break_on_failure),
                                                    vp(assigned), vp(li), vp(ov)))
        return assigned[:enc.P], int(li[0]), int(ov[0])

    def simulate_removals(self, cand_node: Sequence[int], cand_pod_off: Sequence[int], cand_pods: Sequence[int], hint_node=None,
                          node_ok=None, persist: bool = True, max_removable: int = 0, last_index: int = 0,
                          trace_cap: Optional[int] = None):
        """RemovalSimulator.SimulateNodeRemoval for every candidate in turn on the snapshot of the last load
        (cae_simulate_removals).  Returns (result[n_cand], trace_off[n_cand+1], trace_pod, trace_node, lastIndex afterwards).
        The trace buffers start at `trace_cap` entries (default: twice the pods listed) and grow once, to the size no trace
        can exceed, when the engine answers that they are too small."""
        P = self.enc.P
        cn = np.ascontiguousarray(cand_node, np.int32)
        off = np.ascontiguousarray(cand_pod_off, np.int32)
        pods = np.ascontiguousarray(cand_pods, np.int32)
        hn = None if hint_node is None else np.ascontiguousarray(hint_node, np.int32)
        ok = None if node_ok is None else np.ascontiguousarray(node_ok, np.uint8)
        n = len(cn)
        cap = 2 * len(pods) + 64 if trace_cap is None else int(trace_cap)
        result = np.zeros(max(n, 1), np.int32)
        toff = np.zeros(n + 1, np.int32)
        li = np.zeros(1, np.int32)
        vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        for attempt in range(2):
            tpod, tnode = np.zeros(max(cap, 1), np.int32), np.zeros(max(cap, 1), np.int32)
            rc = self.lib.cae_simulate_removals(self.h, n, vp(cn), vp(off), vp(pods), vp(hn), vp(ok), int(bool(persist)),
                                                int(max_removable), int(last_index), vp(result), cap, vp(toff), vp(tpod), vp(tnode),
                                                vp(li))
            if rc == 1 and attempt == 0 and b"trace" in (self.lib.cae_last_error() or b""):
                cap = max(2 * cap, n * P)   # every simulated list holds distinct pending pods
                continue
            self._check(rc)
            break
        k = int(toff[n])
        return result[:n], toff, tpod[:k], tnode[:k], int(li[0])

    # ---- fused histogram exchange over peer memory (multi-GPU dense pass) -------------------------
    def peer_handle(self) -> bytes:
        buf = C.create_string_buffer(capi.CONST["CAE_PEER_HANDLE_BYTES"])
        self._check(self.lib.cae_peer_handle(self.h, buf))
        return buf.raw

    def peer_attach(self, handles: Sequence[bytes]) -> None:
        blob = b"".join(handles)
        assert len(blob) == capi.CONST["CAE_PEER_HANDLE_BYTES"] * self.world_size
        self._check(self.lib.cae_peer_attach(self.h, C.create_string_buffer(blob, len(blob)), self.world_size))

    def stats(self) -> capi.cae_stats:
        s = capi.cae_stats()
        self._check(self.lib.cae_get_stats(self.h, C.byref(s)))
        return s

    def stream(self) -> int:
        """cudaStream_t of the engine (e.g. for torch.cuda.ExternalStream)."""
        return int(self.lib.cae_stream(self.h) or 0)

    def device_buffer(self, which: int) -> Tuple[int, int]:
        n = C.c_size_t(0)
        p = self.lib.cae_device_buffer(self.h, which, C.byref(n))
        return int(p or 0), int(n.value)


def expander_chain(chain: Sequence[int], node_count, pod_count, waste) -> np.ndarray:
    """The expander filter chain on the host (cae_expander_chain): needs the library, not a GPU."""
    lib = capi.load_engine_lib()
    ch = np.asarray(chain, np.int32)
    nc = np.ascontiguousarray(node_count, np.int32)
    pc = np.ascontiguousarray(pod_count, np.int32)
    w = np.ascontiguousarray(waste, np.float64)
    mask = np.zeros(len(nc), np.uint8)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = lib.cae_expander_chain(vp(ch), len(ch), len(nc), vp(nc), vp(pc), vp(w), vp(mask))
    if rc != 0:
        raise EngineError("cae_expander_chain status %d: %s" % (rc, (lib.cae_last_error() or b"").decode()))
    return mask


def expander_chain_ex(chain: Sequence[int], node_count, pod_count, waste=None, price=None, price_error=None, priority=None) -> np.ndarray:
    """cae_expander_chain_ex: the chain with the price (price.go:166-173) and priority (priority.go:119-165) filters."""
    lib = capi.load_engine_lib()
    ch = np.asarray(chain, np.int32)
    nc = np.ascontiguousarray(node_count, np.int32)
    pc = np.ascontiguousarray(pod_count, np.int32)
    opt = lambda a, dt: None if a is None else np.ascontiguousarray(a, dt)
    w, pr, pe, prio = opt(waste, np.float64), opt(price, np.float64), opt(price_error, np.uint8), opt(priority, np.int32)
    mask = np.zeros(len(nc), np.uint8)
    vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    rc = lib.cae_expander_chain_ex(vp(ch), len(ch), len(nc), vp(nc), vp(pc), vp(w), vp(pr), vp(pe), vp(prio), vp(mask))
    if rc != 0:
        raise EngineError("cae_expander_chain_ex status %d: %s" % (rc, (lib.cae_last_error() or b"").decode()))
    return mask


def resolve_priorities(config: dict, group_ids: Sequence[str]) -> np.ndarray:
    """What the Go shim does for the priority expander: highest priority of the ConfigMap (priority -> regexp list) whose
    list matches the node group id (regexp.FindStringIndex = unanchored search), -1 when no entry matches
    (expander/priority/priority.go:137-150, groupIDMatchesList :171-178)."""
    import re
    out = np.full(len(group_ids), -1, np.int32)
    for i, gid in enumerate(group_ids):
        for prio, res in config.items():
            if any(re.search(r, gid) for r in res):
                out[i] = max(out[i], int(prio))
    return out


def unpack_bits(bits: np.ndarray, P: int) -> np.ndarray:
    """fit_bits [T][Pw] uint32 -> bool [T][P]."""
    b = np.unpackbits(bits.view(np.uint8), axis=1, bitorder="little")
    return b[:, :P].astype(bool)
