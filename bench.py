#!/usr/bin/env python
"""bench.py — (replica x node) affinity scores/sec of the placement hot path.

Contract (driver): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON
line on rank 0.  A "step" = one full placement pass of the whole fleet: every
RoleBasedGroup of the batch is scored against all nodes and assigned, all
dependency levels (waves).  Workload at N=1 = BASELINE.json configs[2] (the one
the metric is quoted on): mooncake 5-role / 7-pod RBGs (examples/mooncake/
pd-disaggregated-with-mooncake.yaml) on a 10 000-node 4-tier synthetic topology,
batched `--groups` RBGs per launch (a single RBG is a ~3 MB, ~1 us problem:
launch-bound, SURVEY.md §0.6 — batching is what makes the roofline meaningful).

  parity : BEFORE any timing, on every rank: the CPU oracle's level / wave loop
          re-places a deterministic sample of 64 groups and the dense matrix bits
          of this rank's slab, the assignment, status and exclusive domain are
          compared with the staged plan; a mismatch aborts the run
  value : scores/s with the multi-wave plan already resident in HBM (kernels only,
          one stream, CUDA events around the K steps, max over ranks)
  e2e   : the same metric through the C-ABI plugin call with HOST buffers:
          rbgtopo_update_nodes(free) + rbgtopo_place_groups(groups blob) per
          step — H2D of the inputs and D2H of the results inside the timed region
  value : K steps with nothing recorded inside a step (k_plan_group is a programmatic
          dependent of k_emit_rows); torch events + barrier / synchronize around them
  roofline : k_emit_rows (dominant kernel): algorithmic bytes / CUDA-event
          duration of its launches vs the measured HBM peak (MEASURED_PEAKS.json),
          from a second leg of the same K steps with per-kernel events recorded inside
          the library on the launching stream (rbgtopo_set_kernel_timing); per-launch
          min / median / max beside it, that leg's step time as ms_per_step_kernel_timing
  cpu_baseline : a CPU port of OUR spec (kind "port": sgl-project/rbg has no such
          path and no Go toolchain exists here) on a bounded sample — the variant
          with the GPU path's algebra (oracle/placer_fast.c), the literal oracle
          beside it
  alt   : cfg4 (BASELINE.json configs[3]: 1 000 RBGs x 8 replicas on 50 000 nodes,
          strong scaling under --gpus N) and cfg5 (configs[4]: continuous reconcile
          under 10 % node churn per step + a small-churn line through
          rbgtopo_update_nodes_delta), each with its own parity block

`--impl reference` times the CPU port as the reference arm; its inputs are built by
oracle-side code only (the product library is never loaded in that process).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "replica_x_node_affinity_scores_per_sec"
UNIT = "scores/s"


# ----------------------------------------------------------------- workload
# A fleet is described by plain dicts (no product or oracle types), so that the two arms build
# their own objects from the same description: ours -> rbg_b200.plugin.RoleBasedGroup (marshalled
# by the plugin mirror through the C ABI), reference / checker -> oracle.wave_loop.OGroup.
CONFIGS = {
    # BASELINE.json configs[2]: the one the metric is quoted on (default, weak scaling on the node axis)
    "cfg3": dict(shape="mooncake", groups=1024, nodes=10000, scaling="weak",
                 what="mooncake RBGs (5 roles / 7 pods, 3 dependency waves)"),
    # BASELINE.json configs[3]: fleet of 1 000 RBGs x 8 replicas over 50 000 nodes, node axis sharded (strong scaling)
    "cfg4": dict(shape="fleet8", groups=1000, nodes=50000, scaling="strong",
                 what="fleet8 RBGs (router 1 / prefill 3 / decode 4 = 8 pods, 1 wave)"),
    # BASELINE.json configs[4]: continuous reconcile under churn, 10 % node add/remove per step, 10 000 nodes
    "cfg5": dict(shape="mooncake", groups=1024, nodes=10000, scaling="strong",
                 what="mooncake RBGs re-placed every step while 10 % of the nodes leave / come back"),
}


def fleet_spec(shape_name: str, n_groups: int, n_nodes: int, seed: int = 0):
    """Group g of the fleet already has (g % 4) scheduled pods (partially deployed groups give
    every group its own anchor term)."""
    from rbg_b200 import synth     # pure numpy generators; loads no native code
    shape = {"mooncake": synth.shape_mooncake, "fleet8": synth.shape_fleet8, "pd144": synth.shape_pd_144}[shape_name]()
    out = []
    for g in range(n_groups):
        placed = [(shape.roles[q].name, node) for node, q, _ in
                  synth.random_anchors(n_nodes, len(shape.roles), g % 4, seed, g)]
        out.append(dict(name=f"rbg{g}", gid=g, roles=[(r.name, r.replicas, tuple(r.deps), r.demand) for r in shape.roles],
                        rules=[tuple(x) for x in shape.policy_rules], placed=placed))
    return out


def to_plugin(specs):
    from rbg_b200.plugin import RoleBasedGroup, RoleSpec
    return [RoleBasedGroup("default", s["name"], [RoleSpec(n, r, d, dm) for n, r, d, dm in s["roles"]], gid=s["gid"],
                           policy_rules=s["rules"], placed=s["placed"]) for s in specs]


def to_oracle(specs):
    from oracle.wave_loop import OGroup, ORole
    return [OGroup(s["name"], s["gid"], [ORole(n, r, d, dm) for n, r, d, dm in s["roles"]], rules=s["rules"],
                   placed=s["placed"]) for s in specs]


def build_fleet(n_groups: int, n_nodes: int, seed: int = 0):   # kept for probes / tests
    return to_plugin(fleet_spec("mooncake", n_groups, n_nodes, seed))


def oracle_wave_blobs(topo, specs):
    """The per-wave step batches of a fleet, derived with the CPU oracle alone (untimed)."""
    from oracle import placer as oracle_placer
    from oracle import wave_loop
    _, blobs = wave_loop.run_fleet(topo, to_oracle(specs), nthreads=oracle_placer.max_threads())
    return blobs


def oracle_scores_per_sec(topo, blobs, nthreads, min_seconds=6.0, max_reps=1 << 30, fast=False):
    """Time ONLY the C oracle (score -> top-K -> greedy, dense matrix emitted) on
    the wave batches; steps of a batch are spread over `nthreads` OpenMP threads.
    fast=True: the variant with the GPU path's algebra (base + sparse corrections, oracle/placer_fast.c)."""
    from oracle import placer as oracle_placer
    place = oracle_placer.place_fast if fast else oracle_placer.place
    per_pass = sum(int(b[4]) for b in blobs) * topo.n
    scores, reps, t0 = 0, 0, time.perf_counter()
    while True:
        for b in blobs:
            r = place(topo, b, want_matrix=True, want_topk=False, nthreads=nthreads, reuse_matrix=True)
            assert r["rc"] == 0
        scores += per_pass
        reps += 1
        dt = time.perf_counter() - t0
        if reps >= max_reps or (dt >= min_seconds and max_reps >= (1 << 30)):   # a rep count, when given, is exact
            break
    return scores / dt, dt, reps


def host_thread_candidates():
    """Thread counts worth trying for the CPU oracle: the affinity mask (torchrun pins
    OMP_NUM_THREADS=1, so the mask is what counts), fractions of it (SMT siblings / memory-bound
    phases often peak below the mask) and the cgroup CPU quota when there is one."""
    aff = len(os.sched_getaffinity(0))
    cand = {aff, max(1, aff // 2), max(1, aff // 4)}
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            cand.add(max(1, min(aff, int(int(quota) / int(period)))))
    except Exception:
        pass
    return sorted(cand)


def best_oracle_threads(topo, blobs, seconds=0.4, fast=False):
    """The thread count at which the oracle is fastest on this host (short calibration passes)."""
    best_nt, best_v = 1, 0.0
    for nt in host_thread_candidates():
        v, _, _ = oracle_scores_per_sec(topo, blobs, nt, min_seconds=seconds, fast=fast)
        if v > best_v:
            best_nt, best_v = nt, v
    return best_nt


def product_so_loaded() -> bool:
    try:
        return "librbgtopo" in open("/proc/self/maps").read()
    except Exception:
        return False


# ------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                 f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class _DevPtr:
    """Zero-copy view of a library-owned device buffer for torch (plumbing only)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes // 8,), "typestr": "<i8", "data": (ptr, False),
                                         "version": 3, "strides": None}


# ------------------------------------------------------------------ parity
def parity_check(eng, topo, specs, gblob, handle, fetched, sample, lo, hi, oracle_threads):
    """The checker: the CPU oracle's level/wave loop on a deterministic sample of the fleet vs the
    staged multi-wave plan this rank just ran — dense matrix bits on the rank's column slab
    (every wave, every replica row of the sampled groups), assignment, status, exclusive domain.
    Groups are independent within a batch (snapshot semantics, DESIGN.md §3.7), so the oracle run
    of the sample alone equals the sample's part of the fleet run."""
    from oracle import wave_loop
    from rbg_b200.engine import plan_steps
    steps = plan_steps(gblob, topo.n, len(topo.domain_owner))
    row_of = {(int(st[0]), int(st[1])): int(st[4]) for st in steps}
    rows = bad_rows = 0
    first_bad = None

    def on_wave(w, active, blob, r):
        nonlocal rows, bad_rows, first_bad
        off = 0
        for st in active:
            cnt = sum(c for _, _, c in st.waves[w])
            row0 = row_of[(sample[st.pos], w)]
            for k in range(cnt):
                got = eng.read_scores(handle, row0 + k)
                exp = r["matrix"][off + k, lo:hi]
                rows += 1
                if not np.array_equal(got.view(np.uint32), exp.view(np.uint32)):
                    bad_rows += 1
                    if first_bad is None:
                        j = int(np.nonzero(got.view(np.uint32) != exp.view(np.uint32))[0][0])
                        first_bad = f"group {sample[st.pos]} wave {w} replica {k} node {lo + j}: gpu {got[j]} oracle {exp[j]}"
            off += cnt

    og = to_oracle([specs[i] for i in sample])
    states = [wave_loop.GroupState(g) for g in og]
    for i, st in enumerate(states):
        st.pos = i
    # run_fleet builds its own states: re-use its loop but with ours (same order) to keep `pos`
    blobs, w = [], 0
    from oracle import placer as oracle_placer
    while True:
        active = [st for st in states if not st.failed and w < len(st.waves)]
        if not active:
            break
        blob = wave_loop.build_blob([st.step(w) for st in active])
        r = oracle_placer.place(topo, blob, want_matrix=True, want_topk=False, nthreads=oracle_threads)
        assert r["rc"] == 0, r["rc"]
        on_wave(w, active, blob, r)
        off = 0
        for i, st in enumerate(active):
            cnt = sum(c for _, _, c in st.waves[w])
            st.absorb(w, r["assign"][off:off + cnt], int(r["status"][i]), int(r["domain"][i]))
            off += cnt
        w += 1
    assign, status, domain = fetched
    bad_groups = 0
    for st in states:
        g = sample[st.pos]
        rec = gblob[8 + 12 * g: 8 + 12 * (g + 1)]
        want = st.assign_in_group_order()
        res = st.result()
        got = assign[rec[8]: rec[8] + rec[9]].tolist()
        if got != want or int(status[g]) != res["status"] or int(domain[g]) != res["domain"]:
            bad_groups += 1
            if first_bad is None:
                first_bad = f"group {g}: gpu {got} status {int(status[g])} domain {int(domain[g])}; oracle {want} {res['status']} {res['domain']}"
    return {"ok": bad_rows == 0 and bad_groups == 0, "groups_checked": len(sample), "rows_checked": rows,
            "waves": w, "bad_rows": bad_rows, "bad_groups": bad_groups, "first_bad": first_bad,
            "checked": "dense matrix bits on this rank's column slab (every wave of the sampled groups), assignment, "
                       "status, exclusive domain vs the CPU oracle's wave loop"}


def placement_parity(topo, specs, sample, gblob, result, oracle_threads):
    """assign / status / domain of the sampled groups (host-buffer results) vs the oracle."""
    from oracle import wave_loop
    states, _ = wave_loop.run_fleet(topo, to_oracle([specs[i] for i in sample]), nthreads=oracle_threads)
    assign, status, domain = result
    bad = 0
    for g, st in zip(sample, states):
        rec = gblob[8 + 12 * g: 8 + 12 * (g + 1)]
        res = st.result()
        if (assign[rec[8]: rec[8] + rec[9]].tolist() != st.assign_in_group_order() or int(status[g]) != res["status"]
                or int(domain[g]) != res["domain"]):
            bad += 1
    return bad


# ------------------------------------------------------------------ outputs
DUMP_LIMIT = 64_000_000   # bytes --dump-outputs writes at most, .npy headers included


def _seeded_sample(n, k, seed):
    """Sorted indices of a fixed sample of k of range(n); all of them when k >= n."""
    if k >= n:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False))


def dump_outputs(path, placement, read_row=None, n_rows=0, n_cols=0, col0=0):
    """Writes what a caller of the timed path received from its last step, one DIR/<name>.npy per array, so that two
    builds run with the same arguments (hence the same seeded inputs) can be compared output for output:
    assign / status / domain as float64 (exact for int32) and, when the path keeps one, the dense score matrix as
    float32 (bit for bit).  An infeasible (replica, node) pair scores -inf (DESIGN.md §3.3); every file holds finite
    values, so such entries are written as 0 in scores and as 0 in scores_feasible (1 elsewhere).  The matrix is far
    larger than DUMP_LIMIT at the default sizes, so it is written as a fixed sample: rows, and columns when one row
    alone would not fit, drawn by seeded generators; scores_rows / scores_cols hold the row and node indices of the
    sample.  read_row(r) returns row r over nodes [col0, col0 + n_cols)."""
    os.makedirs(path, exist_ok=True)
    out = {name: np.asarray(a, dtype=np.float64) for name, a in zip(("assign", "status", "domain"), placement)}
    budget = DUMP_LIMIT - 7 * 4096 - sum(a.nbytes for a in out.values())   # seven files, a header of < 4 KB each
    if budget < 0:
        raise SystemExit(f"--dump-outputs: the placement alone is larger than {DUMP_LIMIT} bytes")
    if read_row is not None and n_rows > 0:
        cols = _seeded_sample(n_cols, budget // 32, seed=1)   # 8 B of index + >= 2 rows of 8 B (score, feasible) per column
        rows = _seeded_sample(n_rows, (budget - 8 * len(cols)) // (8 * len(cols) + 8), seed=2)
        scores = np.stack([read_row(int(r))[cols] for r in rows]).astype(np.float32, copy=False)
        feasible = scores != -np.inf
        out["scores"] = np.where(feasible, scores, np.float32(0))
        out["scores_feasible"] = feasible.astype(np.float32)
        out["scores_rows"] = rows.astype(np.float64)
        out["scores_cols"] = (col0 + cols).astype(np.float64)
    assert sum(a.nbytes for a in out.values()) <= DUMP_LIMIT
    for name, a in out.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


# ------------------------------------------------------------------- ours
class Dist:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", 0))
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.local = int(os.environ.get("LOCAL_RANK", 0))
        torch.cuda.set_device(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        assert self.world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={self.world}"
        self.stream = torch.cuda.Stream()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x: float) -> float:
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def min_over_ranks(self, x: float) -> float:
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return float(t.item())


def make_device_step(D, eng, handles, n_waves, mode):
    """One placement pass of the staged fleet.  replicated: run_staged (no collective on the step
    path).  p2p: the in-library all-gather over NVLink peer memory (rbgtopo_run_staged_p2p).
    allgather: per-wave NCCL all-gather driven from here (north_star's literal scheme)."""
    torch, dist = D.torch, D.dist
    if mode in ("replicated", "groups") or D.world == 1:
        def step():
            for h in handles:
                eng.run_staged(h, 1)
        return step
    if mode == "p2p":
        def step():
            for h in handles:
                eng.run_staged_p2p(h, 1)
        return step
    gathered = {}

    def step():
        with torch.cuda.stream(D.stream):
            for h in handles:
                for w in range(n_waves):
                    ptr, nb = eng.shard_wave_score(h, w)
                    if (h, ptr) not in gathered:   # library buffers are stable per staged batch: wrap them once
                        gathered[(h, ptr)] = (torch.as_tensor(_DevPtr(ptr, nb), device="cuda"),
                                              torch.empty(D.world * (nb // 8), dtype=torch.int64, device="cuda"))
                    src, allk = gathered[(h, ptr)]
                    dist.all_gather_into_tensor(allk, src)
                    need2, p2, nb2 = eng.shard_wave_merge(h, w, allk.data_ptr())
                    g2 = None
                    if need2:
                        if (h, p2, 2) not in gathered:
                            gathered[(h, p2, 2)] = (torch.as_tensor(_DevPtr(p2, nb2), device="cuda"),
                                                    torch.empty(D.world * (nb2 // 8), dtype=torch.int64, device="cuda"))
                        src2, g2 = gathered[(h, p2, 2)]
                        dist.all_gather_into_tensor(g2, src2)
                    eng.shard_wave_assign(h, w, g2.data_ptr() if g2 is not None else None)
    return step


def run_config(D, args, cfg_name, with_clocks, dump_dir=None):
    """Stages one configuration, checks it against the oracle, times the resident-plan leg
    (`value`) and the host-buffer leg (`e2e`).  Returns the pieces of the JSON line.
    dump_dir: rank 0 writes there what the last step of the leg `value` times computed (dump_outputs)."""
    torch = D.torch
    from rbg_b200 import synth
    from rbg_b200.engine import TopoPlacer
    from rbg_b200.plugin import B200TopoPodGroupManager
    cfg = CONFIGS[cfg_name]
    rank, world, local = D.rank, D.world, D.local
    groups = args.groups if cfg_name == "cfg3" else cfg["groups"]
    nodes = args.nodes if cfg_name == "cfg3" else cfg["nodes"]
    mode = args.shard_mode if world > 1 else "replicated"
    by_groups = mode == "groups"   # SURVEY.md §8(e) "alternative": the PROBLEM axis is sharded, every rank sees every node
    n_nodes = nodes * world if (cfg["scaling"] == "weak" and not by_groups) else nodes
    topo = synth.make_topology(n_nodes, seed=0, tiers=4, samples_per_tier=5)
    if by_groups:
        # weak: `groups` RBGs per GPU on the same cluster (the fleet grows with N); strong: the fleet is split
        all_specs = fleet_spec(cfg["shape"], groups * world if cfg["scaling"] == "weak" else groups, n_nodes)
        per = (len(all_specs) + world - 1) // world
        specs = all_specs[rank * per:(rank + 1) * per]
        groups = len(specs)
    else:
        specs = fleet_spec(cfg["shape"], groups, n_nodes)
    rbgs = to_plugin(specs)
    churn = cfg_name == "cfg5"

    eng = TopoPlacer(device=local, rank=0, world=1) if by_groups else TopoPlacer(device=local, rank=rank, world=world)
    eng.set_topology(topo.row_ptr, topo.col_idx, topo.edge_w, topo.free, topo.domain, topo.domain_owner)
    gblob, _ = B200TopoPodGroupManager(eng).groups_blob(rbgs)   # host-side marshalling, identical on every rank
    if mode == "p2p":
        eng.p2p_connect(D)
    eng.set_stream(D.stream.cuda_stream)
    # --slots S > 1: S staged copies of the fleet (independent batches: own matrix, plan and outputs) re-placed round
    # robin, one batch per step — the dense-matrix kernel of a step is chained behind the selection kernel of the
    # step before it (rbgtopo_run_staged_chain)
    slots = args.slots if (mode in ("replicated", "groups") or world == 1) and not churn else 1
    handles = [eng.stage_groups(gblob) for _ in range(slots)]
    total_r = int(gblob[4])
    n_waves = eng.shard_waves(handles[0])
    lo, hi = eng.slab()
    scores_rank = total_r * (hi - lo)
    scores_all = total_r * n_nodes
    if by_groups:   # every rank scores its own groups against all nodes: the job's scores are the sum over ranks
        scores_all = int(round(D.sum_over_ranks(float(total_r * n_nodes))))
    device_step = make_device_step(D, eng, handles[:1], n_waves, mode)

    def device_steps(k):   # k steps, enqueue only
        if slots > 1:
            eng.run_staged_chain(handles, k)
        else:
            for _ in range(k):
                device_step()

    # ---- parity first (DESIGN.md §5): a deterministic sample of the fleet, all waves, on every rank
    from oracle import placer as oracle_placer
    nt_par = max(1, min(16, oracle_placer.max_threads(), len(os.sched_getaffinity(0)) // max(1, world)))
    sample = sorted(set(int(i) for i in np.linspace(0, groups - 1, min(groups, args.parity_groups))))
    device_step()
    D.torch.cuda.synchronize()
    fetched = eng.fetch(handles[0])
    par = parity_check(eng, topo, specs, gblob, handles[0], fetched, sample, lo, hi, nt_par)
    par["ok"] = bool(D.min_over_ranks(1.0 if par["ok"] else 0.0) > 0.5)
    par["ranks_checked"] = world
    if not par["ok"] and not args.keep_going:
        raise SystemExit(f"PARITY FAILED ({cfg_name}, rank {rank}): {par}")

    out = {"config_name": cfg_name, "parity": par}
    steps = args.steps
    if not churn:
        # ---- value: resident inputs, CUDA events on the launching stream
        device_steps(max(args.warmup, 3) * slots)
        for h in handles:
            eng.fetch(h)            # sync + reset the timing window
        sampler = ClockSampler(local)
        if rank == 0 and with_clocks:
            sampler.start()
        # clock soak: K steps last a few ms, far below nvidia-smi's sampling period, so the
        # same step is run untimed for ~0.6 s first; the clock samples cover soak + timed region
        t_soak = time.perf_counter()
        soak_s = args.soak if with_clocks else 0.1
        while True:   # every rank runs the SAME number of steps (the sharded modes are SPMD): rank 0's clock decides
            device_steps(50)
            for h in handles:
                eng.fetch(h)
            more = 1.0 if time.perf_counter() - t_soak < soak_s else 0.0
            if world > 1:
                t = torch.tensor([more], dtype=torch.float64, device="cuda")
                D.dist.broadcast(t, src=0)
                more = float(t.item())
            if more < 0.5:
                break
        launches0 = eng.stats()["kernel_launches"]
        D.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(D.stream)
        device_steps(steps)
        ev1.record(D.stream)
        D.barrier()
        dev_ms = ev0.elapsed_time(ev1)
        launches = eng.stats()["kernel_launches"] - launches0
        post = [eng.fetch(h) for h in handles]
        if dump_dir and rank == 0:   # step k of the timed region placed batch handles[k % slots]
            last = (steps - 1) % slots
            dump_outputs(dump_dir, post[last], lambda r: eng.read_scores(handles[last], r), total_r, hi - lo, lo)
        if slots > 1:   # every slot holds the same fleet: the chained passes must leave what the checked pass left
            rows = sorted(set(int(i) for i in np.linspace(0, total_r - 1, 16)))
            ref_rows = [eng.read_scores(handles[0], r).copy() for r in rows]
            for h, res in zip(handles, post):
                ok = all(np.array_equal(x, y) for x, y in zip(res, fetched))
                ok = ok and all(np.array_equal(eng.read_scores(h, r).view(np.uint32), x.view(np.uint32)) for r, x in zip(rows, ref_rows))
                if not ok and not args.keep_going:
                    raise SystemExit(f"PARITY FAILED after the chained passes ({cfg_name}, rank {rank}, slot {h})")
                par["ok"] = bool(par["ok"] and ok)
            par["slots_checked_after_timing"] = slots
        # per-kernel leg: the SAME K steps again with an event between the two kernels of every pass (recorded
        # inside the library on the launching stream, harvested at fetch).  The event serialises the kernels, so
        # this leg is a little slower than the timed region above (where the selection kernel is a programmatic
        # dependent of the dense-matrix kernel); its step time is reported as ms_per_step_kernel_timing.
        eng.set_kernel_timing(True)
        device_steps(slots)
        for h in handles:
            eng.fetch(h)
        D.barrier()
        kv0, kv1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kv0.record(D.stream)
        device_steps(steps)
        kv1.record(D.stream)
        D.barrier()
        kt_ms = D.max_over_ranks(kv0.elapsed_time(kv1))
        clocks = sampler.stop() if (rank == 0 and with_clocks) else None
        score_ms = algo_bytes = 0.0
        per_score = per_sel = np.zeros(0, dtype=np.float32)
        for h in handles:   # a step is ONE pass over ONE batch: per-step kernel time and bytes = the average over the slots
            eng.fetch(h)
            t = eng.last_timing()
            score_ms += t["score_ms"] / len(handles)
            algo_bytes += t["algo_bytes"] / len(handles)
            ps, pl = eng.last_pass_times()
            per_score, per_sel = np.concatenate([per_score, ps]), np.concatenate([per_sel, pl])
        eng.set_kernel_timing(False)
        out["ms_per_step_kernel_timing"] = kt_ms / steps
        dev_ms = D.max_over_ranks(dev_ms)
        out.update(value=scores_rank * world * steps / (dev_ms * 1e-3) if (cfg["scaling"] == "weak" and not by_groups)
                   else scores_all * steps / (dev_ms * 1e-3),
                   ms_per_step=dev_ms / steps, launches=int(launches), clocks=clocks, score_ms=score_ms,
                   algo_bytes=algo_bytes,
                   emit_launch_us={"min": float(per_score.min()) * 1e3, "median": float(np.median(per_score)) * 1e3,
                                   "max": float(per_score.max()) * 1e3, "n": int(len(per_score))} if len(per_score) else None,
                   select_launch_us={"min": float(per_sel.min()) * 1e3, "median": float(np.median(per_sel)) * 1e3,
                                     "n": int(len(per_sel))} if len(per_sel) else None)

    # ---- e2e: host buffers through the C ABI, H2D + D2H inside
    eng.set_stream(None)
    free0 = np.ascontiguousarray(topo.free, dtype=np.int32)
    if churn:
        # 10 % of the nodes leave (capacity 0) or come back per step: 8 snapshots, cycled
        rng = np.random.default_rng(5)
        gone = np.zeros(n_nodes, dtype=bool)
        frees = []
        for _ in range(8):
            flip = rng.choice(n_nodes, size=n_nodes // 10, replace=False)
            gone[flip] = ~gone[flip]
            frees.append(np.where(gone, 0, free0).astype(np.int32))
    else:
        frees = [free0]
    if mode in ("replicated", "groups") or world == 1:
        def e2e_step(k):
            eng.update_nodes(frees[k % len(frees)])
            return eng.place_groups(gblob)
    else:
        def e2e_step(k):
            eng.update_nodes(frees[k % len(frees)])
            h = eng.stage_groups(gblob)
            eng.set_stream(D.stream.cuda_stream)
            make_device_step(D, eng, [h], n_waves, mode)()
            torch.cuda.synchronize()
            r = eng.fetch(h)
            eng.release(h)
            eng.set_stream(None)
            return r
    if churn:   # parity of two churned snapshots (placements only: the host-buffer call keeps no matrix)
        bad = 0
        for k in (0, 3):
            res = e2e_step(k)
            topo_k = synth.Topology(topo.row_ptr, topo.col_idx, topo.edge_w, frees[k], topo.domain, topo.domain_owner)
            bad += placement_parity(topo_k, specs, sample, gblob, res, nt_par)
        out["parity"]["churn_snapshots_checked"] = 2
        out["parity"]["churn_bad_groups"] = bad
        out["parity"]["ok"] = bool(out["parity"]["ok"] and D.min_over_ranks(1.0 if bad == 0 else 0.0) > 0.5)
        if not out["parity"]["ok"] and not args.keep_going:
            raise SystemExit(f"PARITY FAILED under churn ({cfg_name}, rank {rank})")
    if churn and (mode == "replicated" or world == 1):
        # the same fleet under SMALL churn: 16 nodes change capacity per step (pods bound / deleted), pushed with
        # rbgtopo_update_nodes_delta (incremental base + order repair; world > 1: the library refreshes fully)
        rng = np.random.default_rng(6)
        cur = free0.copy()
        deltas = []
        for _ in range(16):
            nd = rng.choice(n_nodes, size=16, replace=False).astype(np.int32)
            vals = rng.integers(0, 9, size=16).astype(np.int32)
            deltas.append((nd, vals))
        eng.update_nodes(cur)

        def small_step(k):
            nd, vals = deltas[k % len(deltas)]
            eng.update_nodes_delta(nd, vals)
            return eng.place_groups(gblob)
        for k in range(4):                                   # parity of the first snapshots of the delta stream
            res_k = small_step(k)
            cur[deltas[k][0]] = deltas[k][1]
            topo_k = synth.Topology(topo.row_ptr, topo.col_idx, topo.edge_w, cur.copy(), topo.domain, topo.domain_owner)
            if placement_parity(topo_k, specs, sample, gblob, res_k, nt_par):
                out["parity"]["ok"] = False
        out["parity"]["ok"] = bool(D.min_over_ranks(1.0 if out["parity"]["ok"] else 0.0) > 0.5)
        if not out["parity"]["ok"] and not args.keep_going:
            raise SystemExit(f"PARITY FAILED under small churn ({cfg_name}, rank {rank})")
        out["parity"]["delta_snapshots_checked"] = 4
        for k in range(4, 24):
            small_step(k)
        rs = []
        for _ in range(5):
            D.barrier()
            t0 = time.perf_counter()
            for k in range(steps):
                small_step(k)
            torch.cuda.synchronize()
            rs.append((time.perf_counter() - t0) * 1e3)
        sm = D.max_over_ranks(sorted(rs)[len(rs) // 2])
        out["small_churn"] = {"value": scores_all * steps / (sm * 1e-3), "unit": UNIT, "ms_per_step": sm / steps,
                              "nodes_changed_per_step": 16,
                              "refresh": "rbgtopo_update_nodes_delta: base updated on the changed nodes' closed neighbourhoods, "
                                         "background order repaired by merge" + ("" if world == 1 else " (world > 1: full refresh)")}
        eng.update_nodes(frees[0])
    for k in range(max(args.warmup, 3) + 16):   # the host side (threads, caches) cooled down during the value leg
        e2e_step(k)
    rounds = []
    res = None
    for _ in range(5):                            # K steps per round; the median round is reported
        D.barrier()
        t0 = time.perf_counter()
        for k in range(steps):
            res = e2e_step(k)
        torch.cuda.synchronize()
        rounds.append((time.perf_counter() - t0) * 1e3)
    e2e_ms = D.max_over_ranks(sorted(rounds)[len(rounds) // 2])
    if churn and dump_dir and rank == 0:   # the host-buffer call is the timed path here; it keeps no matrix
        dump_outputs(dump_dir, res)
    if not churn:
        # the host-buffer entry point (direct path) against the staged plan the oracle checked above: assignment, status, domain
        assert all(np.array_equal(x, y) for x, y in zip(fetched, res)), "e2e placement differs from the staged path"
    n_plan_words = eng.last_timing()["h2d_words"]          # GROUPS blob + per-step geometry words uploaded
    out.update(e2e_value=(scores_rank * world if (cfg["scaling"] == "weak" and not by_groups) else scores_all) * steps / (e2e_ms * 1e-3),
               e2e_ms=e2e_ms / steps, h2d=int(free0.nbytes + 4 * n_plan_words),
               # results read back per step: the assignment + (status, domain) per group on the direct path of
               # rbgtopo_place_groups (world == 1), per step of the expanded plan on the staged path
               d2h=int(4 * (total_r + 2 * groups)) if (mode in ("replicated", "groups") and not os.environ.get("RBGTOPO_NO_DIRECT"))
               else int(4 * (total_r + 2 * n_waves * groups)),
               n_nodes=n_nodes, groups=groups, total_r=total_r, edges=int(topo.e), slab=(lo, hi), mode=mode,
               topo=topo, specs=specs, what=cfg["what"], scaling=cfg["scaling"])
    out["slots"] = slots
    if churn:   # no resident-plan leg: every step re-uploads a changed snapshot, so the step IS the e2e call
        out.update(value=out["e2e_value"], ms_per_step=out["e2e_ms"], launches=0, clocks=None, score_ms=0.0, algo_bytes=0.0)
    for h in handles:
        eng.release(h)
    eng.close()
    return out


def roofline_of(r, peak, peak_src):
    achieved = (r["algo_bytes"] / 1e9) / (r["score_ms"] * 1e-3) if r.get("score_ms") else 0.0
    step_frac = (r["algo_bytes"] / 1e9) / (r["ms_per_step"] * 1e-3) / peak if r.get("ms_per_step") else None
    traffic = None
    traffic_src = None
    try:
        with open(os.path.join(ROOT, "profiles", "score_select_dram_bytes.json")) as f:
            j = json.load(f)
            traffic = j.get("dram_bytes_per_step")
            traffic_src = "static_from_profile: " + str(j.get("source", "ncu --set full capture kept under profiles/"))
    except Exception:
        pass
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_source": traffic_src,
            "kernel": "k_emit_rows (one launch per step and rank emits the dense rows of every wave)",
            "kernel_timing": "CUDA events recorded inside the library around every launch of the kernel, on the launching stream, "
                             "over a second leg of the same K steps (an event between the two kernels of a step serialises them: "
                             "the timed region itself launches the selection kernel as a programmatic dependent)",
            "ms_per_step_kernel_timing": r.get("ms_per_step_kernel_timing"),
            "peak_source": peak_src, "algo_bytes_per_step": r["algo_bytes"], "kernel_ms_per_step": r["score_ms"],
            "kernel_launch_us": r.get("emit_launch_us"), "select_launch_us": r.get("select_launch_us"),
            "frac_of_nominal_8000": achieved / 8000.0,
            "frac_note": "the peak is the measured COPY bandwidth (reads + writes); a write-only stream can exceed it, and at the "
                         "end of a launch part of the stream is still dirty in the 126 MB L2 (see traffic): "
                         "dram_frac_in_kernel = traffic / kernel time / peak is the HBM rate inside the launch itself",
            "dram_frac_in_kernel": (traffic / 1e9) / (r["score_ms"] * 1e-3) / peak if (traffic and r.get("score_ms") and peak
                                                                                     and r.get("config_name") == "cfg3") else None,
            "whole_step_frac": step_frac,
            "whole_step_note": "the same algorithmic bytes over ms_per_step (dense-matrix kernel + selection/greedy kernel)"}


def run_ours(args):
    D = Dist(args)
    rank, world = D.rank, D.world
    main = run_config(D, args, args.config, with_clocks=True, dump_dir=args.dump_outputs)
    alts = {}
    if args.alt:
        for name in ("cfg4", "cfg5"):
            if name != args.config:
                alts[name] = run_config(D, args, name, with_clocks=False)
    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        topo, specs = main["topo"], main["specs"]
        n_nodes, lo, hi = main["n_nodes"], *main["slab"]
        replicated = main["mode"] == "replicated"
        # ---- cpu_baseline (bounded sample, N=1 only)
        cpu = None
        if world == 1 and not args.no_cpu:
            from oracle import placer as oracle_placer
            sample = specs[:min(len(specs), args.cpu_groups)]
            sblobs = oracle_wave_blobs(topo, sample)
            # the honest CPU baseline: the variant with the GPU path's algebra (oracle/placer_fast.c, bit-checked
            # against the literal oracle in tests/test_oracle_fast.py); the literal oracle is reported beside it
            nt = best_oracle_threads(topo, sblobs, fast=True)
            v, dt, reps = oracle_scores_per_sec(topo, sblobs, nt, min_seconds=args.cpu_seconds, fast=True)
            v1, _, _ = oracle_scores_per_sec(topo, sblobs, 1, min_seconds=args.cpu_seconds / 4, fast=True)
            lblobs = oracle_wave_blobs(topo, sample[:max(8, min(len(sample), 128))])   # the literal oracle is ~50x slower: a smaller sample
            ntl = best_oracle_threads(topo, lblobs)
            vl, dtl, _ = oracle_scores_per_sec(topo, lblobs, ntl, min_seconds=args.cpu_seconds / 2)
            cpu = {"value": v, "unit": UNIT, "cores": nt, "kind": "port",
                   "sample": f"{len(sample)} of the {len(specs)} RBGs x {reps} passes, same {n_nodes}-node topology, "
                             f"{dt:.1f} s of wall time on {nt} OpenMP threads (the fastest of "
                             f"{host_thread_candidates()}); 1 thread: {v1:.3e} scores/s",
                   "single_thread_value": v1,
                   "variant": "oracle/placer_fast.c: the GPU path's algebra on the host (base vector + background order per "
                              "snapshot, one multiply per score, sparse patches, partial selection)",
                   "literal": {"value": vl, "cores": ntl,
                               "note": "oracle/placer_oracle.c: the literal spec restatement (a full SpMV per role row, qsort "
                                       "of every feasible key) — the checker, not a fair baseline"},
                   "note": "CPU oracle of OUR frozen spec, not sgl-project/rbg code (the reference has no such path)"}

        def alt_line(r):
            d = {"workload": f"{r['config_name']}: {r['groups']} {r['what']} x {r['n_nodes']}-node topology",
                 "scaling": r["scaling"], "parity": r["parity"],
                 "e2e": {"value": r["e2e_value"], "unit": UNIT, "ms_per_step": r["e2e_ms"],
                         "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"]}}
            if "small_churn" in r:
                d["small_churn"] = r["small_churn"]
                d["refresh"] = "10 % of the nodes change per step: rbgtopo_update_nodes (full k_prep + k_base + sort)"
            if r.get("score_ms"):
                d.update(value=r["value"], unit=UNIT, ms_per_step=r["ms_per_step"], gpu_launches=r["launches"],
                         roofline=roofline_of(r, peak, peak_src))
            return d
        line = {
            "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": main["ms_per_step"], "higher_is_better": True,
            "scaling": main["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "ms_per_step_kernel_timing": main.get("ms_per_step_kernel_timing"),
            "config": {
                "workload": f"{args.config}: {main['groups']} {main['what']} x "
                            f"{n_nodes}-node NVLink/PCIe/RDMA/VPC topology"
                            + ("" if world == 1 else
                               (f"; PROBLEM axis sharded over {world} GPUs: {main['groups']} RBGs per rank, every rank scores "
                                "its groups against all nodes, no collective (SURVEY.md §8(e) alternative)") if main["mode"] == "groups" else
                               f", node axis sharded over {world} GPUs ({(hi - lo)} nodes on rank 0): "
                               + ("dense matrix column-sharded, selection replicated on every rank over all nodes "
                                  "(identical placements, no per-step collective)" if replicated else
                                  ("per-shard top-K lists all-gathered per wave by the library's own kernels over NVLink "
                                   "peer memory (no NCCL call on the step path)" if main["mode"] == "p2p" else
                                   "one NCCL all-gather of per-shard top-K lists per wave"))),
                "parallelism": "single GPU" if world == 1 else
                               (f"problem-axis x{world}" if main["mode"] == "groups" else f"node-axis x{world}, " + main["mode"]),
                "launch": "eager: k_emit_rows, then k_plan_group as its programmatic dependent (griddepcontrol), per step" if (replicated or main["mode"] == "groups") else main["mode"],
                "groups": main["groups"], "nodes": n_nodes, "edges": main["edges"], "replicas_per_step": main["total_r"],
                "emit_matrix": True,
                "l2": "dense-matrix write stream per step "
                      f"({main['total_r'] * (hi - lo) * 4 / 1e6:.0f} MB) exceeds the 126 MB L2; inputs are L2-resident by design",
                "slots": main.get("slots", 1),
                "value_leg": ("" if main.get("slots", 1) == 1 else
                              f"{main.get('slots')} staged copies of the fleet (independent batches: own matrix, plan, outputs) re-placed round "
                              "robin, one batch per step, the dense-matrix kernel of a step chained behind the selection kernel of the step "
                              "before it (rbgtopo_run_staged_chain); results of every slot re-checked after the timed region; ") +
                             "multi-wave plan resident in HBM (rbgtopo_stage_groups), base vector resident "
                             "(recomputed by update_nodes, which is inside the e2e leg)",
                "e2e_leg": "rbgtopo_update_nodes + rbgtopo_place_groups with host buffers (the direct path — GROUPS blob up, "
                           "k_group_rtab, k_emit_rows, k_plan_group<direct>, results down; no expanded plan), median of 5 rounds of "
                           "K steps; marshalling RBG objects into the groups blob is the caller's (Go shim) job "
                           "and is outside",
            },
            "e2e": {"value": main["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": main["h2d"],
                    "d2h_bytes_per_step": main["d2h"], "ms_per_step": main["e2e_ms"]},
            "gpu_launches": main["launches"],
            "clocks": dict(main["clocks"] or {}, window="clock soak (--soak s of identical untimed steps) + timed region"),
            "roofline": roofline_of(main, peak, peak_src),
            "parity": main["parity"],
            "cpu_baseline": cpu,
            "alt": {k: alt_line(v) for k, v in alts.items()},
        }
        print(json.dumps(line))
    if world > 1:
        D.dist.destroy_process_group()


# -------------------------------------------------------------- reference
def run_reference(args):
    """Reference arm: the reference has no implementation of this path and no Go
    toolchain exists here, so (per the task's tier rules) the arm times the CPU
    oracle port on all host threads, on the same config and metric.  Inputs are built by
    oracle-side code only (oracle/wave_loop.py): the product library is never loaded here."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    from oracle import placer as oracle_placer
    from rbg_b200 import synth      # pure numpy generators
    cfg = CONFIGS[args.config]
    groups = args.groups if args.config == "cfg3" else cfg["groups"]
    nodes = args.nodes if args.config == "cfg3" else cfg["nodes"]
    n_nodes = nodes * args.gpus if cfg["scaling"] == "weak" else nodes
    topo = synth.make_topology(n_nodes, seed=0, tiers=4, samples_per_tier=5)
    specs = fleet_spec(cfg["shape"], groups, n_nodes)
    sample = specs[:min(len(specs), args.ref_groups)]
    blobs = oracle_wave_blobs(topo, sample)
    # torchrun pins OMP_NUM_THREADS=1: take the fastest thread count within the affinity mask.  The arm
    # times the CPU variant with the GPU path's algebra (the honest baseline); the literal oracle beside it.
    nt = best_oracle_threads(topo, blobs, fast=True)
    for _ in range(min(args.warmup, 1)):
        oracle_scores_per_sec(topo, blobs, nt, min_seconds=0.0, max_reps=1, fast=True)
    v, dt, reps = oracle_scores_per_sec(topo, blobs, nt, min_seconds=0.0, max_reps=args.steps, fast=True)
    lblobs = oracle_wave_blobs(topo, sample[:max(8, min(len(sample), 128))])   # the literal oracle is ~50x slower: a smaller sample
    ntl = best_oracle_threads(topo, lblobs)
    vl, _, _ = oracle_scores_per_sec(topo, lblobs, ntl, min_seconds=0.0, max_reps=max(1, args.steps // 4))
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3 / args.steps, "higher_is_better": True, "scaling": cfg["scaling"],
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.config}: {cfg['what']} x {n_nodes}-node topology; each step = "
                               f"{len(sample)} of the {groups} RBGs", "groups": groups, "nodes": n_nodes},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": nt, "kind": "port",
                         "sample": f"{len(sample)} RBGs per step x {args.steps} steps on {nt} OpenMP threads "
                                   f"(the fastest of {host_thread_candidates()})",
                         "variant": "oracle/placer_fast.c (same algebra as the GPU path); the dense matrix is emitted",
                         "literal": {"value": vl, "cores": ntl, "note": "oracle/placer_oracle.c, the literal restatement"}},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "product_so_loaded": product_so_loaded(),
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg3", choices=sorted(CONFIGS),
                    help="cfg3 (default, BASELINE.json configs[2]: the metric's config), cfg4 (fleet, 50 000 nodes, "
                         "strong scaling), cfg5 (continuous reconcile under 10 %% churn)")
    ap.add_argument("--no-alt", dest="alt", action="store_false",
                    help="skip the cfg4 / cfg5 measurements reported under `alt`")
    ap.add_argument("--groups", type=int, default=1024, help="cfg3: RBGs per step")
    ap.add_argument("--nodes", type=int, default=10000, help="cfg3: nodes per GPU")
    ap.add_argument("--parity-groups", type=int, default=64, help="groups the oracle re-places before timing")
    ap.add_argument("--keep-going", action="store_true", help="report a parity failure in the line instead of aborting")
    ap.add_argument("--cpu-groups", type=int, default=1024, help="groups per pass of the cpu_baseline leg (the whole fleet)")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--ref-groups", type=int, default=1024, help="groups per step of the reference arm (the whole fleet: same config as ours)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--shard-mode", default="replicated", choices=["replicated", "allgather", "p2p", "groups"],
                    help="N > 1: 'replicated' = dense matrix column-sharded, selection replicated on every rank, "
                         "no per-step collective; 'p2p' = per-shard top-K lists exchanged per wave by the library's "
                         "own kernels over NVLink peer memory; 'allgather' = the same exchange as NCCL all-gathers "
                         "driven from Python")
    ap.add_argument("--slots", type=int, default=1,
                    help="staged copies of the fleet re-placed round robin in the resident leg (independent batches, one per "
                         "step); > 1 chains the dense-matrix kernel of a step behind the selection kernel of the step before it")
    ap.add_argument("--soak", type=float, default=0.6, help="seconds of untimed identical steps before the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32 / float64, "
                         "at most 64 MB: a fixed seeded sample of the score matrix), rank 0 only")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes what the GPU path computed: it does not apply to --impl reference")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
