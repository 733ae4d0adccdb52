#!/usr/bin/env python
"""bench.py — SPF recomputations/sec on the BASELINE.json workloads (default: C2).

A "step" is one pass of the hot path over one batch of synthetic input.  Default workload C2
(the configuration BASELINE.json's metric is quoted on): 1000 SPF roots over the synthetic
OSPFv2 10k-router / 40k-directed-link LSDB (seed 0x484F4C4F+2) on each GPU (weak scaling: every
rank runs its own 1000 roots; at N>1 the per-rank result planes are all-gathered over NVLink,
the path's one exchange step, SURVEY.md §8e).  `--config C1|C3|C4|C5` runs the other
BASELINE.json configs (one JSON line each, same keys).

  value      whole-job SPF/s with the graph, the job list and the result planes resident in
             HBM (device-pointer C-ABI call), CUDA-event timed on the engine's stream.
  e2e        same metric through the host-pointer C-ABI call a holo caller makes: H2D of the job
             list from pinned memory, kernels, D2H of the result planes into pinned host buffers
             (chunks of the batch copy back while the next chunk computes), inside the timed
             region.  OSPF configs ask for what holo-ospf's Vertex keeps (distance, hops, next-hop
             set: holo-ospf/src/spf.rs:38-46) in 16-bit planes = 6 bytes per vertex; `e2e.variants`
             also times all five planes in 16 and in 32/64 bits.
  roofline   algorithmic bytes (12E+20V per SPF, SURVEY.md §8d) / kernel time vs the measured
             HBM peak in MEASURED_PEAKS.json.
  cpu_baseline  the reference-faithful oracle (oracle/, "port") on the host cores, native thread
             pool, bounded sample; with the single-thread figure, the binary-heap Dijkstra on all
             cores, and the measured worth of the visible cores.

`--impl reference` times the CPU oracle instead (all usable host threads), same config.
`--dump-outputs DIR` writes the result planes of the last timed step as .npy files (dump_outputs).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")

import numpy as np  # noqa: E402

METRIC = "SPF recomputations/sec (10k-node LSDB)"
UNIT = "SPF/s"
JOBS_PER_GPU = 1000
DELTA = 0   # bucket width override (0 = library default)


# ----------------------------------------------------------------------------- workloads
class Work:
    """One uploaded graph and the batch of jobs that runs on it."""

    def __init__(self, csr, roots, overrides=None, label=""):
        self.csr = csr
        self.roots = np.ascontiguousarray(roots, dtype=np.uint32)
        self.overrides = overrides          # list (per job) of [(edge, cost), ...] or None
        self.label = label

    @property
    def n(self):
        return len(self.roots)


def alg_bytes(csr) -> int:
    return 12 * csr.n_edges + 20 * csr.n_vertices


def adjacency_edges(csr, t, vertex_of):
    """adjacency k of topology t -> its two directed CSR edges (parallel adjacencies in order)."""
    row, col = csr.row_ptr, csr.col
    first = {}
    for u in range(csr.n_vertices):
        for e in range(row[u], row[u + 1]):
            first.setdefault((u, int(col[e])), []).append(e)
    seen, pair = {}, []
    for k in range(t.n_p2p):
        a, b = vertex_of(t.p2p_a[k]), vertex_of(t.p2p_b[k])
        key = (min(a, b), max(a, b))
        nth = seen.get(key, 0)
        seen[key] = nth + 1
        pair.append((first[(a, b)][nth], first[(b, a)][nth]))
    return pair


def build_workload(name: str, rank: int, world: int, jobs: int):
    """Returns (description dict, [Work, ...], scaling)."""
    from holo_b200 import synth, shard
    if name == "C2":
        t = synth.random_topology(10000, 40000, synth.SEED_BASE + 2)
        csr = synth.topology_csr(t, delta=DELTA)
        lo, hi = shard.job_range(jobs * world, rank, world)          # weak scaling: `jobs` per rank
        roots = (np.arange(lo, hi) % 10000 + len(t.lans)).astype(np.uint32)
        desc = {"workload": "C2: OSPFv2 single-area synthetic LSDB, 10000 routers / 40000 directed p2p links, "
                            f"cost U[1,100], {jobs} SPF roots per GPU per step",
                "seed": hex(synth.SEED_BASE + 2), "protocol": "ospfv2"}
        return desc, [Work(csr, roots, label="C2")], "weak"
    if name == "C1":
        t = synth.random_topology(100, 400, synth.SEED_BASE + 1)
        csr = synth.topology_csr(t, delta=DELTA)
        desc = {"workload": "C1: OSPFv2 single-area synthetic LSDB, 100 routers / 400 directed p2p links, 1 SPF root "
                            "(the reference's own CPU-runnable case: one launch per root, latency bound)",
                "seed": hex(synth.SEED_BASE + 1), "protocol": "ospfv2"}
        return desc, [Work(csr, np.asarray([0], np.uint32), label="C1")], "weak"
    if name == "C3":
        from holo_b200 import isis
        from holo_b200.capi import COST_DISABLED
        t = synth.random_topology(10000, 40000, synth.SEED_BASE + 3, cost_lo=1, cost_hi=1000)
        f = isis.Flat(isis.synth_level(t))
        csr = f.csr
        csr.delta = DELTA
        root = f.vertex(isis.sysid(0) << 8)
        pair = adjacency_edges(csr, t, lambda i: f.vertex(isis.sysid(int(i)) << 8))
        n = jobs * 10                                               # 10 000 perturbation jobs per GPU
        lo = rank * n
        ov = [[(pair[(lo + j) % len(pair)][0], COST_DISABLED), (pair[(lo + j) % len(pair)][1], COST_DISABLED)]
              for j in range(n)]
        desc = {"workload": "C3: IS-IS L2 synthetic LSDB, 10000 systems / 40000 directed adjacencies, wide metrics "
                            f"U[1,1000], {n} what-if SPFs per GPU per step (same root, job j removes adjacency j mod 20000)",
                "seed": hex(synth.SEED_BASE + 3), "protocol": "isis"}
        return desc, [Work(csr, np.full(n, root, np.uint32), ov, label="C3")], "weak"
    if name == "C4":
        from holo_b200 import ospfv3
        n_areas, per = 25, 2000
        mine = [k for k in range(n_areas) if k % world == rank]     # areas have equal size: round robin is balanced
        works = []
        for k in mine:
            t = synth.random_topology(per, 8000, synth.SEED_BASE + 4 + 100 * k, cost_lo=1, cost_hi=100,
                                      lan_fraction=0.05 if k % 8 == 0 else 0.0)
            rids = ospfv3.RID_BASE + k * per + np.arange(per)
            area = ospfv3.synth_area(t, root=0, max_links_per_fragment=6, rids=rids, area_id=k)
            f = ospfv3.Flat(area)
            f.csr.delta = DELTA
            works.append(Work(f.csr, np.nonzero(f.is_router)[0].astype(np.uint32), label=f"C4 area {k}"))
        desc = {"workload": "C4: OSPFv3 multi-area synthetic LSDB, 25 areas x 2000 routers / 8000 directed links (50000 "
                            "routers, 200000 links), every router of every area is an SPF root over its area (50000 SPFs "
                            f"per step), areas sharded over {world} GPU(s)",
                "seed": hex(synth.SEED_BASE + 4), "protocol": "ospfv3"}
        return desc, works, "strong"
    if name == "C5":
        from holo_b200 import ospfv2
        t = synth.random_topology(10000, 40000, synth.SEED_BASE + 5, cost_choices=[10, 20], lan_fraction=0.05)
        area = ospfv2.synth_area(t, root=0, sr=True)
        f = ospfv2.Flat(area)
        f.csr.delta = DELTA
        routers = np.nonzero(f.is_router)[0].astype(np.uint32)
        lo, hi = shard.job_range(jobs * world, rank, world)
        roots = routers[np.arange(lo, hi) % len(routers)]
        desc = {"workload": "C5: OSPFv2 ECMP + SR synthetic LSDB, 10000 routers, costs {10,20}, 5% of the adjacencies on "
                            f"broadcast LANs, prefix-SIDs; {jobs} SPF roots per GPU per step on the device (SPT + next-hop "
                            "sets); the route / label stage is timed separately in `route_stage`",
                "seed": hex(synth.SEED_BASE + 5), "protocol": "ospfv2", "_area": area}
        return desc, [Work(f.csr, roots, label="C5")], "weak"
    raise SystemExit(f"unknown config {name}")


EXCHANGE_TEXT = {
    "none": "none",
    "nccl": "one NCCL all-gather of the step's result planes per step, overlapped with the next step's kernel",
    "fused": "fused into the batch kernel: every finished job's rows of the travelling planes are pushed by its CTA straight "
             "into this rank's slot on every peer GPU over NVLink (16-byte stores) while the batch computes "
             "(hspf_ctx_set_peer_slots); only "
             "4-byte sequence flags follow behind the kernel (stream memory-op waits, no collective kernel); checked "
             "once against an NCCL all-gather before the timed region",
    "p2p": "all-gather of the step's result planes per step by the copy engines over NVLink peer memory "
           "(hspf_xchg_*: one copy stream per peer, sequence flags behind the data, stream memory-op waits, no SM), "
           "overlapped with the next step's kernel; checked once against an NCCL all-gather before the timed region",
}


def config_dict(world, desc, works, exchange, planes):
    c = {k: v for k, v in desc.items() if not k.startswith("_")}
    c.update({
        "V": int(works[0].csr.n_vertices), "E": int(works[0].csr.n_edges),
        "jobs_per_gpu": int(sum(w.n for w in works)), "graphs_per_gpu": len(works),
        "parallelism": f"jobs sharded over {world} GPU(s), graph(s) replicated",
        "result_planes": ("dist hops first_parent n_parents nh_mask, all u16 (hspf_result16): 10 B per vertex"
                          if planes == "16-bit" else
                          "dist:u32 hops:u16 first_parent:u32 n_parents:u16 nh_mask:u64 (hspf_result): 20 B per vertex"),
        "l2": ("flushed between timed steps (256 MiB memset, untimed)" if exchange == "none" else
               "no explicit flush: each step writes its result planes and receives the other ranks' (> 126 MB L2 in "
               "total); the graph is cache-resident by design"),
        "exchange": EXCHANGE_TEXT.get(exchange, exchange),
    })
    return c


DUMP_PLANES = (("dist", "dist"), ("hops", "hops"), ("first_parent", "fp"), ("n_parents", "npar"), ("nh_mask", "nh"))
DUMP_BYTES = 64_000_000         # all files of one --dump-outputs run, .npy headers included
NPY_HEADER_BYTES = 4096         # per graph: 8 files of 128-byte headers, with room to spare


def dump_outputs(out_dir, works, lay, buf, bpv, prefix="", budget=DUMP_BYTES):
    """Write the result planes one timed step left in `buf` (what the device-pointer call hands its
    caller) as DIR/<prefix><plane>.npy, prefixed g<i>_ as well when the step runs several graphs.
    16-bit planes become float32 and 32-bit ones float64; a 64-bit plane becomes two float64 planes,
    <plane> with its low and <plane>_hi with its high 32 bits, so every value is exact.  The files
    take at most `budget` bytes: when all jobs would not fit, the rows are a fixed, seeded sample of
    the jobs; job_index.npy names them."""
    import torch
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    per_graph = budget // len(works) - NPY_HEADER_BYTES
    for i, (w, o) in enumerate(zip(works, lay)):
        V, n = w.csr.n_vertices, w.n
        row_bytes = V * sum({2: 4, 4: 8, 8: 16}[bpv[k]] for _, k in DUMP_PLANES) + 16   # + job_status, job_index
        k = min(n, per_graph // row_bytes)
        rows = np.arange(n) if k == n else np.sort(np.random.default_rng(i).choice(n, k, replace=False))
        sel = torch.from_numpy(rows).to(buf.device)
        pre = prefix + (f"g{i}_" if len(works) > 1 else "")
        for name, key in DUMP_PLANES:
            b = bpv[key]
            a = buf[o[key]: o[key] + n * V * b].view(n, V * b).index_select(0, sel).cpu().numpy()
            a = a.view({2: np.uint16, 4: np.uint32, 8: np.uint64}[b])
            if b == 8:
                np.save(out / f"{pre}{name}_hi.npy", (a >> np.uint64(32)).astype(np.float64))
                a = a & np.uint64(0xFFFFFFFF)
            np.save(out / f"{pre}{name}.npy", a.astype(np.float32 if b == 2 else np.float64))
        status = buf[o["status"]: o["status"] + 4 * n].cpu().numpy().view(np.uint32)[rows]
        np.save(out / f"{pre}job_status.npy", status.astype(np.float64))
        np.save(out / f"{pre}job_index.npy", rows.astype(np.float64))


def exchange_note(xchg_bytes, tot):
    return (f"{xchg_bytes} of the {tot} plane bytes of a rank travel per step" +
            (" (distance, hops, next-hop set, job status: what holo-ospf's Vertex keeps, holo-ospf/src/spf.rs:38-46)"
             if xchg_bytes < tot else " (all planes)"))


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self._th = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()

    def stop(self):
        self._stop.set()
        if self._th:
            self._th.join(timeout=6)
        sm = sorted(int(float(s[0])) for s in self.samples if s[0].replace(".", "").isdigit())
        mx = [int(float(s[1])) for s in self.samples if s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------- CPU arms
def cpu_arms(works, seconds: float = 8.0):
    """The CPU figures of SURVEY.md §8d on the first graph of the workload, native thread pool
    (oracle/batch_pool.cc), bounded samples.  Returns the cpu_baseline object."""
    from oracle import pyoracle
    w = works[0]
    vec = 1 if (w.csr.flags & 1) else 0
    visible = pyoracle.usable_cores()
    eff = pyoracle.effective_cores(visible)

    def run(mode, thr, secs):
        done, t, reps = 0, 0.0, 0
        while t < 0.6 * secs and reps < 64:       # a fast arm runs out of jobs before the bound: repeat the batch
            r = pyoracle.csr_batch(w.csr, w.roots, overrides=w.overrides, mode=mode, vec_mode=vec, threads=thr,
                                   stop_after_s=secs - t, want_planes=False)
            done += r["jobs_done"]; t += r["seconds"]; reps += 1
        return (done / t if t > 0 else 0.0), done, t

    f_rate, f_done, f_t = run("faithful", visible, seconds)
    s_rate, s_done, s_t = run("faithful", 1, max(3.0, seconds / 2))
    h_rate, h_done, h_t = run("heap", visible, max(5.0, seconds * 0.7))
    h1_rate, h1_done, h1_t = run("heap", 1, 3.0)
    return {
        "value": f_rate, "unit": UNIT, "cores": visible, "kind": "port",
        "sample": f"{f_done} jobs of this step's batch in {f_t:.1f} s, reference-faithful oracle (linear candidate scan + "
                  f"per-edge mutual check, oracle/spf_csr.cc) on a native pool of {visible} threads (oracle/batch_pool.cc)",
        "cores_visible": visible, "cores_effective": round(eff, 2),
        "note": "cores_effective = measured throughput of the visible cores in units of one core (spin workload on 1 "
                "thread and on all); the scaling efficiencies are relative to it",
        "single_thread": {"value": s_rate, "unit": UNIT, "cores": 1, "sample": f"{s_done} jobs, {s_t:.1f} s"},
        "faithful_scaling_efficiency": (f_rate / (s_rate * eff)) if s_rate > 0 else None,
        "optimised": {"value": h_rate, "unit": UNIT, "cores": visible,
                      "kind": "binary-heap Dijkstra, same CSR and parent / next-hop rules (oracle/spf_csr.cc "
                              "oracle_csr_spf_heap)",
                      "sample": f"{h_done} jobs, {h_t:.1f} s",
                      "single_thread": {"value": h1_rate, "sample": f"{h1_done} jobs, {h1_t:.1f} s"},
                      "scaling_efficiency": (h_rate / (h1_rate * eff)) if h1_rate > 0 else None},
    }


def run_reference(args):
    """--impl reference: the reference's CPU path (restated in oracle/, the Rust reference cannot
    be built in this image) on all usable host cores, native thread pool."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from holo_b200.build import build_oracle
    from oracle import pyoracle
    build_oracle()
    desc, works, scaling = build_workload(args.config, 0, 1, args.jobs)
    w = works[0]
    vec = 1 if (w.csr.flags & 1) else 0
    cores = pyoracle.usable_cores()
    eff = pyoracle.effective_cores(cores)
    step_s = 3.0                       # each step: a bounded sample of the step's batch
    k = max(1, min(w.n, cores))
    pyoracle.csr_batch(w.csr, w.roots[:k], overrides=w.overrides[:k] if w.overrides else None,
                       mode="faithful", vec_mode=vec, threads=cores, stop_after_s=1.0, want_planes=False)   # warm-up
    done, t_total = 0, 0.0
    for s in range(args.steps):
        off = (s * cores * 4) % max(w.n, 1)
        roots = np.roll(w.roots, -off)
        ov = (w.overrides[off:] + w.overrides[:off]) if w.overrides else None
        r = pyoracle.csr_batch(w.csr, roots, overrides=ov, mode="faithful", vec_mode=vec, threads=cores,
                               stop_after_s=step_s, want_planes=False)
        done += r["jobs_done"]
        t_total += r["seconds"]
    value = done / t_total
    sample = f"{done} jobs in {t_total:.1f} s: each step a {step_s:.0f} s sample of the step's batch"
    exchange = "none" if (args.gpus == 1 or args.config != "C2") else (
        args.exchange if args.exchange != "auto" else ("fused" if args.gpus > 4 else "p2p"))
    cfg = config_dict(args.gpus, desc, works, exchange, "16-bit" if args.planes == "16" else "32-bit")
    cfg["reference_sample"] = sample
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
        "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "cores_visible": cores, "cores_effective": round(eff, 2)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import ctypes as C
    import torch
    import torch.distributed as dist
    from holo_b200.build import build_all
    from holo_b200 import capi, shard

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    if rank == 0:
        build_all()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()

    desc, works, scaling = build_workload(args.config, rank, world, args.jobs)
    ctx = capi.Context(local_rank)
    graphs = [ctx.upload(w.csr) for w in works]
    fast = all(ctx.graph_info(g)["fast_path"] for g in graphs)
    # 16-bit next-hop planes hold 16 first-hop atoms: a batch with a root that has more (a router on
    # several LANs) runs with the 32/64-bit planes
    max_atoms = max(max(capi.atom_count(w.csr, int(r)) for r in np.unique(w.roots)) for w in works)
    narrow = fast and args.planes == "16" and max_atoms <= 16
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    al = lambda x: (x + 255) // 256 * 256
    bpv = ({"dist": 2, "hops": 2, "fp": 2, "npar": 2, "nh": 2} if narrow else
           {"dist": 4, "hops": 2, "fp": 4, "npar": 2, "nh": 8})

    # ---- device-resident planes (value path): ONE byte buffer per rank and step so that the
    # multi-GPU exchange is a single all-gather; two buffers when there is an exchange (the
    # exchange of step s overlaps the kernels of step s+1)
    # layout: the planes the caller's Vertex keeps (dist, hops, nh) and the status first, so that
    # the exchange can push just that prefix of the slot
    lay, tot, prefix = [], 0, 0
    for w in works:
        V, n = w.csr.n_vertices, w.n
        o = {}
        for k in ("dist", "hops", "nh"):
            o[k] = tot
            tot += al(n * V * bpv[k])
        o["status"] = tot
        tot += al(n * 4)
        prefix = tot
        for k in ("fp", "npar"):
            o[k] = tot
            tot += al(n * V * bpv[k])
        lay.append(o)
    is_ospf = desc.get("protocol", "").startswith("ospf")
    xchg_bytes = prefix if (len(works) == 1 and is_ospf and args.xchg_planes == "vertex") else tot
    exchange = "none"
    if world > 1 and args.config == "C2":
        exchange = args.exchange
        if exchange == "auto":
            # Measured (profiles/r2_n*_*.json): the copy engines hide the exchange behind the kernel at N=2
            # (efficiency 0.97) and deliver ~265-285 GB/s per GPU beyond that (N=4: 0.73); with 7 peers the
            # fused variant (the kernel pushes every finished job's rows into the peers' slots itself) is used.
            exchange = "fused" if (world > 4 and narrow and xchg_bytes == prefix) else "p2p"
        if exchange == "fused" and not (narrow and xchg_bytes == prefix):
            raise SystemExit("--exchange fused needs 16-bit planes and --xchg-planes vertex")
    n_buf = 2 if exchange != "none" else 1
    xchg = None
    if exchange in ("p2p", "fused"):
        try:
            xchg = shard.PeerExchange(ctx, local_rank, rank, world, tot, n_buf)
        except RuntimeError as e:       # raised on every rank together
            if rank == 0:
                print(f"bench: peer exchange unavailable ({e}); using NCCL all-gather", file=sys.stderr)
            exchange = "nccl"
    if xchg is not None:
        xchg.set_push_bytes(xchg_bytes)
        bufs = [shard.raw_cuda_tensor(xchg.slot_ptr(b, rank), tot, dev) for b in range(n_buf)]
        gathered_p2p = [xchg.buffer_tensor(b, dev) for b in range(n_buf)]
        gathered = None
    else:
        bufs = [torch.empty(tot, dtype=torch.uint8, device=dev) for _ in range(n_buf)]
        gathered = torch.empty((world, xchg_bytes), dtype=torch.uint8, device=dev) if exchange == "nccl" else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    # device-resident job lists
    keep, jss = [], []
    for w in works:
        js = capi.JobsStruct()
        js.n_jobs = w.n
        d_roots = torch.from_numpy(w.roots.astype(np.int64)).to(torch.int32).to(dev)
        js.roots = C.cast(d_roots.data_ptr(), C.POINTER(C.c_uint32))
        keep.append(d_roots)
        if w.overrides is not None:
            off = np.zeros(w.n + 1, np.int64)
            ed, co = [], []
            for j, ov in enumerate(w.overrides):
                for e, c in ov:
                    ed.append(e); co.append(c)
                off[j + 1] = len(ed)
            d_off = torch.from_numpy(off).to(torch.int32).to(dev)
            d_ed = torch.from_numpy(np.asarray(ed or [0], np.uint32).view(np.int32).copy()).to(dev)
            d_co = torch.from_numpy(np.asarray(co or [0], np.uint32).view(np.int32).copy()).to(dev)
            js.ov_off = C.cast(d_off.data_ptr(), C.POINTER(C.c_uint32))
            js.ov_edge = C.cast(d_ed.data_ptr(), C.POINTER(C.c_uint32))
            js.ov_cost = C.cast(d_co.data_ptr(), C.POINTER(C.c_uint32))
            keep += [d_off, d_ed, d_co]
        jss.append(js)
    torch.cuda.synchronize()

    def result_struct(buf, o):
        base = buf.data_ptr()
        if narrow:
            r = capi.Result16Struct()
            for k, f in (("dist", "dist"), ("hops", "hops"), ("fp", "first_parent"), ("npar", "n_parents"), ("nh", "nh_mask")):
                setattr(r, f, C.cast(base + o[k], C.POINTER(C.c_uint16)))
        else:
            r = capi.ResultStruct()
            r.dist = C.cast(base + o["dist"], C.POINTER(C.c_uint32))
            r.hops = C.cast(base + o["hops"], C.POINTER(C.c_uint16))
            r.first_parent = C.cast(base + o["fp"], C.POINTER(C.c_uint32))
            r.n_parents = C.cast(base + o["npar"], C.POINTER(C.c_uint16))
            r.nh_mask = C.cast(base + o["nh"], C.POINTER(C.c_uint64))
            r.nh_words = 1
        r.job_status = C.cast(base + o["status"], C.POINTER(C.c_uint32))
        return r

    rss = [[result_struct(b, o) for o in lay] for b in bufs]
    comm_stream = torch.cuda.Stream(device=dev, priority=-1) if exchange == "nccl" else None
    cons_stream = torch.cuda.ExternalStream(xchg.consumer_stream, device=dev) if xchg is not None else None

    def launch_all(b):
        for g, js, rs in zip(graphs, jss, rss[b]):
            if narrow:
                ctx.run_device16(g, js, rs, sync=False)
            else:
                ctx.run_device(g, js, rs, sync=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    mode = {"x": exchange}

    def run_steps(n_steps):
        """No exchange: [flush, kernels] per step, per-step events.  With an exchange: kernels on
        the engine stream, the all-gather beside them, double buffered."""
        evs, ag_done = [], [None] * n_buf
        for s in range(n_steps):
            b = s % n_buf
            if exchange == "none":
                with torch.cuda.stream(stream):
                    flush.fill_(1)
            elif xchg is not None and mode["x"] == "fused":
                xchg.acquire_direct(b)                 # ... and every peer has released its copy of the slot
                ctx.set_peer_slots(xchg.peer_deltas(b))
            elif xchg is not None:
                xchg.acquire(b)                        # own slot of buffer b has left the device
            elif ag_done[b] is not None:
                stream.wait_event(ag_done[b])          # buffer b is free again
            e0 = torch.cuda.Event(enable_timing=True)
            ek = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            launch_all(b)
            ek.record(stream)
            if xchg is not None:
                if mode["x"] == "fused":
                    ctx.set_peer_slots([])
                    xchg.publish(b)  # the planes are already there: flags only
                else:
                    xchg.push(b)    # copy engines: slot -> every peer, flags behind the data
                xchg.wait(b)        # consumer stream: all slots of buffer b have arrived
                xchg.release(b)     # (no consumer work in the bench) peers may reuse buffer b
            elif exchange == "nccl":
                comm_stream.wait_event(ek)
                with torch.cuda.stream(comm_stream):
                    dist.all_gather_into_tensor(gathered.view(-1), bufs[b][:xchg_bytes])
                    ag_done[b] = torch.cuda.Event()
                    ag_done[b].record(comm_stream)
            evs.append((e0, ek))
        if xchg is not None:
            done = torch.cuda.Event()
            done.record(cons_stream)
            stream.wait_event(done)                    # the timed region ends when every slot is in
        elif exchange == "nccl":
            for e in ag_done:
                if e is not None:
                    stream.wait_event(e)
        return evs

    run_steps(args.warmup)
    barrier()
    if xchg is not None:
        # one-time check of the peer exchange against an NCCL all-gather of the same planes
        xchg.sync()
        b_last = (args.warmup - 1) % n_buf
        ref = torch.empty((world, xchg_bytes), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(ref.view(-1), bufs[b_last][:xchg_bytes])
        same = torch.tensor([1 if torch.equal(ref, gathered_p2p[b_last][:, :xchg_bytes]) else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        del ref
        barrier()
        if int(same.item()) != 1:
            if mode["x"] == "fused":
                # never expected; keep the run valid by measuring the copy-engine exchange instead
                if rank == 0:
                    print("bench: fused exchange delivered planes that differ from the NCCL all-gather; "
                          "falling back to --exchange p2p", file=sys.stderr)
                mode["x"] = exchange = "p2p"
                xchg.sync()
                barrier()
                run_steps(args.warmup)
                barrier()
            else:
                raise SystemExit("bench: peer exchange delivered planes that differ from the NCCL all-gather")
    st_all = torch.cat([bufs[0][o["status"]: o["status"] + 4 * w.n].view(torch.int32) for o, w in zip(lay, works)])
    assert int(st_all.abs().sum().item()) == 0, "job_status != 0"

    launches0 = ctx.launch_count
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    wall0 = time.perf_counter()
    t_begin = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    t_begin.record(stream)
    ev = run_steps(args.steps)
    t_end.record(stream)
    barrier()
    wall = time.perf_counter() - wall0
    launches = ctx.launch_count - launches0
    kern_ms = [e0.elapsed_time(ek) for e0, ek in ev]
    kernel_ms_avg = float(sum(kern_ms) / len(kern_ms))
    # no exchange: the L2 flush between steps is untimed (sum of per-step kernel events); with an
    # exchange: the whole pipelined region (kernels + exchanges), no flush needed (see config.l2)
    total_ms = float(sum(kern_ms)) if exchange == "none" else float(t_begin.elapsed_time(t_end))
    if args.dump_outputs:     # every rank its own jobs' planes; together they are the whole step's output
        dump_outputs(args.dump_outputs, works, lay, bufs[(args.steps - 1) % n_buf], bpv,
                     prefix=f"r{rank}_" if world > 1 else "", budget=DUMP_BYTES // world)

    # ---- e2e: host-pointer C-ABI call, pinned host buffers ----------------------------------

    def e2e_variant(which):
        """which: 'caller16' (what the protocol's caller keeps, 16-bit), 'all16', 'all32'.  Returns
        (SPF/s, h2d bytes, d2h bytes, steps) or None if not applicable."""
        use16 = which != "all32"
        if use16 and not (fast and max_atoms <= 16):
            return None
        planes = ("dist", "hops", "nh") if (which == "caller16" and is_ospf) else ("dist", "hops", "fp", "npar", "nh")
        hbufs, calls, d2h, h2d = [], [], 0, 0
        for w, g in zip(works, graphs):
            V, n = w.csr.n_vertices, w.n
            hj, kp = capi.make_jobs(w.roots, w.overrides)
            h_roots = torch.from_numpy(w.roots.astype(np.int64)).to(torch.int32).pin_memory()
            hj.roots = C.cast(h_roots.data_ptr(), C.POINTER(C.c_uint32))
            h2d += n * 4 + ((8 * sum(len(o) for o in w.overrides) + 4 * (n + 1)) if w.overrides else 0)
            hb = {"status": torch.zeros((n,), dtype=torch.int32).pin_memory()}
            if use16:
                hr = capi.Result16Struct()
                for k, f in (("dist", "dist"), ("hops", "hops"), ("fp", "first_parent"), ("npar", "n_parents"), ("nh", "nh_mask")):
                    if k in planes:
                        hb[k] = torch.empty((n, V), dtype=torch.int16).pin_memory()
                        setattr(hr, f, C.cast(hb[k].data_ptr(), C.POINTER(C.c_uint16)))
                        d2h += n * V * 2
                fn = ctx.lib.hspf_run_batch16
            else:
                hr = capi.ResultStruct()
                hb["dist"] = torch.empty((n, V), dtype=torch.int32).pin_memory()
                hb["hops"] = torch.empty((n, V), dtype=torch.int16).pin_memory()
                hb["fp"] = torch.empty((n, V), dtype=torch.int32).pin_memory()
                hb["npar"] = torch.empty((n, V), dtype=torch.int16).pin_memory()
                hb["nh"] = torch.empty((n, V), dtype=torch.int64).pin_memory()
                hr.dist = C.cast(hb["dist"].data_ptr(), C.POINTER(C.c_uint32))
                hr.hops = C.cast(hb["hops"].data_ptr(), C.POINTER(C.c_uint16))
                hr.first_parent = C.cast(hb["fp"].data_ptr(), C.POINTER(C.c_uint32))
                hr.n_parents = C.cast(hb["npar"].data_ptr(), C.POINTER(C.c_uint16))
                hr.nh_mask = C.cast(hb["nh"].data_ptr(), C.POINTER(C.c_uint64))
                hr.nh_words = 1
                d2h += n * V * 20
                fn = ctx.lib.hspf_run_batch
            hr.job_status = C.cast(hb["status"].data_ptr(), C.POINTER(C.c_uint32))
            d2h += n * 4
            hbufs.append((hb, h_roots, kp))
            calls.append((fn, g, hj, hr))

        def step():
            for fn, g, hj, hr in calls:
                rc = fn(ctx.handle, g.handle, C.byref(hj), C.byref(hr), 0)
                if rc != 0:
                    raise RuntimeError(f"host-pointer call rc={rc}: {ctx.last_error()}")

        n_e2e = args.steps
        for _ in range(2):
            step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            step()       # blocking: returns when results are in host memory
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        # the D2H'd distances must equal the device-resident ones (same jobs, same kernel)
        o, w = lay[0], works[0]
        dd = bufs[0][o["dist"]: o["dist"] + w.n * w.csr.n_vertices * bpv["dist"]].view(torch.int16 if narrow else torch.int32)
        hd = hbufs[0][0]["dist"].view(-1)
        if hd.dtype == dd.dtype:
            assert torch.equal(hd, dd.cpu()), "host-pointer planes differ from the device-resident ones"
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        tj = torch.tensor([sum(w.n for w in works)], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dist.all_reduce(tj)
        return int(tj.item()) * n_e2e / float(tt.item()), int(h2d), int(d2h), n_e2e

    e2e_main = e2e_variant("caller16") or e2e_variant("all32")
    e2e_extra = {}
    if args.e2e_variants:
        for k in ("all16", "all32"):
            r = e2e_variant(k)
            if r:
                e2e_extra[k] = {"value": r[0], "h2d_bytes_per_step": r[1], "d2h_bytes_per_step": r[2]}
    clocks = sampler.stop()

    # ---- C5: the route / label stage behind the device SPT (host code today) -----------------
    route_stage = None
    if args.config == "C5" and rank == 0:
        from holo_b200 import ospfv2
        area = desc["_area"]
        k = args.steps
        ospfv2.run_area(ctx, area)
        t0 = time.perf_counter()
        for _ in range(k):
            ospfv2.run_area(ctx, area)
        route_stage = {"ms_per_root": 1e3 * (time.perf_counter() - t0) / k,
                       "what": "hspf_ospfv2_run_area: flatten + one device SPF + next-hop resolution, router table, "
                               f"intra-area routes with SR labels (host C++ behind the device SPT), LSDB-level call, {k} calls"}
        # the batched form: SPTs and the intra-area route cells of every root on the device
        # (hspf_ospfv2_run_area_batch), then the host decode of ONE root (the local router's)
        flat = ospfv2.Flat(area)
        rids = flat.ids[works[0].roots].astype(np.uint32)
        ospfv2.run_area_batch(ctx, area, rids[:8])
        t0 = time.perf_counter()
        b = ospfv2.run_area_batch(ctx, area, rids)
        t_batch = time.perf_counter() - t0
        rt = ospfv2.RouteTable(flat)
        j = int(np.nonzero(rids == area.router_id)[0][0]) if (rids == area.router_id).any() else None
        dec_ms = None
        if j is not None and b.status[j] == 0:
            gv, gn = b.gather(j)
            t0 = time.perf_counter()
            dec = ospfv2.routes_from_cells(area, rt, b.cells[j], gv, gn)
            dec_ms = 1e3 * (time.perf_counter() - t0)
            ref = ospfv2.run_area(ctx, area)
            keep = [n for n in dec.routes.dtype.names if n != "nh_off"]
            if dec.rc != 0 or not np.array_equal(dec.routes[keep], ref.routes[keep]):
                raise SystemExit("route cells of the local root do not decode to hspf_ospfv2_run_area's routes")
        route_stage["device_batch"] = {
            "roots": int(len(rids)), "prefixes": int(rt.n_prefixes), "advertisers": int(rt.n_contributors),
            "refused_roots": int((b.status != 0).sum()),
            "spt_batch_ms": b.device_ms[0], "route_kernel_ms": b.device_ms[1],
            "route_kernel_us_per_root": 1e3 * b.device_ms[1] / max(len(rids), 1),
            "cell_bytes": int(b.cells.nbytes),
            "route_kernel_GBps": b.cells.nbytes / max(b.device_ms[1], 1e-9) / 1e6,
            "call_wall_ms": 1e3 * t_batch,
            "host_decode_ms_one_root": dec_ms,
            "what": "hspf_ospfv2_run_area_batch: flatten + route table + one SPT batch + one thread per (root, prefix) "
                    "over the advertisers (update_rib_intra_area, route.rs:343-446) + cells back to pageable host memory; "
                    "hspf_ospfv2_routes_from_cells decodes one root's cells into interface next hops and SR labels",
        }

    # ---- max over ranks ----------------------------------------------------------------------
    tm = torch.tensor([total_ms, kernel_ms_avg, wall], dtype=torch.float64, device=dev)
    tj = torch.tensor([sum(w.n for w in works)], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(tj)
    total_ms, kernel_ms_avg, wall = [float(x) for x in tm.tolist()]
    jobs_per_step = int(tj.item())

    if rank == 0:
        value = jobs_per_step * args.steps / (total_ms * 1e-3)
        peaks = {}
        pk = ROOT / "MEASURED_PEAKS.json"
        if pk.exists():
            peaks = json.loads(pk.read_text())
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        alg = sum(alg_bytes(w.csr) * w.n for w in works)          # rank 0's launches of one step
        achieved = alg / (kernel_ms_avg * 1e-3) / 1e9
        traffic, traffic_src = None, None
        tjson = ROOT / "profiles" / "traffic.json"
        if tjson.exists() and args.config == "C2":
            try:
                tr = json.loads(tjson.read_text())
                # the capture is of the fast path with 16-bit planes: any other combination has no traffic figure
                if fast and narrow and str(tr.get("kernel", "")).startswith("spf_quad_kernel"):
                    traffic, traffic_src = tr.get("dram_bytes_per_launch"), tr.get("source")
            except Exception:
                traffic = None
        cpu = None if args.no_cpu_baseline else cpu_arms(works, seconds=args.cpu_seconds)
        if cpu and cpu.get("optimised", {}).get("value"):
            cpu["gpu_e2e_over_optimised_cpu"] = e2e_main[0] / cpu["optimised"]["value"]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": dict(config_dict(world, desc, works, exchange, "16-bit" if narrow else "32-bit"),
                           **({"exchange_bytes": exchange_note(xchg_bytes, tot)} if exchange != "none" else {})),
            "clocks": clocks,
            "e2e": {"value": e2e_main[0], "unit": UNIT, "h2d_bytes_per_step": e2e_main[1],
                    "d2h_bytes_per_step": e2e_main[2], "steps": e2e_main[3],
                    "planes": ("distance, hops, next-hop set (what holo-ospf's Vertex keeps), 16-bit" if (fast and is_ospf and max_atoms <= 16) else
                               "all five planes, 16-bit" if (fast and max_atoms <= 16) else "all five planes, 32/64-bit"),
                    "variants": e2e_extra or None},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "spf_quad_kernel" if fast else "spf_batch_kernel",
                         "kernel_ms": kernel_ms_avg, "launches_per_step": len(works),
                         "algorithmic_bytes_per_step": alg, "peak_source": peak_src},
            "cpu_baseline": cpu,
            "wall_ms_per_step": 1e3 * wall / args.steps,
        }
        if route_stage:
            line["route_stage"] = route_stage
        print(json.dumps(line))
    if xchg is not None:
        xchg.sync()
        barrier()          # nobody unmaps while a peer may still copy
        xchg.close()
    for g in graphs:
        g.free()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    global DELTA, JOBS_PER_GPU
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2", choices=["C1", "C2", "C3", "C4", "C5"],
                    help="BASELINE.json config (default C2, the one the metric is quoted on)")
    ap.add_argument("--planes", default="16", choices=["16", "32"],
                    help="result planes of the device-resident path: 16-bit (hspf_result16) where the fast path "
                         "serves the graph, else / or 32/64-bit (hspf_result)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=8.0, help="time bound of the faithful all-cores CPU sample")
    ap.add_argument("--no-e2e-variants", dest="e2e_variants", action="store_false")
    ap.add_argument("--exchange", default="auto", choices=["auto", "fused", "p2p", "nccl"],
                    help="N>1, C2 only: how the result planes reach the other GPUs: stored by the batch kernel itself "
                         "into peer memory (fused), copied by the copy engines over peer memory (p2p), or one NCCL "
                         "all-gather per step; auto = p2p up to 4 GPUs, fused above (16-bit vertex planes); peer memory "
                         "that cannot be mapped falls back to nccl")
    ap.add_argument("--xchg-planes", default="vertex", choices=["vertex", "all"],
                    help="N>1, C2: what every GPU receives from every other: the planes holo-ospf's Vertex keeps "
                         "(distance, hops, next-hop set + job status) or all five planes")
    ap.add_argument("--delta", type=int, default=0, help="SSSP bucket width (tuning; 0 = library default)")
    ap.add_argument("--jobs", type=int, default=JOBS_PER_GPU, help="SPF roots per GPU per step (tuning; BASELINE: 1000)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the result planes of the last one as DIR/<plane>.npy in "
                         "float32 / float64 (r<rank>_<plane>.npy with several GPUs), at most 64,000,000 bytes in all "
                         "(a seeded sample of the jobs), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm keeps no result planes)")
    DELTA = args.delta
    JOBS_PER_GPU = args.jobs
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
