#!/usr/bin/env python3
"""bench.py -- placements/sec of the topology-aware GPU placement scorer.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1], SURVEY.md 8(d) "C2"): 100,000 nodes x 10,000 pods, 8 GPUs per node,
k in {1,2,4,8}, seeded synthetic.  One "step" = one pass of the hot path over the whole pod batch: every pod
scored against every node (per pair: every k-subset of the node's free GPUs), best (cost, node, mask) per pod.
With N > 1 GPUs the node list is sharded contiguously over the ranks (strong scaling: cluster and batch stay
fixed), each rank scores its shard and the per-pod bests are exchanged over NVLink (--exchange: the peer-memory
push kernel, or NCCL all-gather + K2).

Prints ONE JSON line on rank 0.  Beyond the base contract:
  parity_in_run   the TIMED keys compared with the CPU oracle in the same run (all pods at N = 1, a sample at
                  N > 1); a mismatch fails the run.
  roofline        the binding resource of the headline kernel is warp-instruction issue, not HBM: achieved warp
                  instructions/s (ncu count of this build, profiles/k1s_counts.json) against SMs x 4 schedulers x
                  the SM clock sampled under load.  The algorithmic-bytes figure (260 B per pair, SURVEY.md 8(d))
                  is kept as `hbm_algorithmic` with the measured DRAM traffic beside it.
  hbm_regime      the same kernel where HBM IS the roof: millions of nodes, 1 .. 64 pods (node records streamed
                  once, hardly reused): DRAM GB/s against the measured copy peak.
  c5, c3          BASELINE configs[4] / configs[2] on this run's GPUs.
  noncollapsible  batches whose per-pod work cannot be memoised by k (per-pod min_mem; every pod distinct), with
                  their own CPU twin and parity check.
  memoised        what the snapshot collapse makes possible: GPU memo_by_k against the CPU's memoised twin.
  stateful_sequential   K3 against the CPU twin with the same two-level minima (one thread: the chain is serial).
  state_churn, upload   cost of state changes (1 % of the nodes change their masks before every step) and of ingest.
  multi_device_handle   (N > 1) rank 0 also scores C2 through ONE handle over all N devices
                        (kgpu_create(devs, N): in-library NCCL all-gather), keys compared.
  cpu_baseline    Oracle B (tuned C port, all host cores) on a bounded pod sample.
`--dump-outputs DIR` (rank 0) writes the keys of the last timed step, unpacked as a caller does (scorer.unpack_key), to
DIR/cost.npy, DIR/node_id.npy and DIR/gpu_mask.npy: float64[10000], exact (every field < 2**53); a pod without a fit
(KGPU_NO_FIT) reads 0xFFFFFF / 0xFFFFFFFF / 0xFF.  The inputs are seeded, so two builds can be compared file for file.
`--impl reference` times the CPU port of the path instead (the reference itself is Go with un-vendored
dependencies and cannot be built here: DESIGN.md "Oracle").
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

N_NODES = 100_000
N_PODS = 10_000
METRIC = "placements/sec on 100k-node x 10k-pod synthetic"
UNIT = "placements/s"
WORKLOAD = "C2: 100k nodes x 10k pods, 8 GPUs/node, k in {1,2,4,8}, seed 0xB2000001"
NO_FIT = np.uint64(0xFFFFFFFFFFFFFFFF)
RECORD_BYTES = 120          # what K1s streams per node: 112 B compacted pair costs + 4 B permutation/free count + 4 B node id


def algorithmic_bytes(n_nodes: int, n_pods: int) -> float:
    """SURVEY.md 8(d): 260 B per (pod,node) pair + 24 B per pod."""
    return 260.0 * n_nodes * n_pods + 24.0 * n_pods


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


KERNEL_SOURCES = ("score_pairs_sparse.cuh", "subset_dp_sparse_gen.cuh", "score_pairs.cuh", "sparse_work.h")


def kernel_source_sha() -> str:
    h = hashlib.sha256()
    for f in KERNEL_SOURCES:
        with open(os.path.join(ROOT, "kubegpu_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:12]


def dump_keys(out_dir: str, keys: np.ndarray) -> None:
    """--dump-outputs: the per-pod keys as the three fields a caller unpacks, float64 (lossless)."""
    os.makedirs(out_dir, exist_ok=True)
    fields = {"cost": keys >> np.uint64(40), "node_id": (keys >> np.uint64(8)) & np.uint64(0xFFFFFFFF), "gpu_mask": keys & np.uint64(0xFF)}
    for name, a in fields.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def committed_counts():
    """ncu counters of the headline kernel on C2 (one launch), written by scripts/refresh_counts.py from a
    `--metrics smsp__inst_executed.sum,dram__bytes_*` pass over THIS build's kernel sources."""
    try:
        with open(os.path.join(ROOT, "profiles", "k1s_counts.json")) as f:
            d = json.load(f)
        d["matches_this_build"] = d.get("kernel_source_sha") == kernel_source_sha()
        return d
    except Exception:
        return None


# ---------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, cuda_index: int):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.handle = None
        try:
            import pynvml
            import torch
            self.nv = pynvml
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(cuda_index).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            try:
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # NVML missing: report that instead of inventing numbers
            self.error = repr(e)

    def run(self):
        if self.handle is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def finish(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": getattr(self, "error", "no samples")}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------
def usable_cores() -> int:
    """Threads the CPU arm may really use: the scheduler affinity capped by the cgroup CPU quota
    (the GPU boxes show 128 logical CPUs but a 16- to 24-CPU quota)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def _sized_cpu_run(fn, n_pods, cores, target_s):
    """Grow the pod sample until one run takes >= target_s/2 (per-thread table building is a
    fixed cost, so a linear guess from a tiny probe undershoots).  fn(S) -> keys.  Returns (S, seconds, keys)."""
    S = min(n_pods, 2 * cores)
    while True:
        t0 = time.perf_counter()
        keys = fn(S)
        dt = max(time.perf_counter() - t0, 1e-6)
        if dt >= target_s / 2 or S >= n_pods:
            return S, dt, keys
        S = int(min(n_pods, max(S + cores, S * min(8.0, target_s / dt))))
        S = min(n_pods, (S + cores - 1) // cores * cores)


def cpu_baseline(topo, free, pods, gpu_keys, target_s: float = 10.0):
    """Oracle B (tuned port, all cores) on a bounded sample: the first S pods of the workload against ALL
    nodes, and the parity gate: those S keys must equal the keys the GPU produced in the timed region."""
    from oracle import oracle_b
    cores = usable_cores()
    S, dt, keys = _sized_cpu_run(lambda s: oracle_b.score_batch(topo, free, pods[:s], fast=True, nthreads=cores), len(pods), cores, target_s)
    mism = int((keys != gpu_keys[:S]).sum())
    out = {"value": S / dt, "unit": UNIT, "cores": cores, "kind": "port",
           "sample": "first %d of %d pods x all %d nodes, oracle/oracle_b.c tuned variant (per pair: the feasible "
                     "k-subsets of the node's free GPUs, like the GPU kernel), %d threads, %.2f s" % (S, len(pods), len(free), cores, dt)}
    t0 = time.perf_counter()
    oracle_b.score_batch(topo, free, pods[:16], fast=True, nthreads=1)
    out["single_thread"] = {"value": 16 / (time.perf_counter() - t0), "unit": UNIT, "sample": "16 pods x all nodes"}
    try:
        out["reference_algorithm_per_call"] = oracle_a_per_call_cost()
    except Exception as e:     # never let the context line break the bench
        out["reference_algorithm_per_call"] = {"error": repr(e)}
    return out, {"ok": mism == 0, "pods_checked": int(S), "mismatches": mism,
                 "against": "oracle/oracle_b.c on the host cores, same run, the keys of the timed region"}


def oracle_a_per_call_cost(n_nodes: int = 500, n_pods: int = 40):
    """Restatement of the reference algorithm (NOT Go): PodFitsDevice once per (node, pod) pair on a
    subsample, as SURVEY.md 8(d) asks; python, single thread."""
    from oracle import oracle_a as oa
    shapes = ([[8]], [[4], [4]], [[2, 2], [2, 2]], [[4, 4]])
    sched = oa.NvidiaGPUScheduler()
    nodes = []
    for i in range(n_nodes):
        ni = oa.NodeInfo(Allocatable=oa.shape_to_resources(shapes[i % 4]), KubeAlloc={oa.RESOURCE_GPU: 8})
        sched.AddNode("n%d" % i, ni)
        nodes.append(ni)
    t0 = time.perf_counter()
    calls = 0
    for p in range(n_pods):
        for ni in nodes:
            pod = oa.PodInfo(RunningContainers={"c": oa.ContainerInfo(Requests={oa.RESOURCE_GPU: (1, 2, 4, 8)[p % 4]})})
            sched.PodFitsDevice(ni, pod, False)
            calls += 1
    dt = time.perf_counter() - t0
    return {"us_per_PodFitsDevice_call": 1e6 * dt / calls, "calls": calls,
            "placements_per_s_if_100k_nodes": 1.0 / (dt / calls * 100_000),
            "note": "oracle/oracle_a.py (Python restatement of gpuschedulerplugin/gpu.go:94-324), 1 thread; "
                    "the Go original would be faster per call but does the same regex/map/tree work per pair"}


def run_reference(args):
    """--impl reference: the CPU port of the path on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from kubegpu_b200 import synth
    from oracle import oracle_b
    topo, free, pods = synth.gen_c2(N_NODES, N_PODS)
    cores = usable_cores()
    oracle_b.lib()
    # size each step's pod sample so that warmup+steps finish in a few minutes (<= ~6 s per step)
    budget = min(6.0, 150.0 / max(1, args.steps + args.warmup))
    S, _, _ = _sized_cpu_run(lambda s: oracle_b.score_batch(topo, free, pods[:s], fast=True, nthreads=cores), N_PODS, cores, budget)
    for _ in range(args.warmup):
        oracle_b.score_batch(topo, free, pods[:S], fast=True, nthreads=cores)
    t0 = time.perf_counter()
    for i in range(args.steps):
        off = (i * S) % max(1, N_PODS - S + 1)
        oracle_b.score_batch(topo, free, pods[off:off + S], fast=True, nthreads=cores)
    dt = time.perf_counter() - t0
    value = args.steps * S / dt
    sample = "each step: %d of %d pods x all %d nodes, oracle/oracle_b.c tuned variant, %d threads" % (S, N_PODS, N_NODES, cores)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps * (N_PODS / S),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32",
        "data": "synthetic", "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference is Go with un-vendored deps (no toolchain here): CPU port of the path timed instead; "
                "ms_per_step is extrapolated to the full 10k-pod batch",
    }))


# ---------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="kgpu", choices=["kgpu", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-variants", action="store_true", help="skip every context / sub-object line (headline only)")
    ap.add_argument("--exchange", default="auto", choices=["auto", "nccl", "allreduce", "push"],
                    help="multi-GPU key exchange: peer-memory push kernel (auto when it connects), NCCL all-gather + K2, "
                         "or one NCCL all-reduce(min)")
    ap.add_argument("--graph", action="store_true", help="replay the NCCL-path step as one CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the keys of the last timed step to DIR/*.npy (kgpu arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the kgpu arm")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from kubegpu_b200 import _lib, synth
    from kubegpu_b200.distributed import all_reduce_min_keys, shard_range
    from kubegpu_b200.scorer import Scorer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d (launch with torch.distributed.run for N>1)" % (args.gpus, world))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: kubegpu_b200 has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"                      # no version banner on stdout: one JSON line only
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
        host_group = dist.new_group(backend="gloo")            # host-side barriers: waiting ranks must not spin on their GPU
    W = max(3, args.warmup)
    K = args.steps
    peak, peak_src = measured_peak_gbs()
    props = torch.cuda.get_device_properties(local_rank)
    stream = torch.cuda.Stream(device=dev)          # everything (K1, exchange, copies) is enqueued here
    torch.cuda.set_stream(stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- inputs: this rank's contiguous node shard, the full pod batch -----------------
    lo, hi = shard_range(N_NODES, world, rank)
    topo, free, pods = synth.gen_c2(hi - lo, N_PODS, node_start=lo)
    scorer = Scorer((local_rank,))
    scorer.set_variant(_lib.VARIANT_SPARSE)                   # headline kernel K1s (per-pair work, see DESIGN.md)
    scorer.upload_nodes(topo, free, node_id_base=lo)          # resident in HBM before timing
    upload_ms_c2 = scorer.last_upload_ms

    d_pods = torch.from_numpy(pods).to(dev)
    d_local = torch.empty(N_PODS, dtype=torch.int64, device=dev)
    d_gather = torch.empty((world, N_PODS), dtype=torch.int64, device=dev) if world > 1 else None
    d_final = torch.empty(N_PODS, dtype=torch.int64, device=dev) if world > 1 else d_local
    h_pods = torch.from_numpy(pods).pin_memory()
    h_keys = torch.empty(N_PODS, dtype=torch.int64).pin_memory()

    # ---- exchange: peer-memory exchange (one kernel: stores into every rank's slot array over NVLink
    # + flag barrier) when every rank can map every peer; else NCCL all-gather + K2 -------------------------
    exchange = args.exchange
    if exchange == "auto":
        exchange = "push" if world > 1 and not args.graph else "nccl"
    push = False
    max_pods_x = 131_072                                       # also serves the C3 sub-run (100k pods)
    if exchange == "push":
        ok = 1
        try:
            mine = scorer.exchange_init(world, rank, max_pods_x)
            handles = [None] * world
            if world > 1:
                dist.all_gather_object(handles, mine)
            else:
                handles = [mine]
            scorer.exchange_connect(handles)
        except Exception as e:                                  # no peer access / IPC: fall back, all ranks together
            ok = 0
            sys.stderr.write("rank %d: peer exchange unavailable (%r), using NCCL\n" % (rank, e))
        t = torch.tensor([ok], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
        push = bool(int(t.item()))
        if not push:
            exchange = "nccl"
    wrapped = {}

    class _DeviceKeys:                              # zero-copy view of the handle-owned result array
        def __init__(self, ptr, n):
            self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i8", "data": (ptr, False), "version": 3}

    def step_on(sc, dp, n_pods, local, gather, final):
        """pods already in HBM -> final keys in HBM on every rank; returns the tensor holding them."""
        sptr = torch.cuda.current_stream().cuda_stream          # the capture stream while a graph is recorded
        if push:
            ptr = sc.score_batch_exchange(dp.data_ptr(), n_pods, sptr, _lib.BATCH_NO_MIN_MEM)
            if (ptr, n_pods) not in wrapped:
                wrapped[(ptr, n_pods)] = torch.as_tensor(_DeviceKeys(ptr, n_pods), device=dev)
            return wrapped[(ptr, n_pods)]
        sc.score_batch_device(dp.data_ptr(), n_pods, local.data_ptr(), sptr, _lib.BATCH_NO_MIN_MEM)
        if world > 1 and exchange == "allreduce":                # one collective, no K2
            return all_reduce_min_keys(local)
        if world > 1:
            dist.all_gather_into_tensor(gather.view(-1), local)
            sc.reduce_shards_device(gather.data_ptr(), world, n_pods, final.data_ptr(), sptr)
            return final
        return local

    last_keys = [None]                              # the tensor the last (or the graph-captured) step left its keys in

    def step_device():
        last_keys[0] = step_on(scorer, d_pods, N_PODS, d_local, d_gather, d_final)
        return last_keys[0]

    def step_e2e():
        """host pods -> host keys through the public call."""
        if world == 1 and not push:
            scorer.score_batch_ptr(h_pods.data_ptr(), N_PODS, h_keys.data_ptr())   # kgpu_score_batch: H2D + K1 + D2H
        else:
            d_pods.copy_(h_pods, non_blocking=True)
            h_keys.copy_(step_device(), non_blocking=True)
            stream.synchronize()

    def timed(fn, steps, rendezvous=True):
        """CUDA-event time of `steps` calls of fn on the bench stream, L2 flushed before each; max over ranks of the SUM."""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        token = torch.zeros(1, device=dev)
        for a, b in ev:
            flush.zero_()
            if world > 1 and rendezvous:               # device-side rendezvous so no rank times another's flush
                if push:
                    scorer.exchange_barrier(stream.cuda_stream)   # the exchange kernel's own flag barrier: ranks leave within ~1 us
                else:
                    dist.all_reduce(token)             # (a ring all-reduce releases its ranks several us apart)
            a.record(stream)
            fn()
            b.record(stream)
        barrier()
        return max_over_ranks(sum(a.elapsed_time(b) for a, b in ev))

    # ---- headline: device-resident timing -> `value`, kernel-only timing -> the roofline ------------------
    for _ in range(W):
        flush.zero_()
        step_device()
    graph = None
    launches_before_capture = scorer.kernel_launches
    if args.graph and not push:
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            step_device()
    if graph is not None:
        launches_before_capture = scorer.kernel_launches - launches_before_capture      # launches recorded into the graph
    barrier()
    launches0 = scorer.kernel_launches
    sampler = ClockSampler(local_rank)
    sampler.start()
    total_ms = timed(graph.replay if graph is not None else step_device, K)
    gpu_launches = scorer.kernel_launches - launches0 if graph is None else K * (scorer.kernel_launches - launches_before_capture)
    timed_keys = last_keys[0].cpu().numpy().view(np.uint64).copy()   # the last timed step's keys, kept for the parity gate
    if rank == 0 and args.dump_outputs:
        dump_keys(args.dump_outputs, timed_keys)
    # kernel only (no exchange): K1s launch(es) on this rank's shard
    k1_total_ms = timed(lambda: scorer.score_batch_device(d_pods.data_ptr(), N_PODS, d_local.data_ptr(), stream.cuda_stream,
                                                          _lib.BATCH_NO_MIN_MEM), K)
    clocks = sampler.finish()
    ms_per_step = total_ms / K
    value = N_PODS / (ms_per_step * 1e-3)
    kernel_ms = k1_total_ms / K

    # ---- end to end through the host-buffer call ---------------------------------------
    for _ in range(W):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        step_e2e()
    t1 = time.perf_counter()        # step_e2e is synchronous: this rank's K results are in host memory now
    barrier()                       # (closing barrier outside the interval: a dist.barrier() costs up to milliseconds, K steps take 2-9 ms)
    e2e_value = N_PODS * K / max_over_ranks(t1 - t0)
    e2e_keys = h_keys.numpy().view(np.uint64).copy()

    line = None
    if rank == 0:
        counts = committed_counts()
        sm_mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0
        issue_peak = props.multi_processor_count * 4 * sm_mhz * 1e6 / 1e9              # G warp-instructions / s
        roof = {"bound": "issue", "unit": "Gwarp-inst/s", "peak": issue_peak,
                "peak_source": "%d SMs x 4 schedulers x %.0f MHz (SM clock sampled under load)" % (props.multi_processor_count, sm_mhz),
                "kernel": "score_pairs_sparse<PER_PAIR, !MEM, BYTE_KEYS>", "kernel_ms": kernel_ms}
        if counts and world == 1:
            inst = float(counts["inst_per_launch_c2"])
            roof.update({"achieved": inst / (kernel_ms * 1e-3) / 1e9, "inst_per_launch": inst,
                         "inst_source": "profiles/k1s_counts.json (ncu smsp__inst_executed.sum of this workload)",
                         "inst_matches_this_build": counts["matches_this_build"],
                         "traffic": counts.get("dram_bytes_per_launch_c2")})
            roof["frac"] = roof["achieved"] / issue_peak
        else:
            roof.update({"achieved": None, "frac": None, "traffic": counts.get("dram_bytes_per_launch_c2") if counts else None,
                         "note": "instruction count is per 1-GPU launch; see the N=1 line"})
        alg = algorithmic_bytes(hi - lo, N_PODS) / (kernel_ms * 1e-3) / 1e9
        roof["hbm_algorithmic"] = {"achieved": alg, "peak": peak, "unit": "GB/s", "frac": alg / peak, "peak_source": peak_src,
                                   "note": "260 B/pair + 24 B/pod (SURVEY.md 8(d)) / kernel time; > 1 because a staged node is reused "
                                           "for every pod of the block: DRAM traffic per launch is `traffic`, not the algorithmic bytes; "
                                           "HBM as the roof is measured in `hbm_regime`"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "nodes": N_NODES, "pods": N_PODS,
                       "parallelism": ("node list sharded over %d GPU(s), " % world + {"push": "peer-memory exchange: stores into every rank's slots + flag barrier + local min (1 kernel over NVLink)",
                                                                                       "allreduce": "1 NCCL all-reduce(min)",
                                                                                       "nccl": "1 NCCL all-gather + K2"}[exchange]) if world > 1 else "1 GPU, no collective",
                       "kernel": "score_pairs_sparse (per pair: every k-subset of the node's free-GPU positions; not memoised by k: see `memoised`)",
                       "l2": "flushed between timed iterations (256 MiB write); node records are 12 MB < L2",
                       "graph": bool(graph is not None)},
            "roofline": roof,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": N_PODS * 16, "d2h_bytes_per_step": N_PODS * 8,
                    "call": "kgpu_score_batch(host pods, host keys)" if world == 1 and not push else "pinned H2D + kgpu_score_batch_exchange / K1 + exchange + D2H"},
            "gpu_launches": int(gpu_launches),
            "clocks": clocks,
            "no_fit_pods": int((timed_keys == NO_FIT).sum()),
            "keys_sha256_12": hashlib.sha256(timed_keys.tobytes()).hexdigest()[:12],
            "upload": {"c2_shard_nodes": int(hi - lo), "upload_ms": upload_ms_c2,
                       "what": "kgpu_upload_nodes: pageable H2D + device-side value check + counting-sort order + compacted records"},
        }
        if not (e2e_keys == timed_keys).all():
            line["parity_in_run"] = {"ok": False, "mismatches": int((e2e_keys != timed_keys).sum()), "against": "e2e keys vs device-path keys"}

    # ---- parity gate: the timed keys against the CPU oracle, in this run ------------------------------------
    if rank == 0 and not args.no_cpu_baseline:
        if world == 1:
            line["cpu_baseline"], par = cpu_baseline(topo, free, pods, timed_keys)
        else:
            from oracle import oracle_b
            ftopo, ffree, _ = synth.gen_c2(N_NODES, 0)
            S = 512
            want = oracle_b.score_batch(ftopo, ffree, pods[:S], fast=True, nthreads=usable_cores())
            mism = int((want != timed_keys[:S]).sum())
            par = {"ok": mism == 0, "pods_checked": S, "mismatches": mism,
                   "against": "oracle/oracle_b.c over all %d nodes on rank 0's host cores, same run" % N_NODES}
        if "parity_in_run" not in line:
            line["parity_in_run"] = par
    elif rank == 0 and world == 1:
        line["cpu_baseline"] = None

    extras = not args.no_variants
    # ---- context: the other K1 variants, and what memoising by k does (N = 1) -------------------------------
    if extras and world == 1 and not push:
        variants = {}
        for name, var, reps in (("lane_per_node_dense_all_C8k_subsets", _lib.VARIANT_LANE_PER_NODE, 5),
                                ("warp_per_pair_north_star_mapping", _lib.VARIANT_WARP_PER_PAIR, 2),
                                ("tile_memo_not_headline", _lib.VARIANT_TILE_MEMO, 10),
                                ("memo_by_k_not_headline", _lib.VARIANT_MEMO_BY_K, 10)):
            scorer.set_variant(var)
            step_device()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(reps):
                step_device()
            b.record(stream)
            torch.cuda.synchronize()
            ms = a.elapsed_time(b) / reps
            same = bool((d_local.cpu().numpy().view(np.uint64) == timed_keys).all())
            variants[name] = {"ms_per_step": ms, "value": N_PODS / (ms * 1e-3), "unit": UNIT, "keys_identical_to_headline": same}
        line["variants"] = variants
        # memoised: e2e through kgpu_score_batch with the memo variant against the CPU's memoised twin
        scorer.set_variant(_lib.VARIANT_MEMO_BY_K)
        for _ in range(3):
            scorer.score_batch_ptr(h_pods.data_ptr(), N_PODS, h_keys.data_ptr())
        t0 = time.perf_counter()
        for _ in range(20):
            scorer.score_batch_ptr(h_pods.data_ptr(), N_PODS, h_keys.data_ptr())
        memo_e2e = 20 * N_PODS / (time.perf_counter() - t0)
        memo_same = bool((h_keys.numpy().view(np.uint64) == timed_keys).all())
        scorer.set_variant(_lib.VARIANT_SPARSE)
        from oracle import oracle_b
        cores = usable_cores()
        oracle_b.score_batch_memo(topo, free, pods, nthreads=cores)
        t0 = time.perf_counter()
        for _ in range(3):
            ck = oracle_b.score_batch_memo(topo, free, pods, nthreads=cores)
        cpu_memo = 3 * N_PODS / (time.perf_counter() - t0)
        line["memoised"] = {"gpu_e2e_value": memo_e2e, "gpu_kernel_ms": variants["memo_by_k_not_headline"]["ms_per_step"],
                            "cpu_value": cpu_memo, "cpu_cores": cores, "unit": UNIT, "ratio_e2e": memo_e2e / cpu_memo,
                            "keys_identical": memo_same and bool((ck == timed_keys).all()),
                            "note": "with snapshot scoring and no per-pod constraint a pod's key depends on the pod only through k: best[k] "
                                    "over all nodes once, then a gather (KGPU_VARIANT_MEMO_BY_K / oracle score_batch_memo).  The headline "
                                    "does the per-pair work north_star names; this object is what a caller who only has such pods gets."}

    # ---- non-collapsible batches: per-pod memory requirements (N = 1) ----------------------------------------
    if extras and world == 1 and not push:
        from oracle import oracle_b
        cores = usable_cores()
        topo6, free6, mem6, pods6 = synth.gen_c6()
        pods7 = pods6.copy()                       # every pod a DISTINCT requirement: nothing repeats within a k
        pods7[:, 3] = 1_000 + (synth.rand_below(synth.SEED_C6, 21, len(pods7), 180_000) // 10_000) * 10_000 + np.arange(len(pods7)) % 10_000
        nc = {}
        with Scorer((local_rank,)) as s6:
            s6.set_variant(_lib.VARIANT_SPARSE)
            s6.upload_nodes(topo6, free6)
            s6.upload_gpu_memory(mem6)
            for tag, pp, what in (("c6_min_mem_classes", pods6, "C6: 100k heterogeneous nodes, per-GPU memory classes, 10k pods, k in 1..8, 4 of 7 pods with one of 4 min_mem values"),
                                  ("c7_distinct_min_mem", pods7, "C6's nodes, every pod with its own min_mem (10k distinct values): no two pods share a requirement")):
                dp = torch.from_numpy(pp).to(dev)
                dk = torch.empty(len(pp), dtype=torch.int64, device=dev)
                for _ in range(3):
                    s6.score_batch_device(dp.data_ptr(), len(pp), dk.data_ptr(), stream.cuda_stream)
                ms = timed(lambda: s6.score_batch_device(dp.data_ptr(), len(pp), dk.data_ptr(), stream.cuda_stream), 5) / 5
                got = dk.cpu().numpy().view(np.uint64)
                S, dt, want = _sized_cpu_run(lambda s: oracle_b.score_batch(topo6, free6, pp[:s], fast=True, nthreads=cores, mem=mem6), len(pp), cores, 4.0)
                hp, hk = torch.from_numpy(pp).pin_memory(), torch.empty(len(pp), dtype=torch.int64).pin_memory()
                s6.score_batch_ptr(hp.data_ptr(), len(pp), hk.data_ptr())
                t0 = time.perf_counter()
                for _ in range(5):
                    s6.score_batch_ptr(hp.data_ptr(), len(pp), hk.data_ptr())
                e2e6 = 5 * len(pp) / (time.perf_counter() - t0)
                nc[tag] = {"workload": what, "kernel_ms": ms, "value": len(pp) / (ms * 1e-3), "e2e_value": e2e6, "unit": UNIT,
                           "vs_c2_kernel_ms": ms / kernel_ms, "cpu_value": S / dt, "cpu_cores": cores,
                           "cpu_sample": "first %d pods x all nodes, %.2f s" % (S, dt), "ratio_e2e": e2e6 / (S / dt),
                           "parity": {"ok": bool((got[:S] == want).all() and (hk.numpy().view(np.uint64) == got).all()), "pods_checked": int(S)}}
            # sequential + memory-aware (one table set per distinct requirement of the batch; <= 7)
            s6.place_batch(pods6[:256])
            s6.upload_nodes(topo6, free6)
            s6.upload_gpu_memory(mem6)
            s6.place_batch(pods6)
            nc["c6_sequential_ms_per_batch"] = s6.last_kernel_ms
        nc["note"] = ("K1s for the pods without a requirement + K1m (MEM instantiation: per-(pod,node) eligibility masks) for the others; "
                      "algorithmic bytes 292 B per pair on the K1m path (+32 B memory row)")
        line["noncollapsible"] = nc

    # ---- stateful sequential placement (K3) against the CPU twin with the same two-level minima -------------
    if extras and world == 1:
        from oracle import oracle_b
        scorer.place_batch(pods[:256])                     # warm-up (changes the masks: re-upload below)
        seq_ms = []
        for _ in range(3):
            scorer.upload_nodes(topo, free, node_id_base=lo)
            got = scorer.place_batch(pods)
            seq_ms.append(scorer.last_kernel_ms)
        masks_after = scorer.get_free_masks()
        scorer.upload_nodes(topo, free, node_id_base=lo)
        ms = float(np.median(seq_ms))
        t0 = time.perf_counter()
        want, wf = oracle_b.place_batch(topo, free, pods, tiled=True)
        cpu_s = time.perf_counter() - t0
        line["stateful_sequential"] = {
            "kernel": "place_init + place_sequential (kgpu_place_batch)", "ms_per_batch": ms, "value": N_PODS / (ms * 1e-3),
            "cpu_twin_value": N_PODS / cpu_s, "cpu_twin": "oracle kgpu_oracle_place_batch_tiled: same node keys / 128-node tile minima / "
                                                          "supertile minima, 1 thread (the chain is serial), table build included",
            "ratio": (N_PODS / (ms * 1e-3)) / (N_PODS / cpu_s), "unit": UNIT,
            "parity": {"ok": bool((got == want).all() and (masks_after == wf).all()), "pods_checked": N_PODS, "final_masks_checked": True},
            "note": "each pod sees the free masks left by the pods before it (no snapshot collapse); exact and order dependent"}

    # ---- state changes: 1 % of the nodes change their free masks before every step (N = 1) ------------------
    if extras and world == 1 and not push:
        rng = np.random.default_rng(1)
        cur = free.copy()
        churn_ms, upd_ms = [], []
        for it in range(6):
            idx = rng.choice(N_NODES, size=N_NODES // 100, replace=False).astype(np.int64)
            masks = rng.integers(0, 256, size=len(idx)).astype(np.int32)
            cur[idx] = masks
            t0 = time.perf_counter()
            scorer.set_free_masks(idx, masks)
            t1 = time.perf_counter()
            scorer.score_batch_ptr(h_pods.data_ptr(), N_PODS, h_keys.data_ptr())
            t2 = time.perf_counter()
            if it > 0:
                upd_ms.append(1e3 * (t1 - t0))
                churn_ms.append(1e3 * (t2 - t0))
        from oracle import oracle_b
        S = 256
        ok = bool((oracle_b.score_batch(topo, cur, pods[:S], fast=True, nthreads=usable_cores()) == h_keys.numpy().view(np.uint64)[:S]).all())
        scorer.upload_nodes(topo, free, node_id_base=lo)
        line["state_churn"] = {"step_after_1pct_mask_churn_ms": float(np.median(churn_ms)), "set_free_masks_ms": float(np.median(upd_ms)),
                               "nodes_changed_per_step": N_NODES // 100, "e2e_value": N_PODS / (float(np.median(churn_ms)) * 1e-3), "unit": UNIT,
                               "parity": {"ok": ok, "pods_checked": S},
                               "what": "kgpu_set_free_masks (1 H2D + 1 kernel: scatter + refresh of those nodes' records; re-sort when > n/200 "
                                       "nodes have changed) + kgpu_score_batch, host buffers, wall clock"}
        # PodFitsDevice served from the (node, k) fit table
        scorer.build_fit_table()
        t0 = time.perf_counter()
        for i in range(20_000):
            scorer.fit_lookup(i, 1 + (i & 7))
        line["pod_fits_device"] = {"us_per_lookup_through_ctypes": 1e6 * (time.perf_counter() - t0) / 20_000,
                                   "what": "kgpu_fit_lookup: a host read of the handle's (node, k) table (built by one launch, rows refreshed by "
                                           "state changes); the time is Python's ctypes call overhead, no launch or copy per call"}

    # ---- BASELINE configs[4] (C5): node-count sweep on this run's GPUs; configs[2] (C3) ----------------------
    if extras:
        c5 = []
        for n_total in (10_000, 100_000, 1_000_000):
            l5, h5 = shard_range(n_total, world, rank)
            t5, f5, p5 = synth.gen_c2(h5 - l5, N_PODS, seed=synth.SEED_C5, node_start=l5)
            with Scorer((local_rank,)) as s5:
                s5.set_variant(_lib.VARIANT_SPARSE)
                s5.upload_nodes(t5, f5, node_id_base=l5)
                up = s5.last_upload_ms
                dp = torch.from_numpy(p5).to(dev)
                dl = torch.empty(N_PODS, dtype=torch.int64, device=dev)
                dg = torch.empty((world, N_PODS), dtype=torch.int64, device=dev) if world > 1 else None
                df = torch.empty(N_PODS, dtype=torch.int64, device=dev) if world > 1 else dl
                fn = lambda: s5.score_batch_device(dp.data_ptr(), N_PODS, dl.data_ptr(), stream.cuda_stream, _lib.BATCH_NO_MIN_MEM)
                if world > 1:
                    def fn(s5=s5, dp=dp, dl=dl, dg=dg, df=df):   # NCCL exchange for the sub-runs (the push buffers belong to `scorer`)
                        s5.score_batch_device(dp.data_ptr(), N_PODS, dl.data_ptr(), stream.cuda_stream, _lib.BATCH_NO_MIN_MEM)
                        dist.all_gather_into_tensor(dg.view(-1), dl)
                        s5.reduce_shards_device(dg.data_ptr(), world, N_PODS, df.data_ptr(), stream.cuda_stream)
                for _ in range(3):
                    fn()
                barrier()                              # ranks enter the timed steps together (their device-side rendezvous waits on the GPU)
                reps = 5 if n_total <= 100_000 else 3
                ms = timed(fn, reps) / reps
                if rank == 0:
                    c5.append({"nodes": n_total, "pods": N_PODS, "ms_per_step": ms, "value": N_PODS / (ms * 1e-3), "gpairs_per_s": n_total * N_PODS / ms / 1e6,
                               "algorithmic_gbs_per_gpu": algorithmic_bytes(h5 - l5, N_PODS) / ms / 1e6,
                               "dram_gbs_min_per_gpu": RECORD_BYTES * (h5 - l5) / ms / 1e6, "upload_ms": up,
                               "keys_sha256_12": hashlib.sha256(df.cpu().numpy().tobytes()).hexdigest()[:12]})
                del dp, dl, dg, df
        if rank == 0:
            line["c5"] = {"points": c5, "unit": UNIT,
                          "note": "BASELINE configs[4]: C2's distributions, seed 0xB2000005, sharded over this run's GPUs (NCCL all-gather + K2); "
                                  "dram_gbs_min = node records (120 B/node) once per launch: with 10k pods the kernel is issue bound at every N "
                                  "(the records are read once and reused for every pod), so DRAM GB/s falls as reuse grows; "
                                  "the 10M-node point and the DRAM-bound regime are in `hbm_regime`"}
        # C3: 1M nodes x 100k pods, k uniform 1..8
        l3, h3 = shard_range(1_000_000, world, rank)
        t3, f3, p3 = synth.gen_c3(h3 - l3, 100_000, node_start=l3)
        with Scorer((local_rank,)) as s3:
            s3.set_variant(_lib.VARIANT_SPARSE)
            s3.upload_nodes(t3, f3, node_id_base=l3)
            P3 = len(p3)
            dp = torch.from_numpy(p3).to(dev)
            dl = torch.empty(P3, dtype=torch.int64, device=dev)
            dg = torch.empty((world, P3), dtype=torch.int64, device=dev) if world > 1 else None
            df = torch.empty(P3, dtype=torch.int64, device=dev) if world > 1 else dl

            def fn3():
                s3.score_batch_device(dp.data_ptr(), P3, dl.data_ptr(), stream.cuda_stream, _lib.BATCH_NO_MIN_MEM)
                if world > 1:
                    dist.all_gather_into_tensor(dg.view(-1), dl)
                    s3.reduce_shards_device(dg.data_ptr(), world, P3, df.data_ptr(), stream.cuda_stream)
            fn3()
            barrier()
            ms3 = timed(fn3, 2) / 2
            k3 = df.cpu().numpy().view(np.uint64)
        if rank == 0:
            from oracle import oracle_b
            S3 = 16
            ft3, ff3, _ = synth.gen_c3(1_000_000, 0)
            ok3 = bool((oracle_b.score_batch(ft3, ff3, p3[:S3], fast=True, nthreads=usable_cores()) == k3[:S3]).all())
            del ft3, ff3
            line["c3"] = {"workload": "C3: 1M nodes x 100k pods, k uniform 1..8, seed 0xB2000002, node list sharded over %d GPU(s)" % world,
                          "ms_per_step": ms3, "value": 100_000 / (ms3 * 1e-3), "unit": UNIT, "gpairs_per_s": 1e11 / ms3 / 1e6,
                          "algorithmic_gbs_per_gpu": algorithmic_bytes(h3 - l3, 100_000) / ms3 / 1e6,
                          "keys_sha256_12": hashlib.sha256(k3.tobytes()).hexdigest()[:12],
                          "parity": {"ok": ok3, "pods_checked": S3, "against": "oracle over all 1M nodes"}}
        del t3, f3

    # ---- the regime where HBM is the roof: millions of nodes, 1 .. 64 pods (N = 1) --------------------------
    if extras and world == 1:
        n_big = 10_485_760
        tb, fb, _ = synth.gen_c2(n_big, 0, seed=synth.SEED_C5)
        with Scorer((local_rank,)) as sb:
            sb.set_variant(_lib.VARIANT_SPARSE)
            sb.upload_nodes(tb, fb)
            up_big = sb.last_upload_ms
            pts = []
            from oracle import oracle_b
            for pcount in (1, 8, 16, 32, 64):
                _, _, pb = synth.gen_c2(0, pcount, seed=synth.SEED_C5)
                dp = torch.from_numpy(pb).to(dev)
                dk = torch.empty(pcount, dtype=torch.int64, device=dev)
                f = lambda: sb.score_batch_device(dp.data_ptr(), pcount, dk.data_ptr(), stream.cuda_stream, _lib.BATCH_NO_MIN_MEM)
                for _ in range(3):
                    f()
                ms = timed(f, 5) / 5
                gbs = RECORD_BYTES * n_big / ms / 1e6
                ok = bool((oracle_b.score_batch_memo(tb, fb, pb, nthreads=usable_cores()) == dk.cpu().numpy().view(np.uint64)).all())
                pts.append({"pods": pcount, "ms": ms, "dram_gbs_min": gbs, "frac_of_hbm_peak": gbs / peak,
                            "algorithmic_gbs": algorithmic_bytes(n_big, pcount) / ms / 1e6, "placements_per_s": pcount / (ms * 1e-3),
                            "parity": {"ok": ok, "pods_checked": pcount, "against": "oracle score_batch_memo over all nodes (pods without min_mem)"}})
        del tb, fb
        line["hbm_regime"] = {"nodes": n_big, "points": pts, "peak_gbs": peak, "peak_source": peak_src, "upload_ms": up_big,
                              "bytes_per_node_streamed": RECORD_BYTES,
                              "note": "1.26 GB of node records (> 126 MB L2), L2 flushed before every launch: every record comes from DRAM once; "
                                      "dram_gbs_min = 120 B x nodes / time is a lower bound of the DRAM rate (ncu: profiles/r02_k1s_tma_p{1,32}_ncu_raw.txt: dram__bytes_read = 1.2002 GB for 10M nodes, no over-fetch). Up to 64 pods the tiles are staged by cp.async.bulk (TMA) into shared memory, 7 / 8 blocks per SM. "
                                      "The algorithmic figure counts 260 B per pair, i.e. the uncompacted matrix."}

    # ---- N > 1: the single-process multi-device handle (in-library NCCL all-gather), on rank 0 ---------------
    if world > 1 and extras:
        # The other ranks wait on the HOST (gloo): an NCCL barrier would keep a spinning kernel on their GPUs and
        # rank 0's work on those devices would be time-sliced against it.
        torch.cuda.synchronize()
        dist.barrier(group=host_group)
        if rank == 0:
            md = {}
            try:
                ftopo, ffree, _ = synth.gen_c2(N_NODES, 0)
                with Scorer(tuple(range(world))) as sm:
                    sm.set_variant(_lib.VARIANT_SPARSE)
                    sm.upload_nodes(ftopo, ffree)
                    hk = torch.empty(N_PODS, dtype=torch.int64).pin_memory()
                    for _ in range(3):
                        sm.score_batch_ptr(h_pods.data_ptr(), N_PODS, hk.data_ptr())
                    t0 = time.perf_counter()
                    for _ in range(10):
                        sm.score_batch_ptr(h_pods.data_ptr(), N_PODS, hk.data_ptr())
                    dt = (time.perf_counter() - t0) / 10
                    md = {"devices": world, "ms_per_call": 1e3 * dt, "e2e_value": N_PODS / dt, "kernel_ms_max_over_devices": sm.last_kernel_ms,
                          "keys_identical": bool((hk.numpy().view(np.uint64) == timed_keys).all()), "unit": UNIT,
                          "call": "kgpu_create(devs, %d) + kgpu_score_batch(host pods, host keys): per-device K1s, grouped ncclAllGather, K2 on device 0" % world}
            except Exception as e:
                md = {"error": repr(e)}
            line["multi_device_handle"] = md
        dist.barrier(group=host_group)

    if rank == 0:
        par = line.get("parity_in_run")
        subs = [line[k]["parity"]["ok"] for k in ("stateful_sequential", "state_churn", "c3") if k in line and "parity" in line[k]]
        subs += [v["parity"]["ok"] for v in line.get("noncollapsible", {}).values() if isinstance(v, dict) and "parity" in v]
        subs += [p["parity"]["ok"] for p in line.get("hbm_regime", {}).get("points", [])]
        line["parity_all_subruns_ok"] = all(subs)
        print(json.dumps(line))
        if (par is not None and not par["ok"]) or not all(subs):
            sys.stderr.write("bench.py: PARITY FAILURE in the timed run: %r / sub-runs %r\n" % (par, subs))
            scorer.close()
            if world > 1:
                dist.destroy_process_group()
            sys.exit(3)
    scorer.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
