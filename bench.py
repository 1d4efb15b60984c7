#!/usr/bin/env python
"""bench.py — endpoint picks/sec at 64K requests x 1024 endpoints (BASELINE.json headline), all four
scorers (queue 2, kv 2, prefix 3, lora 1), 2 KB shared-prefix prompts, on N B200s of one node.

A "step" = one pass of the hot path over one batch of R requests per GPU:
    prepare_endpoints + prepare_adapters (side stream) ‖ hash_bodies + hash_chain (chained XXH64 of every prompt)  →  pick_sparse (table probe, 4 scorers, weighted float64 sum, arg-max pick) + the full-matrix kernel
    on the requests pick_sparse deferred — 6 kernel launches replayed as one CUDA graph, nothing else.
`value`  : whole-job picks/s with the inputs already resident in HBM (CUDA events, max over ranks).
`e2e`    : the same metric through the C ABI with HOST (pinned) buffers: H2D of prompts/seeds/adapters
           and D2H of picks/scores/tie counts inside the timed region.
`roofline`: algorithmic bytes of the dominant kernel / its CUDA-event duration, vs MEASURED_PEAKS.json; `step_frac` = the
           step's compulsory HBM bytes / ms_per_step / peak; `dram_frac` = measured DRAM traffic of that kernel / time / peak.
`closed_loop`: schedule -> PreRequest commit -> schedule ... with the commit (device-resident index) inside the timed region;
           on N GPUs every rank all-gathers the shards' commits (NCCL) and replays them in global request order.
`cpu_baseline`: the CPU oracle port (oracle/oracle.c; the Go reference cannot be built here) on the
           box's host cores, same workload.
`--impl reference` times that CPU port alone (all host threads) with the same JSON contract.
`--workload E` runs BASELINE.json's last configuration (1M requests x 4096 endpoints, request-sharded over the N GPUs).
`--dump-outputs DIR` writes what the last timed step returned to its caller (pick, pick_score, tie_count) as DIR/<name>.npy
           in float64 (DIR/<name>_rank<r>.npy per rank on N > 1); the inputs are seeded, so two builds run with the same
           arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests.helpers import synth_prompts, synth_snapshot, zipf_adapters  # noqa: E402  (seeded workload generators)

R_PER_GPU = 65536
M = 1024
A = 64
PROMPT_LEN = 2048
BLOCK_CHARS = 64
MAX_BLOCKS = 256
BLOCKS = PROMPT_LEN // BLOCK_CHARS
SCORERS = [("queue", 2.0), ("kv", 2.0), ("prefix", 3.0), ("lora", 1.0)]
NSETS = 4  # rotating input sets: 4 x 128 MiB of prompts > 126 MB L2, so no step re-reads L2-resident inputs
METRIC = "endpoint picks/sec at 64K reqs x 1024 endpoints"
WORKLOAD = "headline: 64K requests/GPU x 1024 endpoints, queue+kv+prefix+lora, 2KB prompts (150 shared-prefix groups), B=32 blocks"


def set_workload(name: str, world: int):
    """BASELINE.json configs: 'headline' (the metric's config, per GPU) or 'E' (1M x 4096 sharded over the GPUs)."""
    global R_PER_GPU, M, NSETS, METRIC, WORKLOAD
    if name == "E":
        M = 4096
        R_PER_GPU = 1048576 // world
        NSETS = 2
        METRIC = "endpoint picks/sec at 1M reqs x 4096 endpoints (request-sharded)"
        WORKLOAD = (f"config E: 1M requests x 4096 endpoints sharded over {world} GPU(s) ({R_PER_GPU} per GPU), "
                    "queue+kv+prefix+lora, 2KB prompts (150 shared-prefix groups), B=32 blocks")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def config_dict(n_gpus):
    return {"workload": WORKLOAD, "requests_per_gpu": R_PER_GPU, "endpoints": M, "adapters": A,
            "prompt_bytes": PROMPT_LEN, "block_chars": BLOCK_CHARS, "scorers": "queue:2,kv:2,prefix:3,lora:1",
            "picker": "max-score (lowest-index tie-break)", "parallelism": f"request-sharded x{n_gpus}",
            "l2": f"inputs rotate over {NSETS} x {R_PER_GPU * PROMPT_LEN >> 20}MiB prompt sets (> L2); prefix table + snapshot steady-state resident"}


# ------------------------------------------------------------------------------------------------
# workload (identical on the GPU arm and the CPU arm)
# ------------------------------------------------------------------------------------------------
def build_workload(rank: int, nsets: int, R: int):
    snap = synth_snapshot(M, A=A, seed=0)
    sets = []
    for s in range(nsets):
        prompts, off, _ = synth_prompts(R, prompt_len=PROMPT_LEN, groups=150, shared=1024, seed=100 * rank + s, prefix_seed=7)
        sets.append(dict(prompts=prompts, off=off, adapters=zipf_adapters(R, A=A, seed=100 * rank + s)))
    return snap, sets


def oracle_setup(snap):
    """CPU oracle objects + the warm prefix index (4*M earlier requests routed and committed)."""
    from oracle import oracle_py as o
    osnap = o.SnapshotData(**snap)
    prof = o.make_profile([({"queue": 0, "kv": 1, "prefix": 2, "lora": 3}[k], w) for k, w in SCORERS])
    idx = o.Index()
    seed = o.model_seed("bench-model")
    wp, woff, _ = synth_prompts(4 * M, prompt_len=PROMPT_LEN, groups=150, shared=1024, seed=4242, prefix_seed=7)
    nthreads = os.cpu_count() or 1
    warm = o.schedule_batch(osnap, prof, idx, 4 * M, prompt_bytes=wp, prompt_off=woff,
                            model_seed=np.full(4 * M, seed, np.uint64), adapter_id=zipf_adapters(4 * M, A=A, seed=4242),
                            block_chars=BLOCK_CHARS, max_blocks=MAX_BLOCKS, want_hashes=True, n_threads=nthreads)
    idx.commit(warm["pick"], warm["hashes_out"], warm["total_blocks"])
    return o, osnap, prof, idx, seed, warm


def oracle_batch(o, osnap, prof, idx, seed, wset, n, n_threads=None, base=0, **kw):
    return o.schedule_batch(osnap, prof, idx, n, prompt_bytes=wset["prompts"][: wset["off"][n]], prompt_off=wset["off"][: n + 1],
                            model_seed=np.full(n, seed, np.uint64), adapter_id=wset["adapters"][:n], block_chars=BLOCK_CHARS,
                            max_blocks=MAX_BLOCKS, n_threads=n_threads or os.cpu_count() or 1, request_base=base, **kw)


def time_oracle(o, osnap, prof, idx, seed, wset, R, n_threads, min_seconds=2.0, max_iters=20):
    times = []
    t_all = time.perf_counter()
    while True:
        t0 = time.perf_counter()
        oracle_batch(o, osnap, prof, idx, seed, wset, R, n_threads)
        times.append(time.perf_counter() - t0)
        if len(times) >= max_iters or (time.perf_counter() - t_all) > min_seconds and len(times) >= 3:
            break
    return float(np.median(times)), len(times)


def dump_outputs(path, arrays):
    """--dump-outputs: one float64 .npy per array (int32 picks and tie counts are exact in float64)."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def host_cpus():
    """What the box really offers the CPU arm: logical CPUs, the affinity mask and the cgroup CPU quota (a container may see
    128 CPUs and be allowed ten of them)."""
    info = {"logical": os.cpu_count() or 1}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        pass
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:  # noqa: BLE001
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:  # noqa: BLE001
            pass
    info["cgroup_quota_cpus"] = quota
    return info


def best_thread_count(step, R, cores):
    """The CPU arm gets the thread count that serves IT best: every count in {cores, cores/2, cores/4, 32, 16, 8} (deduplicated,
    <= cores) runs one quarter-size step after a warm-up; returns (best count, {count: picks/s})."""
    n = max(2048, R // 4)
    cands = sorted({c for c in (cores, cores // 2, cores // 4, 32, 16, 8) if 1 <= c <= cores}, reverse=True)
    t_warm = time.perf_counter()
    while time.perf_counter() - t_warm < 2.0:   # first-touch / thread start-up transients (about a second) must not pick the count
        step(cores, n)
    rates = {}
    for c in cands:
        best = 0.0
        for _ in range(3):
            t0 = time.perf_counter()
            step(c, n)
            best = max(best, n / (time.perf_counter() - t0))
        rates[c] = best
    best = max(rates, key=rates.get)
    return best, {str(k): round(v) for k, v in rates.items()}


# ------------------------------------------------------------------------------------------------
# --impl reference : the CPU port of the reference path on the host cores
# ------------------------------------------------------------------------------------------------
def run_reference(args):
    """The CPU arm on the SAME configuration as the GPU arm (R requests per step, same generator, same scorers):
    oracle/oracle.c on every host thread through its persistent worker pool; `value` = R / median step time."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    R = min(R_PER_GPU, 65536)  # (config E: a 64K sample of the shard keeps the arm within minutes; stated in `sample`)
    snap, sets = build_workload(0, 1, R)
    o, osnap, prof, idx, seed, _ = oracle_setup(snap)
    cores = os.cpu_count() or 1

    def step(threads=cores, n=R):
        return oracle_batch(o, osnap, prof, idx, seed, sets[0], n, threads)

    threads, tried = best_thread_count(step, R, cores)
    for _ in range(args.warmup):
        step(threads)
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        res = step(threads)
        times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: res[k] for k in ("pick", "pick_score", "tie_count")})
    med = float(np.median(times))
    value = R / med
    n1 = 4096
    t0 = time.perf_counter()
    step(1, n1)
    single = n1 / (time.perf_counter() - t0)
    sample = (f"{R} requests x {M} endpoints per step (the GPU arm's batch, same generator), {threads} threads of {cores} logical CPUs "
              f"(the fastest of the counts tried), persistent pool")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "picks/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * med, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_dict(args.gpus),
            "cpu_baseline": {"value": value, "unit": "picks/s", "cores": threads, "kind": "port", "sample": sample,
                             "single_thread_value": single, "threads_tried_picks_per_s": tried, "host_cpus": host_cpus()},
            "e2e": {"value": value, "unit": "picks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "timing": {"statistic": "median of the timed steps", "mean_ms_per_step": 1e3 * float(np.mean(times)),
                       "min_ms_per_step": 1e3 * float(np.min(times)), "max_ms_per_step": 1e3 * float(np.max(times))},
            "note": "CPU port (oracle/oracle.c) of the Go reference path; no Go toolchain in this image, so oracle/_ref does not exist"}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# clocks sampling during the timed region (NVML)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                 0x80: "hw_power_brake_slowdown"}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, n in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv:
            self._stop.clear()
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr:
            self._stop.set()
            self._thr.join()
            self._thr = None

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
def run_gpu(args):
    import faulthandler
    faulthandler.dump_traceback_later(1500, exit=True)  # never hang a GPU box: dump and die instead
    import torch
    import torch.distributed as dist

    import _pkg
    pkg = _pkg.load()   # the library __graft_entry__.build() made; bench.py compiles nothing and writes nothing in the tree
    import importlib
    sharding = importlib.import_module(_pkg.NAME + ".sharding")   # the multi-GPU host helpers (commit-stream exchange)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    R = R_PER_GPU
    full = args.workload == "headline" and not args.quick   # the side legs (per-kernel timing, §8f profiles, CPU baselines)
    snap, sets = build_workload(rank, NSETS, R)

    def make_engine(scorers=SCORERS, **kw):
        kw.setdefault("prefix_capacity", 1 << 19)
        return pkg.Engine(pkg.default_config(scorers, max_endpoints=M, max_adapters=A, block_chars=BLOCK_CHARS,
                                             max_blocks=MAX_BLOCKS, **kw), device=local)

    eng = make_engine()
    if args.dev_split is not None:
        eng.set_debug(5, args.dev_split)
    if args.dev_streams is not None:
        eng.set_debug(6, args.dev_streams)
    stream = torch.cuda.Stream(device=dev)  # an explicit stream: events and every launch below share it
    torch.cuda.set_stream(stream)
    sptr = stream.cuda_stream
    RMAX, RMIN = (dist.ReduceOp.MAX, dist.ReduceOp.MIN)

    def allreduce(x, op):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=op)
        return float(t.item())

    # ---- endpoint snapshot: built on rank 0, ONE NCCL broadcast of the packed tile over NVLink ----
    order = ["kv_usage", "queue", "running", "lora_active", "lora_waiting", "lora_nmodels", "lora_max"]

    def pack(sn):
        return np.concatenate([np.ascontiguousarray(sn[k]).view(np.uint8).reshape(-1) for k in order])

    packed = pack(snap)
    tpack = torch.from_numpy(packed).to(dev) if rank == 0 else torch.empty(len(packed), dtype=torch.uint8, device=dev)
    if world > 1:
        dist.broadcast(tpack, src=0)

    def views_of(t):
        v, o_ = {}, 0
        for k in order:
            v[k] = t.data_ptr() + o_
            o_ += np.ascontiguousarray(snap[k]).nbytes
        return v

    views = views_of(tpack)
    torch.cuda.synchronize()
    side = torch.cuda.Stream(device=dev)  # snapshot preparation runs here, concurrently with the prompt hashing

    def apply_snapshot(e, on=None, v=None):
        # device-resident snapshot, used in place: 2 kernels (prepare_endpoints, prepare_adapters)
        v = v or views
        e.set_snapshot(v["kv_usage"], v["queue"], v["running"], v["lora_active"], v["lora_waiting"], v["lora_nmodels"], v["lora_max"],
                       device=True, stream=(on or sptr), M=M, lora_words=1)

    apply_snapshot(eng)

    # ---- prefix index: 4*M earlier requests are routed by the oracle; the resulting COMMIT STREAM (picks + block hashes)
    #      is broadcast from rank 0 with NCCL and every rank replays it through eppscore_commit_picks_device — the index is a
    #      deterministic function of the ordered commits, so all replicas are identical (SURVEY §8e).  Every rank also
    #      builds its own oracle (same seeds) so that EVERY rank's results are parity-checked, not only rank 0's. ----
    o, osnap, prof, idx, seed, warm = oracle_setup(snap)
    W = 4 * M
    if rank == 0:
        w_pick = torch.from_numpy(warm["pick"]).to(dev)
        w_hash = torch.from_numpy(np.ascontiguousarray(warm["hashes_out"]).view(np.int64)).to(dev)
        w_nh = torch.from_numpy(warm["total_blocks"].astype(np.int16)).to(dev)
    else:
        w_pick = torch.empty(W, dtype=torch.int32, device=dev)
        w_hash = torch.empty((W, MAX_BLOCKS), dtype=torch.int64, device=dev)
        w_nh = torch.empty(W, dtype=torch.int16, device=dev)
    if world > 1:
        for t in (w_pick, w_hash, w_nh):
            dist.broadcast(t.view(torch.uint8), src=0)  # (NCCL has no int16: ship the bytes)
    if not np.array_equal(w_pick.cpu().numpy(), warm["pick"]):
        raise SystemExit(f"bench: rank {rank}: the broadcast commit stream differs from this rank's oracle")
    torch.cuda.synchronize()
    t_commit = time.perf_counter()
    eng.commit_picks_device(w_pick, w_hash, w_nh, touch_bound=W * BLOCKS, stream=sptr)
    torch.cuda.synchronize()
    t_commit = time.perf_counter() - t_commit  # includes the one-time allocation of the per-endpoint LRU regions

    # ---- device-resident inputs ----
    dsets = []
    for s in sets:
        dsets.append(dict(prompts=torch.from_numpy(s["prompts"]).to(dev), off=torch.from_numpy(s["off"]).to(dev),
                          seeds=torch.from_numpy(np.full(R, seed, np.uint64).view(np.int64)).to(dev),
                          adapters=torch.from_numpy(s["adapters"]).to(dev)))
    out = dict(pick=torch.empty(R, dtype=torch.int32, device=dev), pick_score=torch.empty(R, dtype=torch.float64, device=dev),
               tie_count=torch.empty(R, dtype=torch.int32, device=dev))

    def raw_step(i, e=None, outs=None):
        """One full pass of the hot path from raw inputs: snapshot preparation + prompt hashing + score/pick."""
        e = e or eng
        d = dsets[i % NSETS]
        side.wait_stream(stream)                    # fork: the snapshot does not depend on the prompts ...
        apply_snapshot(e, side.cuda_stream)         # ... so it is prepared on a second stream while the batch is hashed;
        e.schedule(R, prompt_bytes=d["prompts"], prompt_off=d["off"], model_seed=d["seeds"], adapter_id=d["adapters"],
                   request_base=rank * R, device=True, stream=sptr, out=outs or out)

    def barrier():
        if world > 1:
            dist.barrier()

    def check_parity(set_index, n, what):
        want = oracle_batch(o, osnap, prof, idx, seed, sets[set_index], n, base=rank * R)
        ok = (np.array_equal(out["pick"][:n].cpu().numpy(), want["pick"]) and
              np.array_equal(out["pick_score"][:n].cpu().numpy(), want["pick_score"]) and
              np.array_equal(out["tie_count"][:n].cpu().numpy(), want["tie_count"]))
        if allreduce(1.0 if ok else 0.0, RMIN) < 1.0:
            raise SystemExit(f"bench: rank {rank}: GPU picks differ from the oracle ({what}) — refusing to report a number"
                             if not ok else f"bench: another rank failed the parity check ({what})")

    # ---- parity spot check against the oracle on EVERY rank before any timing ----
    l0 = eng.stats().kernel_launches
    raw_step(0)
    torch.cuda.synchronize()
    launches_per_step = int(eng.stats().kernel_launches - l0)
    check_parity(0, 4096, "before timing")

    # ---- capture one CUDA graph per input set (the step is launch-bound from Python otherwise) ----
    def make_graphs(fn, n=NSETS):
        gs = []
        for i in range(n):
            fn(i)  # warm: all scratch buffers allocated before capture
        torch.cuda.synchronize()
        for i in range(n):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                fn(i)
            gs.append(g)
        return gs

    use_graph = True
    try:
        graphs = make_graphs(raw_step)
    except Exception as ex:  # noqa: BLE001
        sys.stderr.write(f"[bench] CUDA graph capture unavailable ({ex}); timing direct launches\n")
        use_graph = False
        torch.cuda.synchronize()

    def step(i):
        if use_graph:
            graphs[i % NSETS].replay()
        else:
            raw_step(i)

    # ---- value: K steps, device-resident, CUDA events on the launch stream, max over ranks ----
    for i in range(args.warmup):
        step(i)
    clocks = ClockSampler(local)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.synchronize()
    clocks.start()
    e0.record(stream)
    for i in range(args.steps):
        step(args.warmup + i)
    e1.record(stream)
    torch.cuda.synchronize()
    clocks.stop()
    barrier()
    ms_max = allreduce(e0.elapsed_time(e1), RMAX)
    value = world * R * args.steps / (ms_max * 1e-3)
    if args.dump_outputs:
        sfx = f"_rank{rank}" if world > 1 else ""
        dump_outputs(args.dump_outputs, {k + sfx: v.cpu().numpy() for k, v in out.items()})
    # the timed steps must still produce oracle-exact picks on every rank (last step used set (warmup+steps-1)%NSETS)
    check_parity((args.warmup + args.steps - 1) % NSETS, 2048, "timed region")

    # ---- e2e: the same work through the host-buffer C-ABI calls (pinned host memory) ----
    hsnap = {k: torch.from_numpy(np.ascontiguousarray(snap[k]).reshape(-1).view(np.int64 if snap[k].dtype == np.uint64 else snap[k].dtype)).pin_memory()
             for k in order}

    def host_snapshot():
        eng.set_snapshot(hsnap["kv_usage"].numpy(), hsnap["queue"].numpy(), hsnap["running"].numpy(),
                         hsnap["lora_active"].numpy().view(np.uint64), hsnap["lora_waiting"].numpy().view(np.uint64),
                         hsnap["lora_nmodels"].numpy(), hsnap["lora_max"].numpy(), M=M, lora_words=1)

    hsets = []
    for s in sets:
        hp = torch.from_numpy(s["prompts"]).pin_memory()
        hs = torch.from_numpy(np.full(R, seed, np.uint64).view(np.int64)).pin_memory()
        ha = torch.from_numpy(s["adapters"]).pin_memory()
        ho = torch.from_numpy(s["off"]).pin_memory()
        hh = torch.empty((R, BLOCKS), dtype=torch.int64).pin_memory()      # host-hash mode: the block hashes ...
        hn = torch.empty(R, dtype=torch.int16).pin_memory()                # ... and their counts, pinned
        hsets.append(dict(prompts=hp.numpy(), off=ho.numpy(), seeds=hs.numpy().view(np.uint64), adapters=ha.numpy(),
                          hashes=hh.numpy().view(np.uint64), nh=hn.numpy().view(np.uint16), keep=(hp, hs, ha, ho, hh, hn)))
    h2d = int(hsets[0]["prompts"].nbytes + hsets[0]["off"].nbytes + hsets[0]["seeds"].nbytes + hsets[0]["adapters"].nbytes + len(packed))
    h2d_hh = int(hsets[0]["hashes"].nbytes + hsets[0]["nh"].nbytes + hsets[0]["adapters"].nbytes + len(packed))
    d2h = R * (4 + 8 + 4)

    def e2e_step(i):
        h = hsets[i % NSETS]
        host_snapshot()
        return eng.schedule(R, prompt_bytes=h["prompts"], prompt_off=h["off"], model_seed=h["seeds"], adapter_id=h["adapters"],
                            request_base=rank * R, want_total=False)

    def e2e_hosthash_step(i):
        # the host hashes the prompts (library worker pool, all cores) and ships 8 bytes per block instead of 64
        h = hsets[i % NSETS]
        host_snapshot()
        pkg.Engine.hash_prompts_host(h["prompts"], h["off"], h["seeds"], block_chars=BLOCK_CHARS, max_blocks=BLOCKS, stride=BLOCKS,
                                     out=(h["hashes"], h["nh"]))
        return eng.schedule(R, hashes_in=h["hashes"], n_hashes_in=h["nh"], hash_stride=BLOCKS, adapter_id=h["adapters"],
                            request_base=rank * R, want_total=False)

    def time_host(fn, nsteps):
        for i in range(3):
            fn(i)
        lat = []
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = None
        for i in range(nsteps):
            t1 = time.perf_counter()
            res = fn(3 + i)
            lat.append(time.perf_counter() - t1)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        barrier()
        dt = allreduce(dt, RMAX)
        return world * R * nsteps / dt, dt / nsteps, lat, res

    e2e_steps = max(5, min(args.steps, 50))
    e2e_value, e2e_dt, lat, res = time_host(e2e_step, e2e_steps)
    n_chk = 2048
    want = oracle_batch(o, osnap, prof, idx, seed, sets[(3 + e2e_steps - 1) % NSETS], n_chk, base=rank * R)
    if not (np.array_equal(res["pick"][:n_chk], want["pick"]) and np.array_equal(res["pick_score"][:n_chk], want["pick_score"])):
        raise SystemExit("bench: e2e picks differ from the oracle")
    hh_error = None
    try:
        hh_value, hh_dt, _, res = time_host(e2e_hosthash_step, e2e_steps)
        if not (np.array_equal(res["pick"][:n_chk], want["pick"]) and np.array_equal(res["pick_score"][:n_chk], want["pick_score"])):
            hh_error = "picks differ from the oracle"   # reported in the line (an extra leg must not take the headline down)
    except Exception as ex:  # noqa: BLE001
        hh_value, hh_dt, hh_error = 0.0, 0.0, repr(ex)
    apply_snapshot(eng)

    # ---- closed loop: schedule -> PreRequest commit -> schedule ..., the commit inside the timed region.  The snapshot
    #      changes every batch (as the metrics refresh would), all shards' commits are all-gathered and replayed by every rank
    #      in global request order, so the replicated index stays identical on all GPUs. ----
    closed = None
    try:
        KL = 4
        loop_snaps = [synth_snapshot(M, A=A, seed=500 + k) for k in range(KL)]
        loop_tiles = [torch.from_numpy(pack(sn)).to(dev) for sn in loop_snaps]
        loop_views = [views_of(t) for t in loop_tiles]

        def loop_warm():
            """The index the loop starts from: the same 4*M earlier requests, but routed in 8 sub-batches under 8 different
            snapshots with a commit after each (a history under changing load: the shared prefixes end up spread over many
            endpoints instead of the dozen that win under one static snapshot).  Returns the oracle index + the commit stream."""
            from oracle import oracle_py as oo
            ix = oo.Index()
            wp, woff, _ = synth_prompts(W, prompt_len=PROMPT_LEN, groups=150, shared=1024, seed=4242, prefix_seed=7)
            wa = zipf_adapters(W, A=A, seed=4242)
            picks, hashes, nhs = [], [], []
            nb = 8
            per = W // nb
            for b in range(nb):
                sn = oo.SnapshotData(**synth_snapshot(M, A=A, seed=900 + b))
                lo_, hi_ = b * per, (b + 1) * per
                ws = dict(prompts=wp[lo_ * PROMPT_LEN: hi_ * PROMPT_LEN], off=woff[: per + 1], adapters=wa[lo_:hi_])
                w = oracle_batch(oo, sn, prof, ix, seed, ws, per, want_hashes=True)
                ix.commit(w["pick"], w["hashes_out"], w["total_blocks"])
                picks.append(w["pick"])
                hashes.append(w["hashes_out"])
                nhs.append(w["total_blocks"])
            return ix, np.concatenate(picks), np.concatenate(hashes), np.concatenate(nhs)

        idx_l, lw_pick, lw_hash, lw_nh = loop_warm()
        lw = (torch.from_numpy(lw_pick).to(dev), torch.from_numpy(np.ascontiguousarray(lw_hash).view(np.int64)).to(dev),
              torch.from_numpy(lw_nh.astype(np.int16)).to(dev))
        outc = dict(pick=torch.empty(R, dtype=torch.int32, device=dev), pick_score=torch.empty(R, dtype=torch.float64, device=dev),
                    tie_count=torch.empty(R, dtype=torch.int32, device=dev), total_blocks=torch.empty(R, dtype=torch.int16, device=dev),
                    hashes_out=torch.zeros((R, MAX_BLOCKS), dtype=torch.int64, device=dev))
        if world > 1:
            g_pick = torch.empty(world * R, dtype=torch.int32, device=dev)
            g_nh = torch.empty(world * R, dtype=torch.int16, device=dev)
            g_hash = torch.empty((world * R, MAX_BLOCKS), dtype=torch.int64, device=dev)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4 * KL + 1)]

        def loop_batch(k, e, timed):
            d = dsets[k % NSETS]
            apply_snapshot(e, None, loop_views[k % KL])
            if timed:
                ev[4 * k].record(stream)
            e.schedule(R, prompt_bytes=d["prompts"], prompt_off=d["off"], model_seed=d["seeds"], adapter_id=d["adapters"],
                       request_base=(k * world + rank) * R, device=True, stream=sptr, out=outc)
            if timed:
                ev[4 * k + 1].record(stream)
            if world > 1:  # the shards' commits, concatenated in rank order == global request order
                cp, cn, ch = sharding.gather_commit_stream(dist, outc["pick"], outc["total_blocks"], outc["hashes_out"], g_pick, g_nh, g_hash)
            else:
                cp, ch, cn = outc["pick"], outc["hashes_out"], outc["total_blocks"]
            if timed:
                ev[4 * k + 2].record(stream)
            e.commit_picks_device(cp, ch, cn, touch_bound=world * R * BLOCKS, stream=sptr)
            if timed:
                ev[4 * k + 3].record(stream)

        eng_c = make_engine()
        eng_c.commit_picks_device(*lw, touch_bound=W * BLOCKS, stream=sptr)
        loop_batch(0, eng_c, False)  # warm-up: allocations, NCCL channels
        torch.cuda.synchronize()
        eng_c.close()
        eng_c = make_engine()
        eng_c.commit_picks_device(*lw, touch_bound=W * BLOCKS, stream=sptr)
        barrier()
        torch.cuda.synchronize()
        for k in range(KL):
            loop_batch(k, eng_c, True)
        ev[4 * KL].record(stream)
        torch.cuda.synchronize()
        barrier()
        t_loop = allreduce(ev[0].elapsed_time(ev[4 * KL]), RMAX) * 1e-3
        t_sched = sum(ev[4 * k].elapsed_time(ev[4 * k + 1]) for k in range(KL)) * 1e-3
        t_gather = sum(ev[4 * k + 1].elapsed_time(ev[4 * k + 2]) for k in range(KL)) * 1e-3
        t_com = sum(ev[4 * k + 2].elapsed_time(ev[4 * k + 3]) for k in range(KL)) * 1e-3
        st = eng_c.stats()
        closed = {"batches": KL, "requests_per_batch": world * R, "picks_per_s": world * R * KL / t_loop, "ms_per_batch": 1e3 * t_loop / KL,
                  "schedule_ms": 1e3 * t_sched / KL, "allgather_ms": 1e3 * t_gather / KL, "commit_ms": 1e3 * t_com / KL,
                  "commit_requests_per_s": world * R * KL / t_com if t_com > 0 else None,
                  "collective": "3 x ncclAllGather (picks 4 B, counts 2 B, block hashes 8 B x 256 per request)" if world > 1 else "none (1 GPU)",
                  "collective_share": t_gather / t_loop,
                  "index": {"live_hashes": int(st.prefix_live_hashes), "slots_used": int(st.prefix_hashes), "lru_entries": int(st.lru_entries),
                            "rebuilds": int(st.prefix_rebuilds), "overflow_rows": int(st.prefix_overflow_rows), "error": int(st.index_error)}}
        # replicas must agree: every rank holds the same index
        sig = float(st.prefix_live_hashes * 1000003 + st.lru_entries)
        if allreduce(sig, RMAX) != allreduce(sig, RMIN):
            raise SystemExit("bench: closed loop: the ranks' index replicas diverged")
        closed["replicas_identical"] = True
        closed["distinct_endpoints_picked_last_batch"] = int(torch.unique(outc["pick"]).numel())
        closed["workload"] = ("64K requests per GPU per batch, a fresh snapshot every batch; the index starts from 4*M earlier requests routed in 8 "
                              "sub-batches under 8 snapshots (prefixes spread over many endpoints)")
        if world <= 2 and full:
            # parity of the whole loop against the oracle (scheduler + indexer): last batch's picks of this rank's shard,
            # LRU contents of a sample of endpoints, len(hashToPods)
            o2, prof2, idx2, seed2 = o, prof, idx_l, seed
            t_cpu = time.perf_counter()
            last = None
            for k in range(KL):
                osk = o2.SnapshotData(**loop_snaps[k % KL])
                ws = []
                for rk in range(world):
                    if rk == rank:
                        wsk = sets[k % NSETS]
                    else:  # the other rank's shard of this batch (same generator, its seeds)
                        pr, of, _ = synth_prompts(R, prompt_len=PROMPT_LEN, groups=150, shared=1024, seed=100 * rk + k % NSETS, prefix_seed=7)
                        wsk = dict(prompts=pr, off=of, adapters=zipf_adapters(R, A=A, seed=100 * rk + k % NSETS))
                    ws.append(oracle_batch(o2, osk, prof2, idx2, seed2, wsk, R, base=(k * world + rk) * R, want_hashes=True))
                for rk in range(world):
                    idx2.commit(ws[rk]["pick"], ws[rk]["hashes_out"], ws[rk]["total_blocks"])
                last = ws[rank]
            t_cpu = time.perf_counter() - t_cpu
            ok = np.array_equal(outc["pick"].cpu().numpy(), last["pick"]) and np.array_equal(outc["pick_score"].cpu().numpy(), last["pick_score"])
            ok = ok and int(st.prefix_live_hashes) == idx2.num_hashes()
            for m in list(range(0, M, 97)) + [int(x) for x in np.unique(last["pick"])[:8]]:
                ok = ok and eng_c.prefix_lru_keys(m) == idx2.lru_keys(m)
            closed["parity_vs_oracle"] = {"bit_exact": bool(ok), "checked": "picks + scores of the last batch (this rank's shard), LRU keys "
                                          "oldest->newest of 19 endpoints, len(hashToPods)"}
            closed["cpu_port"] = {"picks_per_s": world * R * KL / t_cpu, "cores": os.cpu_count(),
                                  "note": "oracle schedule (all threads) + indexer.Add in request order (one thread, like the reference's indexer.mu)"}
            if not ok:
                raise SystemExit("bench: closed loop differs from the oracle")
        eng_c.close()
    except SystemExit:
        raise
    except Exception as ex:  # noqa: BLE001
        closed = {"error": repr(ex)}

    # ---- strong scaling beside the weak curve: a FIXED batch of 64K requests split over the N GPUs ----
    strong = None
    try:
        Rs = 65536 // world
        sp, so, _ = synth_prompts(65536, prompt_len=PROMPT_LEN, groups=150, shared=1024, seed=999, prefix_seed=7)
        sa = zipf_adapters(65536, A=A, seed=999)
        lo = rank * Rs
        dp = torch.from_numpy(sp[lo * PROMPT_LEN:(lo + Rs) * PROMPT_LEN]).to(dev)
        do = torch.from_numpy(so[: Rs + 1]).to(dev)
        da = torch.from_numpy(sa[lo: lo + Rs]).to(dev)
        ds = torch.from_numpy(np.full(Rs, seed, np.uint64).view(np.int64)).to(dev)
        outs = dict(pick=torch.empty(Rs, dtype=torch.int32, device=dev), pick_score=torch.empty(Rs, dtype=torch.float64, device=dev),
                    tie_count=torch.empty(Rs, dtype=torch.int32, device=dev))

        def strong_step(i):
            side.wait_stream(stream)
            apply_snapshot(eng, side.cuda_stream)
            eng.schedule(Rs, prompt_bytes=dp, prompt_off=do, model_seed=ds, adapter_id=da, request_base=lo, device=True, stream=sptr, out=outs)

        sg = make_graphs(strong_step, 1)[0]
        for _ in range(5):
            sg.replay()
        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        torch.cuda.synchronize()
        a_.record(stream)
        for _ in range(50):
            sg.replay()
        b_.record(stream)
        torch.cuda.synchronize()
        t_s = allreduce(a_.elapsed_time(b_), RMAX) / 50 * 1e-3
        strong = {"total_requests": 65536, "requests_per_gpu": Rs, "us_per_step": t_s * 1e6, "picks_per_s": 65536 / t_s,
                  "note": "fixed 64K-request batch split by request over the GPUs (the same inputs every step: L2-resident at this size); "
                          "no collective on the data path"}
    except Exception as ex:  # noqa: BLE001
        strong = {"error": repr(ex)}

    extra = {}
    if rank == 0:
        extra["closed_loop"] = closed
        extra["strong_scaling"] = strong
        extra["commit_picks"] = {"requests": W, "hashes_per_request": BLOCKS, "seconds": t_commit,
                                 "note": "warm-up replay through eppscore_commit_picks_device, incl. the one-time allocation of the LRU regions"}
        extra["e2e_host_hash"] = {"value": hh_value, "unit": "picks/s", "h2d_bytes_per_step": h2d_hh, "d2h_bytes_per_step": d2h,
                                  "ms_per_step": 1e3 * hh_dt, "host_threads": os.cpu_count(),
                                  "note": "prompts hashed on the host cores (eppscore_hash_prompts_host) inside the timed region; "
                                          "hashes_in crosses PCIe instead of the prompt bytes; "
                                          + ("picks bit-equal" if hh_error is None else "FAILED: " + hh_error)}
        if hh_error is not None:
            extra["e2e_host_hash"]["error"] = hh_error
    if rank == 0 and full:
        peak, peak_src = peaks()
        traffic = {}
        tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                traffic = json.load(f)

        def time_kernel(fn, iters=40, graph=True):
            """CUDA-event time per call of fn(i); fn is captured into one CUDA graph per input set so that the host's launch
            rate cannot be what is measured."""
            gs = None
            if graph:
                try:
                    gs = make_graphs(fn)
                except Exception:  # noqa: BLE001
                    gs = None
                    torch.cuda.synchronize()
            call = (lambda i: gs[i % NSETS].replay()) if gs else fn
            for i in range(5):
                call(i)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record(stream)
            for i in range(iters):
                call(5 + i)
            b.record(stream)
            torch.cuda.synchronize()
            return a.elapsed_time(b) / iters * 1e-3

        # ---- per-kernel timing (each stage alone, rotating inputs) ----
        L = pkg.lib()
        hsets_dev = [(torch.zeros((R, MAX_BLOCKS), dtype=torch.uint64, device=dev), torch.zeros(R, dtype=torch.uint16, device=dev))
                     for _ in range(NSETS)]

        def hash_only(i):
            d = dsets[i % NSETS]
            hh, nn = hsets_dev[i % NSETS]
            rc = L.eppscore_hash_prompts(eng._h, R, 1, d["prompts"].data_ptr(), d["off"].data_ptr(), None, d["seeds"].data_ptr(),
                                         BLOCK_CHARS, MAX_BLOCKS, hh.data_ptr(), nn.data_ptr(), sptr)
            assert rc == 0

        def pick_only(i, e=None):
            hh, nn = hsets_dev[i % NSETS]
            (e or eng).schedule(R, hashes_in=hh, n_hashes_in=nn, hash_stride=MAX_BLOCKS, adapter_id=dsets[i % NSETS]["adapters"],
                                request_base=rank * R, device=True, stream=sptr, out=out)

        t_hash = time_kernel(hash_only)         # hash_bodies + hash_chain
        eng.set_debug(2, 1)                     # diagnostics knob: body kernel only
        t_bodies = time_kernel(hash_only)
        eng.set_debug(2, 18)                    # chain kernel only (re-chains the buffer in place: same work)
        t_chain = time_kernel(hash_only)
        eng.set_debug(2, 2)                     # the warp-tile form of the chain kernel
        t_chain_w = time_kernel(hash_only)
        eng.set_debug(2, 8)                     # experimental: the warp-tile fused kernel
        t_wfused = time_kernel(hash_only)
        eng.set_debug(2, 4)                     # experimental: the CTA-tile (warp-specialised) fused kernel
        t_cta = time_kernel(hash_only)
        eng.set_debug(2, 19)
        for i in range(NSETS):                  # real hashes for the pick-only timing below
            hash_only(i)
        torch.cuda.synchronize()
        t_pick = time_kernel(pick_only)
        t_prep = time_kernel(lambda i: apply_snapshot(eng))
        nhv = hsets_dev[0][1].cpu().numpy().astype(np.int64)
        B = float(nhv.mean())
        res_m = eng.schedule(4096, prompt_bytes=sets[0]["prompts"][: sets[0]["off"][4096]], prompt_off=sets[0]["off"][:4097],
                             model_seed=np.full(4096, seed, np.uint64), want_match=True)
        hits = float(res_m["match_blocks"].max(axis=1).mean())
        exc = float((res_m["match_blocks"] > 0).sum(axis=1).mean())
        # algorithmic bytes per launch (DESIGN.md §5): only the probes that are ISSUED are charged — the walk stops at the first
        # miss, so a request reads `hits` slots that hit + 1 that misses, 32 bytes each (the endpoint set travels with the slot)
        plen = float(sets[0]["off"][R])
        bytes_bodies = plen + R * 16 + R * B * 8                              # prompts + offsets in, body states out
        bytes_chain = R * (2 * B * 8 + 8 + 16 + 2)                            # body states in, hashes out, seed, offsets, count
        bytes_pick = R * ((hits + 1) * 8 + (hits + 1) * 32 + 2 + 4 + 16 + 16)   # hashes read, slots probed, count, adapter, summary, outputs
        bytes_prep = M * (8 + 8 + 8 + 8 + 8 + 4 + 4) + M * 8 * 3 + (A + 1) * (3 * M // 8 + 16)
        kern = {"hash_bodies_kernel": (t_bodies, bytes_bodies), "hash_chain_kernel": (t_chain, bytes_chain), "pick_sparse_kernel (+ deferred full-matrix pass)": (t_pick, bytes_pick),
                "prepare_snapshot (2 kernels, side stream)": (t_prep, bytes_prep)}
        extra["kernels"] = {k: {"us": t * 1e6, "algorithmic_bytes": b, "gbs": b / t / 1e9, "frac_of_peak": b / t / 1e9 / peak,
                                "traffic": traffic.get(k.split(" ")[0])}
                            for k, (t, b) in kern.items()}
        extra["kernels"]["hash stage"] = {"bodies_plus_chain_us": t_hash * 1e6, "chain_warp_tile_form_us": t_chain_w * 1e6,
                                          "experimental_single_kernel_forms_us": {"warp_tile_fused": t_wfused * 1e6, "cta_tile_fused": t_cta * 1e6},
                                          "note": "fusing the serial chain into the streaming kernel is slower on B200: a warp in its chain phase has no loads in flight"}
        extra["kernels"]["avg_blocks_per_request"] = B
        extra["kernels"]["avg_matched_blocks"] = hits
        extra["kernels"]["avg_endpoints_with_match"] = exc
        dom = max(kern, key=lambda k: kern[k][0] if "prepare" not in k else 0.0)
        t_dom, b_dom = kern[dom]
        tr = traffic.get(dom.split(" ")[0])
        step_bytes = plen + R * (8 + 8 + 4 + 4 + 8 + 4)   # compulsory HBM bytes of a step: prompts, offsets, seeds, adapters in; pick, score, ties out
        extra["roofline"] = {"bound": "hbm", "kernel": dom.split(" ")[0], "achieved": b_dom / t_dom / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": b_dom / t_dom / 1e9 / peak, "traffic": tr, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": b_dom, "us_per_launch": t_dom * 1e6,
                             "share_of_step": t_dom / (t_hash + t_pick),
                             "dram_frac": (tr / t_dom / 1e9 / peak) if tr else None,
                             "step_compulsory_bytes": step_bytes, "step_frac": step_bytes / (ms_max / args.steps * 1e-3) / 1e9 / peak,
                             "traffic_source": "profiles/roofline_traffic.json (ncu --set full capture of this code, dram__bytes_read+write per launch)"}

        # ---- the fully general R x M evaluation (every pair scored; what masks / diagnostics use) ----
        try:
            eng_g = make_engine()
            eng_g.set_debug(1, 1)               # diagnostics knob: always the fully general kernels
            apply_snapshot(eng_g)
            eng_g.commit_picks_device(w_pick, w_hash, w_nh, touch_bound=W * BLOCKS, stream=sptr)
            t_gen = time_kernel(lambda i: pick_only(i, eng_g), iters=10)
            extra["generic_full_matrix"] = {"kernel": "score_matrix_kernel<E,P,L>", "us": t_gen * 1e6, "picks_per_s": R / t_gen,
                                            "pairs_per_s": R * M / t_gen}
            eng_g.close()
        except Exception as ex:  # noqa: BLE001
            extra["generic_full_matrix"] = {"error": str(ex)}

        # ---- candidate masks (the Filter chain's result): every pair scored, per-row queue min/max ----
        try:
            gen = torch.Generator(device=dev)
            gen.manual_seed(5)
            cmask = torch.randint(0, 2 ** 31 - 1, (R, M // 32), generator=gen, device=dev, dtype=torch.int64).to(torch.int32)
            cmask = (cmask ^ (cmask << 1)).contiguous()  # ~50 % of the endpoints are candidates of each request

            def masked_only(i):
                hh, nn = hsets_dev[i % NSETS]
                eng.schedule(R, hashes_in=hh, n_hashes_in=nn, hash_stride=MAX_BLOCKS, adapter_id=dsets[i % NSETS]["adapters"],
                             cand_mask=cmask, request_base=rank * R, device=True, stream=sptr, out=out)

            t_msk = time_kernel(masked_only, iters=10)
            extra["masked_full_matrix"] = {"kernel": "score_matrix_kernel<Q,E,P,L; masked>", "us": t_msk * 1e6, "picks_per_s": R / t_msk,
                                           "pairs_per_s": R * M / t_msk, "candidates_per_request": "~50 % random"}
        except Exception as ex:  # noqa: BLE001
            extra["masked_full_matrix"] = {"error": str(ex)}

        # ---- latency-predictor fold-in (SURVEY §8 f1): the latency-scorer profile of the reference chart —
        #      per (request, endpoint) Bayesian-ridge TTFT/TPOT, headrooms, tier selection, normalised score ----
        try:
            lat_coef = dict(ttft_intercept=12.5, ttft_kv=80.0, ttft_input=0.031, ttft_waiting=7.25, ttft_running=1.5,
                            ttft_prefix=-40.0, tpot_intercept=9.0, tpot_kv=11.0, tpot_input=0.0007, tpot_waiting=0.9,
                            tpot_running=0.35, tpot_generated=0.01, streaming_mode=1)
            eng_l = make_engine([("latency", 1.0)], tie_mode=1, tie_seed=11)
            eng_l.set_latency_params(pkg.latency_params(**lat_coef))
            lrng = np.random.Generator(np.random.PCG64(77))
            lat_ep = dict(min_tpot_slo=lrng.choice([0.0, 0.0, 22.0, 26.5, 60.0], M),
                          dispatched=lrng.integers(0, 3, M).astype(np.int32), prefill_role=(lrng.random(M) < 0.1).astype(np.uint8))
            lat_ep_dev = {k: torch.from_numpy(v).to(dev) for k, v in lat_ep.items()}
            eng_l.set_snapshot(views["kv_usage"], views["queue"], views["running"], device=True, stream=sptr, M=M, lora_words=0,
                               **lat_ep_dev)
            eng_l.commit_picks_device(w_pick, w_hash, w_nh, touch_bound=W * BLOCKS, stream=sptr)
            lat_req = dict(input_tokens=lrng.integers(16, 6000, R).astype(np.int32),
                           ttft_slo=lrng.choice([0.0, 90.0, 140.0, 200.0, 400.0, 1e6], R),
                           tpot_slo=lrng.choice([0.0, 18.0, 24.0, 30.0, 80.0], R))
            lat_req_dev = {k: torch.from_numpy(v).to(dev) for k, v in lat_req.items()}

            def latency_only(i):
                hh, nn = hsets_dev[i % NSETS]
                eng_l.schedule(R, hashes_in=hh, n_hashes_in=nn, hash_stride=MAX_BLOCKS, request_base=rank * R, device=True,
                               stream=sptr, out=out, **lat_req_dev)

            t_lat = time_kernel(latency_only, iters=10)
            extra["latency_fold_in"] = {"kernel": "score_matrix_kernel<T>", "profile": "latency-scorer (weight 1), max-score pick",
                                        "us": t_lat * 1e6, "picks_per_s": R / t_lat, "pairs_per_s": R * M / t_lat,
                                        "predictions_per_s": 2.0 * R * M / t_lat,
                                        "note": "TTFT+TPOT prediction per pair; the reference does one HTTP bulk call of <= 100 rows per request"}
            # parity spot check against the oracle on the first requests of set 0
            n_chk = 512
            latency_only(0)
            torch.cuda.synchronize()
            snap_l = o.SnapshotData(snap["kv_usage"], snap["queue"], snap["running"], **lat_ep)
            prof_l = o.make_profile([(o.SCORER_LATENCY, 1.0)], tie_mode=1, tie_seed=11, latency=o.make_latency_params(**lat_coef))
            hh, nn = hsets_dev[0]
            want_l = o.schedule_batch(snap_l, prof_l, idx, n_chk, hashes_in=hh[:n_chk].cpu().numpy(),
                                      n_hashes_in=nn[:n_chk].cpu().numpy(), max_blocks=MAX_BLOCKS, n_threads=8,
                                      **{k: v[:n_chk] for k, v in lat_req.items()})
            ok = (np.array_equal(out["pick"][:n_chk].cpu().numpy(), want_l["pick"]) and
                  np.array_equal(out["pick_score"][:n_chk].cpu().numpy(), want_l["pick_score"]) and
                  np.array_equal(out["tie_count"][:n_chk].cpu().numpy(), want_l["tie_count"]))
            extra["latency_fold_in"]["parity_vs_oracle"] = {"requests": n_chk, "bit_exact": bool(ok)}
            # the CPU port on the same profile (all host threads), bounded sample
            Rl = 4096
            t0 = time.perf_counter()
            o.schedule_batch(snap_l, prof_l, idx, Rl, hashes_in=hh[:Rl].cpu().numpy(), n_hashes_in=nn[:Rl].cpu().numpy(),
                             max_blocks=MAX_BLOCKS, n_threads=os.cpu_count() or 1, **{k: v[:Rl] for k, v in lat_req.items()})
            extra["latency_fold_in"]["cpu_port_picks_per_s"] = Rl / (time.perf_counter() - t0)
            # the reference chart's whole latency profile on the device: strict affinity filter -> slo-headroom-tier filter ->
            # loose affinity filter -> latency scorer -> weighted-random picker (config/charts/epplib/templates/_config.yaml:66-75)
            try:
                chart_filters = [(pkg.FILTER_PREFIX_AFFINITY, (0.99, 0.01, 5000.0)), (pkg.FILTER_SLO_HEADROOM_TIER, (0.01,)),
                                 (pkg.FILTER_PREFIX_AFFINITY, (0.80, 0.01, 5000.0))]
                eng_ch = make_engine([("latency", 1.0)], filters=chart_filters, pick_mode=pkg.PICK_WEIGHTED_RANDOM, tie_seed=11)
                eng_ch.set_latency_params(pkg.latency_params(**lat_coef))
                eng_ch.set_snapshot(views["kv_usage"], views["queue"], views["running"], device=True, stream=sptr, M=M, lora_words=0,
                                    **lat_ep_dev)
                eng_ch.commit_picks_device(w_pick, w_hash, w_nh, touch_bound=W * BLOCKS, stream=sptr)

                def chart_only(i):
                    hh, nn = hsets_dev[i % NSETS]
                    eng_ch.schedule(R, hashes_in=hh, n_hashes_in=nn, hash_stride=MAX_BLOCKS, request_base=rank * R, device=True,
                                    stream=sptr, out=out, **lat_req_dev)

                t_c = time_kernel(chart_only, iters=6)
                extra["latency_chart_profile"] = {"kernel": "score_matrix_kernel<runtime sequence; LAT; 3 filters; A-Res>",
                                                  "profile": "affinity 0.99 -> slo-headroom-tier -> affinity 0.80 -> latency-scorer -> weighted-random-picker",
                                                  "us": t_c * 1e6, "picks_per_s": R / t_c, "pairs_per_s": R * M / t_c}
                eng_ch.close()
            except Exception as ex:  # noqa: BLE001
                extra["latency_chart_profile"] = {"error": repr(ex)}

            # len(strings.Fields(prompt)) on the device: the prompt stream once more (HBM-bound)
            cnt = torch.empty(R, dtype=torch.int32, device=dev)

            def fields_only(i):
                d = dsets[i % NSETS]
                rc = L.eppscore_count_fields(eng_l._h, R, 1, d["prompts"].data_ptr(), d["off"].data_ptr(), None, cnt.data_ptr(), sptr)
                assert rc == 0

            t_f = time_kernel(fields_only, iters=20)
            plen_f = float(sets[0]["off"][R])
            extra["count_fields"] = {"kernel": "count_fields_kernel", "us": t_f * 1e6, "algorithmic_bytes": plen_f + 12.0 * R,
                                     "gbs": (plen_f + 12.0 * R) / t_f / 1e9, "frac_of_peak": (plen_f + 12.0 * R) / t_f / 1e9 / peak}
            eng_l.close()
        except Exception as ex:  # noqa: BLE001
            extra["latency_fold_in"] = {"error": repr(ex)}

        # ---- stochastic pickers (weighted-random A-Res over the four-scorer profile): every pair scored + one draw per pair ----
        try:
            eng_w = make_engine(pick_mode=pkg.PICK_WEIGHTED_RANDOM, tie_seed=3)
            apply_snapshot(eng_w)
            eng_w.commit_picks_device(w_pick, w_hash, w_nh, touch_bound=W * BLOCKS, stream=sptr)
            t_w = time_kernel(lambda i: pick_only(i, eng_w), iters=10)
            extra["weighted_random_picker"] = {"kernel": "score_matrix_kernel<runtime sequence; A-Res>", "us": t_w * 1e6, "picks_per_s": R / t_w,
                                               "pairs_per_s": R * M / t_w}
            eng_w.close()
        except Exception as ex:  # noqa: BLE001
            extra["weighted_random_picker"] = {"error": repr(ex)}

        # ---- dense-row mode (R x M float4 feature rows streamed from HBM): reported beside the headline, at the metric's 64K ----
        try:
            Rd = R
            feats = []
            for _ in range(2):
                feat = torch.zeros((Rd, M, 4), dtype=torch.float32, device=dev)
                feat[:, :, 0] = (torch.rand((Rd, M), device=dev) < 0.02).float() * 16
                feat[:, :, 1] = torch.randint(0, 4, (Rd, M), device=dev).float()
                feats.append(feat)
            dtot = torch.full((Rd,), 32, dtype=torch.uint16, device=dev)

            def dense_only(i):
                eng.schedule(Rd, dense_feat=feats[i % 2], dense_total=dtot, device=True, stream=sptr, out=out)

            t_dense = time_kernel(dense_only, iters=20, graph=False)
            bytes_dense = 16.0 * Rd * M + 48.0 * M + 16.0 * Rd
            extra["dense_mode"] = {"kernel": "score_dense_fast_kernel<E,P,L>", "requests": Rd, "us": t_dense * 1e6,
                                   "picks_per_s": Rd / t_dense, "algorithmic_bytes": bytes_dense,
                                   "gbs": bytes_dense / t_dense / 1e9, "frac_of_peak": bytes_dense / t_dense / 1e9 / peak,
                                   "traffic": traffic.get("score_dense_fast_kernel"),
                                   "note": "2 x 1 GiB feature sets alternate (> L2)"}
            del feat, feats
        except Exception as ex:  # noqa: BLE001
            extra["dense_mode"] = {"error": str(ex)}
        # ---- R = 1 latency through the host API ----
        one = []
        for i in range(200):
            t1 = time.perf_counter()
            eng.schedule(1, prompt_bytes=hsets[0]["prompts"][:PROMPT_LEN], prompt_off=np.array([0, PROMPT_LEN], np.int64),
                         model_seed=hsets[0]["seeds"][:1], adapter_id=hsets[0]["adapters"][:1], want_total=False)
            one.append(time.perf_counter() - t1)
        extra["latency_ms"] = {"p50_batch_e2e": 1e3 * float(np.median(lat)), "p50_single_request_e2e": 1e3 * float(np.median(one[20:])),
                               "p50_batch_device": ms_max / args.steps}
        # ---- CPU baseline: the oracle port on this box's cores, same workload ----
        if world == 1:
            cores = os.cpu_count() or 1
            Rc = 65536
            try:
                thr_c, tried_c = best_thread_count(lambda c, n: oracle_batch(o, osnap, prof, idx, seed, sets[0], n, c), Rc, cores)
            except Exception as ex:  # noqa: BLE001  (never lose the bench line over the choice of a thread count)
                thr_c, tried_c = cores, {"error": repr(ex)}
            t_mt, n_mt = time_oracle(o, osnap, prof, idx, seed, sets[0], Rc, thr_c)
            t_1, n_1 = time_oracle(o, osnap, prof, idx, seed, sets[0], 4096, 1, min_seconds=1.0, max_iters=5)
            extra["cpu_baseline"] = {"value": Rc / t_mt, "unit": "picks/s", "cores": thr_c, "kind": "port",
                                     "sample": f"{Rc} requests of the same workload x {n_mt} runs (median), {thr_c} threads of {cores} logical CPUs "
                                               f"(the fastest of the counts tried), persistent pool; single-thread: {4096 / t_1:.0f} picks/s",
                                     "single_thread_value": 4096 / t_1, "threads_tried_picks_per_s": tried_c, "host_cpus": host_cpus()}
            # the "Go-shape" restatement (SURVEY §8d form (i)): per-request clones of the candidates, one hash map per
            # scorer, accumulate map, shuffle + stable sort — same results (tests/test_oracle_golden.py), the reference's
            # cost profile.  Labelled Go-shape, not Go: the Go toolchain is not in this image.
            try:
                w0 = sets[0]
                seeds_c = np.full(Rc, seed, np.uint64)

                def goshape(Rg, threads):
                    t0 = time.perf_counter()
                    o.schedule_batch(osnap, prof, idx, Rg, prompt_bytes=w0["prompts"][: w0["off"][Rg]], prompt_off=w0["off"][: Rg + 1],
                                     model_seed=seeds_c[:Rg], adapter_id=w0["adapters"][:Rg], block_chars=BLOCK_CHARS,
                                     max_blocks=MAX_BLOCKS, n_threads=threads, goshape=True, shuffle_seed=1)
                    return time.perf_counter() - t0

                t_g1 = goshape(256, 1)
                Rg = min(Rc, max(cores * 32, 1024))
                t_gm = goshape(Rg, cores)
                # config A of BASELINE.json: 1 request x 4 pods, queue-depth scorer only, per call
                snapA = synth_snapshot(4, A=A, seed=11)
                oA = o.SnapshotData(**snapA)
                profA = o.make_profile([(0, 1.0)])
                nA = 200000
                t0 = time.perf_counter()
                o.schedule_batch(oA, profA, None, nA, n_threads=1, goshape=True)
                t_A = time.perf_counter() - t0
                extra["cpu_baseline_goshape"] = {"value": Rg / t_gm, "unit": "picks/s", "cores": cores, "kind": "port (Go-shape restatement)",
                                                 "sample": f"{Rg} requests of the same workload, {cores} threads; single-thread: {256 / t_g1:.0f} picks/s",
                                                 "single_thread_value": 256 / t_g1,
                                                 "config_A_ns_per_call": 1e9 * t_A / nA,
                                                 "config_A": "1 request x 4 pods, queue-depth scorer only, single thread, 200000 calls"}
            except Exception as ex:  # noqa: BLE001
                extra["cpu_baseline_goshape"] = {"error": repr(ex)}
            # ---- the host layer above the C ABI (C++): BASELINE config A through the product's Scheduler (small-batch host
            # route and forced-GPU route) and per-request latency through the coalescing front vs its window ----
            try:
                import subprocess
                hb = os.path.join(os.path.dirname(os.path.abspath(__file__)), "gateway-api-inference-extension_b200", "host", "host_bench")
                if not getattr(args, "quick", False) and os.path.exists(hb):
                    r = subprocess.run([hb, "64", "200"], capture_output=True, text=True, timeout=180)
                    extra["host_layer"] = json.loads(r.stdout.strip().splitlines()[-1])
                    extra["host_layer"]["note"] = ("C++ host mirror (host/epp_scheduler.hpp, coalescer.hpp) over libeppscore.so; coalescer: 64 "
                                                   "closed-loop caller threads, 256 endpoints, 512-byte prompts, four default scorers")
            except Exception as ex:  # noqa: BLE001
                extra["host_layer"] = {"error": repr(ex)}

    if rank == 0:
        cfg = config_dict(world)
        cfg["step"] = ("prepare_endpoints + prepare_adapters (side stream) || hash_bodies + hash_chain, then pick_sparse + the full-matrix pass over "
                       "deferred requests; snapshot re-prepared every step")
        cfg["cuda_graph"] = use_graph
        line = {"metric": METRIC, "value": value, "unit": "picks/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "config": cfg,
                "e2e": {"value": e2e_value, "unit": "picks/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "steps": e2e_steps, "ms_per_step": 1e3 * e2e_dt, "host_memory": "pinned",
                        "pcie_h2d_gbs": h2d / e2e_dt / 1e9},
                "gpu_launches": int(launches_per_step * args.steps), "clocks": clocks.summary(), "parity_checked": True,
                "parity_checked_ranks": world, "target": {"picks_per_s": 1e8, "met": bool(value >= 1e8)}}
        line.update(extra)
        print(json.dumps(line))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="headline", choices=["headline", "E"])
    ap.add_argument("--dev-split", type=int, default=None, help="experiment: slices per device-resident batch (engine debug key 5)")
    ap.add_argument("--dev-streams", type=int, default=None, help="experiment: streams the slices alternate over (engine debug key 6)")
    ap.add_argument("--quick", action="store_true", help="skip the side legs (per-kernel timing, §8f profiles, CPU baselines)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs (pick, pick_score, tie_count) as DIR/<name>.npy in float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    set_workload(args.workload, int(os.environ.get("WORLD_SIZE", "1")))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
