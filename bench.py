#!/usr/bin/env python
"""bench.py -- offer-scores/sec over the P x G selection grid (+ pods reconciled/sec) on N B200s.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...     # the reference's CPU path (oracle port; Go cannot run here)

One "step" = one pass of the hot path over one batch: the full P x G selection grid (BASELINE config 4:
P = 1M pending pods x G = 100k offers, every (pod, offer) pair evaluated -- no early exit, no class
dedup) and one status sweep over N tracked slots (independent work: it runs on a second stream).  Pod rows and status slots are sharded
contiguously over the ranks (strong scaling: the total is fixed); after the select kernel the per-shard
assignment vector is all-gathered so every GPU holds all P assignments.

`value` = P*G / (max-over-ranks device time per step) with inputs resident in HBM.  `e2e` = the same metric
through the public host C-ABI (`rpk_select` + `rpk_status_diff` on pinned host buffers, one ctx spanning
all N GPUs -- the call a cgo binding makes), H2D and D2H inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "offer-scores/sec (PxG)"
UNIT = "offer-scores/s"
MODEL_BYTES_PER_SCORE = 16  # SURVEY.md 8d streaming model: one (mem, vcpu, ram, price-order) view per score
FALLBACK_HBM_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md fallback


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed region.  NVML is polled in-process every ~2 ms
    (the timed region of this bench is tens of milliseconds, too short for `nvidia-smi -lms`); falls back to
    the profiling recipe's nvidia-smi line when pynvml is unavailable."""

    def __init__(self, dev: int):
        self.dev, self.rows, self.stop_flag, self.t, self.mode = dev, [], False, None, None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.dev]) if vis and vis.split(",")[self.dev].isdigit() else self.dev
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.mode = "nvml"
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
        except Exception:
            self.mode = None

    def _poll(self):
        nv = self.nv
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            try:
                self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM),
                                  nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0, int(get_reasons(self.h))))
            except Exception:
                pass
            time.sleep(0.002)

    def stop(self) -> dict:
        if self.mode != "nvml":
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "NVML unavailable"}
        self.stop_flag = True
        self.t.join(timeout=1)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "no samples"}
        sm = [r[0] for r in self.rows]; mx = [r[1] for r in self.rows]; pw = [r[2] for r in self.rows]
        bits = 0
        for r in self.rows:
            bits |= r[3]
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown"}
        reasons = sorted(n for b_, n in names.items() if bits & b_)
        hi = [s for s, p in zip(sm, pw) if p >= 0.5 * max(pw)] or sm  # samples under load
        return {"sm_mhz": statistics.median(hi), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm),
                "reasons": reasons, "source": "NVML polled every 2 ms from the warm-up steps through the timed region"}


def shard(total, n, r):
    return total * r // n, total * (r + 1) // n


DUMP_MAX_ROWS = 1 << 20  # per array (8 MiB as float64): the six files a dump can hold stay under 64 MiB
DUMP_SEED = 20261017


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy in float64 (every value here is an integer below 2**53, so exact).
    An array longer than DUMP_MAX_ROWS is replaced by a fixed seeded sample of its rows, and the sampled row
    numbers go to <name>_rows.npy: the same output always yields the same files."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a, np.float64)
        if len(a) > DUMP_MAX_ROWS:
            rows = np.sort(np.random.default_rng(DUMP_SEED).choice(len(a), DUMP_MAX_ROWS, replace=False))
            np.save(os.path.join(out_dir, f"{name}_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def host_threads():
    """Host threads the CPU arm may use: the affinity mask, capped by the cgroup CPU quota if one is set (a
    GPU slice of a shared host often sees every core but may run only a share of them)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = max(1, min(n, -(-int(txt[0]) // int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = max(1, min(n, -(-q // per)))
            break
        except Exception:
            continue
    return n


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm on the host cores (oracle port -- the Go toolchain is absent)
# ---------------------------------------------------------------------------------------------------------
def cpu_select_sample(offers, G, seconds, threads, synth, oracle):
    """Time the reference-shaped path (filter -> stable sort by price -> take 5, one GetGPUTypes per pod)
    on a bounded pod sample of the same workload; returns (scores/s, sample description)."""
    n_probe = max(threads * 64, 2048)  # large enough that thread start-up does not dominate the estimate
    probe = synth.make_pods(n_probe, row0=0)
    t0 = time.perf_counter()
    oracle.select(offers, probe, want_top5=True, n_threads=threads)
    dt = max(time.perf_counter() - t0, 1e-4)
    rate = n_probe / dt
    P = int(max(threads * 4, min(rate * seconds * 0.7, 2_000_000)))
    pods = synth.make_pods(P, row0=0)
    t0 = time.perf_counter()
    oracle.select(offers, pods, want_top5=True, n_threads=threads)
    dt = time.perf_counter() - t0
    return P * G / dt, f"{P} pods x {G} offers (rows 0..{P - 1} of the bench table), {dt:.1f} s", P, dt


def run_reference(args, rank, world):
    if rank != 0:
        return
    import importlib

    import oracle

    pkg = importlib.import_module("k8s-runpod-kubelet_b200")
    synth = pkg.synth
    G = args.offers
    threads = host_threads()
    offers = synth.make_offers(G)
    per_step = max(1.0, min(10.0, 120.0 / max(1, args.steps + args.warmup)))
    for _ in range(args.warmup):
        cpu_select_sample(offers, G, per_step / 4, threads, synth, oracle)
    tot_scores, tot_t, desc = 0.0, 0.0, ""
    for _ in range(args.steps):
        v, desc, P, dt = cpu_select_sample(offers, G, per_step, threads, synth, oracle)
        tot_scores += P * G
        tot_t += dt
    value = tot_scores / tot_t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(1, args.steps), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64 prices / int columns", "data": "synthetic",
        "config": {"workload": f"C4: P=1M pods x G={G} offers; each step a bounded sample of pod rows (CPU cannot finish 1M rows)",
                   "sample_per_step": desc},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{args.steps} steps, each {desc}; C restatement of runpod_client.go:465-509 "
                                   "(filter, stable sort by price, take 5) -- Go toolchain absent, reference cannot be compiled"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
# parity: the timed result against the oracle (test infrastructure; outside every timed region)
# ---------------------------------------------------------------------------------------------------------
def compared_fields(recs):
    m = recs.copy()
    m[:, 0] &= 0x7F  # the message flag is neither compared nor hashed
    return m


def check_select_parity(best_np, offers, pods_all, oracle, threads, sample=2000):
    """Every row through the class property (all pods of one (mem, vcpu, ram, max_price, cloud) class share the
    oracle's GetGPUTypes answer: O(classes x G)), plus `sample` rows through oracle.select row by row."""
    P = best_np.shape[0]
    key = np.zeros(P, np.int64)
    radix = 1
    uniq_cols = []
    for name in ("req_mem_gb", "req_vcpu", "req_ram_gb", "max_price", "cloud"):
        u, inv = np.unique(pods_all[name], return_inverse=True)
        uniq_cols.append(u)
        key += inv.reshape(-1).astype(np.int64) * radix
        radix *= len(u)
    classes, inv = np.unique(key, return_inverse=True)
    want_class = np.empty(len(classes), np.int32)
    for ci, k in enumerate(classes):
        vals = []
        for u in uniq_cols:
            vals.append(u[k % len(u)])
            k //= len(u)
        m, v, r, mp, c = vals
        ids = oracle.get_gpu_types(offers, int(m), float(mp), int(c) if int(c) in (0, 1) else 2, int(v), int(r))
        want_class[ci] = ids[0] if ids else -1
    bad_class = int((best_np != want_class[inv.reshape(-1)]).sum())
    rows = np.random.default_rng(20260921).choice(P, min(sample, P), replace=False)
    sub = {k: np.ascontiguousarray(v[rows]) for k, v in pods_all.items()}
    ob, _ = oracle.select(offers, sub, want_top5=False, n_threads=threads)
    bad_rows = int((best_np[rows] != ob).sum())
    return {"rows_checked": int(P), "classes": int(len(classes)), "rows_wrong_by_class": bad_class, "sampled_rows": int(len(rows)),
            "sampled_rows_wrong": bad_rows, "ok": bad_class == 0 and bad_rows == 0}


def check_status_parity(got_idx, got_codes, tab_prev, tab_last, oracle):
    """The last executed sweep against the reference's predicate (string / bool compare, oracle) and translateRunPodStatus."""
    want = np.nonzero((compared_fields(tab_prev) != compared_fields(tab_last)).any(axis=1))[0].astype(np.uint32) if tab_prev is not tab_last \
        else np.zeros(0, np.uint32)
    t = oracle.StatusTable(tab_prev.shape[0], tab_prev.shape[1])
    t.diff(tab_prev)
    want_oracle = t.diff(tab_last)
    ok_idx = np.array_equal(np.asarray(got_idx, np.uint32), want_oracle) and np.array_equal(want, want_oracle)
    ok_codes = got_codes is None or np.array_equal(np.asarray(got_codes, np.uint16), oracle.record_codes(tab_last)[want_oracle])
    return {"slots_checked": int(tab_last.shape[0]), "changed": int(len(want_oracle)), "changed_list_ok": bool(ok_idx), "codes_ok": bool(ok_codes),
            "ok": bool(ok_idx and ok_codes)}


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="rpk", choices=["rpk", "reference"])
    ap.add_argument("--pods", type=int, default=1_000_000, help="P (total, sharded by row)")
    ap.add_argument("--offers", type=int, default=100_000, help="G")
    ap.add_argument("--slots", type=int, default=1_000_000, help="tracked status slots (total, sharded)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of the timed result (never do this for a reported number)")
    ap.add_argument("--no-k2-sweep", action="store_true", help="skip the large-N status sweep used for the K2 HBM roofline")
    ap.add_argument("--k2-slots", type=int, default=1 << 24)
    ap.add_argument("--no-weak-probe", action="store_true", help="skip the fixed-work-per-GPU probe (N > 1)")
    ap.add_argument("--stream-seconds", type=float, default=2.0, help="BASELINE config 5 leg per policy (0 = skip)")
    ap.add_argument("--gather", default="p2p", choices=["nccl", "p2p"], help="how the assignment vector is all-gathered (N>1)")
    ap.add_argument("--launch", default="auto", choices=["auto", "graph", "eager"],
                    help="auto: both ways are tried for a few steps after the warm-up and the faster one is timed; graph: each step (status sweep on its side stream + select + fused gather + peer wait) is captured once per "
                         "parity as a CUDA graph and replayed; eager: one C-ABI call per launch group")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0's assignment vector, the sweep's changed "
                         "slot list and codes) as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "rpk":
        ap.error("--dump-outputs writes what the GPU arm computed; the reference arm times a pod sample that varies from run to run")
    args.warmup = max(args.warmup, 3) if args.impl == "rpk" else args.warmup

    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import importlib

    import torch
    import torch.distributed as dist

    pkg = importlib.import_module("k8s-runpod-kubelet_b200")
    synth = pkg.synth
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    host_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        host_group = dist.new_group(backend="gloo")  # CPU-side waits: idle ranks must not spin an NCCL kernel on their GPU
    P, G, NS = args.pods, args.offers, args.slots
    lo, hi = shard(P, world, rank)
    slo, shi = shard(NS, world, rank)
    Pl, Nl = hi - lo, shi - slo
    cap = -(-NS // world) + 1  # per-rank capacity of the changed-list exchange buffers

    # ---- resident inputs ------------------------------------------------------------------------------
    offers = synth.make_offers(G)
    eng = pkg.Engine(1, device_ids=[local_rank])
    eng.upload_offers(offers)
    pods_np = synth.make_pods(Pl, row0=lo)
    d_pods = {k: torch.from_numpy(v).to(dev) for k, v in pods_np.items()}
    recs_np = [synth.make_status_records(Nl, 0, row0=slo), synth.make_status_records(Nl, 1, 0.01, row0=slo)]
    d_recs = [torch.from_numpy(r.reshape(-1)).to(dev) for r in recs_np]
    d_hash_prev = torch.zeros(Nl, dtype=torch.int64, device=dev)
    d_changed = torch.empty(max(Nl, 1), dtype=torch.int32, device=dev)
    d_code = torch.empty(max(Nl, 1), dtype=torch.int16, device=dev)
    d_nchanged = torch.zeros(1, dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    # Two sets of result buffers, used by even / odd steps: a rank that has passed the wait of step e may start step
    # e+1 and push into its peers' buffers while they still read step e's -- with two sets it writes the other one
    # (rpk.h, rpk_peer_bind).
    best_sets = [torch.full((P,), -7, dtype=torch.int32, device=dev) for _ in range(2)]
    gather_ptrs, xchg_ptrs, xchg_views, gather_mode = None, None, None, "n/a"
    if world > 1:
        gather_mode = args.gather
        if args.gather == "p2p":
            ok = torch.ones(1, dtype=torch.int32, device=dev)
            try:
                peer = importlib.import_module("k8s-runpod-kubelet_b200.peer")
                sets = [peer.exchange_peer_buffer(eng, P * 4, rank, world) for _ in range(2)]
                xs = [peer.exchange_peer_buffer(eng, eng.xchg_bytes(world, cap), rank, world) for _ in range(2)]
                flag_ptrs = peer.exchange_peer_buffer(eng, 64 * 4, rank, world)[1]
                eng.peer_bind(flag_ptrs, rank)
                eng.peer_inline_wait(True)  # the last pusher of each kernel also waits for the peers: no wait launch
            except Exception as e:  # IPC not permitted on this box: fall back to the NCCL all-gather
                ok.zero_()
                sys.stderr.write(f"[rank {rank}] p2p gather unavailable ({e}); using NCCL all-gather\n")
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 1:
                best_sets = [peer.as_int32_tensor(own, P, dev) for own, _ in sets]
                gather_ptrs = [ptrs for _, ptrs in sets]
                xchg_ptrs = [ptrs for _, ptrs in xs]
                xchg_views = [peer.as_int32_tensor(own, eng.xchg_bytes(world, cap) // 4, dev) for own, _ in xs]
                for b in best_sets:
                    b.fill_(-7)
            else:
                gather_mode = "nccl (p2p/IPC unavailable)"
    p2p = gather_ptrs is not None
    executed = []  # record-table index of every sweep that actually ran (captures do not run)
    capturing = [False]

    def select_and_gather(par, kev=None):
        if kev:
            kev[0].record()
        if p2p:
            eng.select_device_gather(d_pods, gather_ptrs[par], lo)  # pushes finished blocks and signals the peers by itself
        else:
            eng.select_device(d_pods, best_sets[par][lo:hi])
        if kev:
            kev[1].record()
        if world > 1 and not p2p:
            dist.all_gather_into_tensor(best_sets[par], best_sets[par][lo:hi])

    # the status sweep is independent of the selection: it runs on a second stream, concurrently.  The selection is the
    # latency-critical half: its stream has the higher priority, so when both kernels have CTAs pending the selection's
    # are placed first (the sweep beside a 1M-row select then costs 5 us instead of 15)
    torch.cuda.synchronize()
    torch.cuda.set_stream(torch.cuda.Stream(device=dev, priority=-1))
    side = torch.cuda.Stream(device=dev, priority=0)
    ev_fork, ev_join = torch.cuda.Event(), torch.cuda.Event()

    def status_on_side(par, st_ev=None):
        if st_ev:
            st_ev[0].record(side)
        if p2p:  # sharded sweep: the changed list (count, global ids, codes) goes into every rank's exchange buffer
            eng.status_diff_device_gather(d_recs[par], 32, d_hash_prev, slo, xchg_ptrs[par], cap, rank, d_nchanged, stream=side.cuda_stream)
        else:
            eng.status_diff_device(d_recs[par], 32, d_hash_prev, d_changed, d_nchanged, stream=side.cuda_stream, d_changed_code=d_code)
        if st_ev:
            st_ev[1].record(side)
        if not capturing[0]:
            executed.append(par)

    def step(i):
        par = i & 1
        ev_fork.record()
        side.wait_event(ev_fork)
        status_on_side(par)
        ev_join.record(side)
        select_and_gather(par)
        torch.cuda.current_stream().wait_event(ev_join)  # p2p: both kernels end only when every rank's results have landed here

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def changed_list(par):
        """(slot ids, codes) of the sweep that last wrote result set `par`.  p2p: every rank's region of this rank's
        exchange buffer, in rank order (global slot ids); otherwise this rank's own list (local slot ids)."""
        if p2p:
            xv = xchg_views[par].cpu().numpy()
            counts = xv[:world].astype(np.int64)
            idx = np.concatenate([xv[8 + r * cap: 8 + r * cap + counts[r]] for r in range(world)]).astype(np.uint32)
            codes16 = xv[8 + world * cap:].view(np.uint16)
            return idx, np.concatenate([codes16[r * cap: r * cap + counts[r]] for r in range(world)])
        n = int(d_nchanged.item())
        return d_changed[:n].cpu().numpy().astype(np.uint32), d_code[:n].cpu().numpy().view(np.uint16)

    sampler = ClockSampler(local_rank)  # clocks under this load: polled from the warm-up through the timed steps
    sampler.start()
    for i in range(args.warmup):
        step(i)
    barrier()

    # ---- CUDA graphs: one per parity (the sweep alternates between two record tables, the results between two sets) ----
    # The device entry points enqueue launches only (no allocation or synchronisation once warmed up), so a step
    # captures as is.  All ranks must agree on the mode: a rank that cannot capture drags everyone back to eager.
    graphs, launch_mode, launches_per_step = None, "eager", None
    want_graph = args.launch in ("graph", "auto") and not (world > 1 and not p2p)
    launch_trial = None
    if want_graph:
        ok = torch.ones(1, dtype=torch.int32, device=dev)
        try:
            cap_stream = torch.cuda.Stream(device=dev, priority=-1)
            cap_stream.wait_stream(torch.cuda.current_stream())
            graphs = []
            capturing[0] = True
            for parity in (0, 1):
                g = torch.cuda.CUDAGraph()
                n0 = eng.launch_count()
                with torch.cuda.graph(g, stream=cap_stream, capture_error_mode="relaxed"):
                    step(parity)
                launches_per_step = eng.launch_count() - n0
                graphs.append(g)
            torch.cuda.current_stream().wait_stream(cap_stream)
        except Exception as e:
            ok.zero_()
            graphs = None
            sys.stderr.write(f"[rank {rank}] CUDA graph capture failed ({type(e).__name__}: {e}); eager launches\n")
        capturing[0] = False
        if world > 1:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 1:
            launch_mode = "graph"
            ref_best = [b.clone() for b in best_sets]
            barrier()             # nobody overwrites a peer's vector before that peer has taken its copy
            for b in best_sets:
                b.fill_(-7)
            barrier()
            for i in range(max(args.warmup, 2)):  # replays warm up too (and keep the epochs of all ranks in step)
                graphs[i & 1].replay()
                executed.append(i & 1)
            barrier()
            same = torch.tensor([int(all(bool((b == r).all()) for b, r in zip(best_sets, ref_best)))], dtype=torch.int32, device=dev)
            if world > 1:
                dist.all_reduce(same, op=dist.ReduceOp.MIN)
            if int(same.item()) != 1:  # never time a replay that does not reproduce the eager result
                sys.stderr.write(f"[rank {rank}] graph replay and eager launches disagree on the assignment vector; eager launches\n")
                launch_mode, graphs = "eager (graph replay disagreed with eager launches)", None
            del ref_best
        else:
            graphs = None
        barrier()

    def eager_timed_step(i, ev, st_ev, k_ev, wait_launch=False):
        par = i & 1
        flush.fill_(i & 0xFF)  # L2 flush between timed iterations (outside the event pairs)
        ev[0].record()
        side.wait_event(ev[0])
        status_on_side(par, st_ev)
        select_and_gather(par, k_ev)
        torch.cuda.current_stream().wait_event(st_ev[1])
        if wait_launch:
            eng.peer_wait(3)
        ev[1].record()

    # ---- --launch auto: the same step both ways, a few times each; every rank takes the same decision (max over ranks) ----
    if graphs is not None and args.launch == "auto":
        trial = {}
        for mode in ("graph", "eager"):
            t_evs = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(8)]
            scratch_ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(2)]
            base = executed[-1] ^ 1
            barrier()
            for i in range(8):
                if mode == "graph":
                    flush.fill_(i & 0xFF)
                    t_evs[i][0].record()
                    graphs[(base + i) & 1].replay()
                    executed.append((base + i) & 1)
                    t_evs[i][1].record()
                else:
                    eager_timed_step(base + i, t_evs[i], scratch_ev[0], scratch_ev[1])
            barrier()
            tt = torch.tensor([sum(e[0].elapsed_time(e[1]) for e in t_evs[2:]) / 6.0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            trial[mode] = float(tt.item())
        launch_trial = {"graph_ms_per_step": trial["graph"], "eager_ms_per_step": trial["eager"], "steps_each": 6}
        if trial["eager"] < trial["graph"]:
            graphs, launch_mode = None, "eager"

    # ---- timed region ---------------------------------------------------------------------------------
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(args.steps)]
    st_evs = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(args.steps)]
    k_evs = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(args.steps)]
    launches0 = eng.launch_count()
    base = executed[-1] ^ 1  # keeps the record tables alternating across the phases: every timed sweep sees 1 % changed slots
    barrier()
    wall0 = time.perf_counter()
    for i in range(args.steps):
        if graphs is not None:
            flush.fill_(i & 0xFF)  # L2 flush between timed iterations (outside the event pairs)
            evs[i][0].record()
            graphs[(base + i) & 1].replay()
            executed.append((base + i) & 1)
            evs[i][1].record()
        else:
            eager_timed_step(base + i, evs[i], st_evs[i], k_evs[i])
    barrier()
    wall = time.perf_counter() - wall0
    launches = (launches_per_step * args.steps) if graphs is not None else (eng.launch_count() - launches0)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:  # before the breakdown pass below runs more steps
        idx, codes = changed_list(executed[-1])
        dump_outputs(args.dump_outputs, {"best": best_sets[executed[-1]].cpu().numpy(), "status_changed": idx, "status_codes": codes})
    tot_ms = [e[0].elapsed_time(e[1]) for e in evs]        # whole step: select (+ gather) with the status sweep alongside
    if graphs is not None:
        # per-kernel breakdown: timing events cannot sit inside a captured graph, so the same steps run once more
        # eagerly (not part of `value`); every rank takes part (the wait is collective)
        b_steps = min(args.steps, 10)
        b_evs = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(b_steps)]
        st_evs, k_evs = st_evs[:b_steps], k_evs[:b_steps]
        base = executed[-1] ^ 1
        if p2p:  # the kernels' own durations: here the wait is a launch of its own (with the in-kernel wait the eagerly
            eng.peer_inline_wait(False)  # launched kernels of the faster rank would also count the other rank's launch skew)
        for i in range(b_steps):
            eager_timed_step(base + i, b_evs[i], st_evs[i], k_evs[i], wait_launch=p2p)
        barrier()
        if p2p:
            eng.peer_inline_wait(True)
        scale = args.steps / b_steps  # the sums below are divided by args.steps
        st_ms = [e[0].elapsed_time(e[1]) * scale for e in st_evs]
        sel_ms = [e[0].elapsed_time(e[1]) * scale for e in k_evs]
        eager_ms_per_step = sum(e[0].elapsed_time(e[1]) for e in b_evs) / b_steps
    else:
        st_ms = [e[0].elapsed_time(e[1]) for e in st_evs]      # status sweep on the side stream (overlapped)
        sel_ms = [e[0].elapsed_time(e[1]) for e in k_evs]      # the select launches alone (classify + scatter + grid kernel)
        eager_ms_per_step = None
    t = torch.tensor([sum(tot_ms), sum(sel_ms), sum(st_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        lt = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(lt)
        launches = int(lt.item())
    total_ms, select_ms, status_ms = (float(x) for x in t.tolist())
    ms_per_step = total_ms / args.steps
    value = P * G / (ms_per_step * 1e-3)
    n_changed = int(d_nchanged.item())

    # ---- parity: what was timed is what the reference computes (every rank checks the whole vector it holds) ----
    parity = None
    last_par = executed[-1]
    if not args.no_parity:
        import oracle

        threads = max(1, host_threads() // max(1, world))
        pods_all = pods_np if world == 1 else synth.make_pods(P, row0=0)
        sel = check_select_parity(best_sets[last_par].cpu().numpy(), offers, pods_all, oracle, threads)
        tabs = recs_np if world == 1 else [synth.make_status_records(NS, 0), synth.make_status_records(NS, 1, 0.01)]
        prev_par = executed[-2] if len(executed) > 1 else last_par
        idx, codes = changed_list(last_par)
        n_changed = len(idx)
        if world > 1 and not p2p:  # NCCL comparison mode: each rank checks its own shard (local slot ids)
            tabs = recs_np
        st = check_status_parity(idx, codes, tabs[prev_par], tabs[last_par], oracle)
        flag = torch.tensor([int(sel["ok"] and st["ok"])], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(flag, op=dist.ReduceOp.SUM)
        parity = {"select": sel, "status_sweep": st, "ranks_ok": int(flag.item()), "ranks": world, "ok": int(flag.item()) == world,
                  "what": "the assignment vector each rank holds after the last timed/breakdown step (all P rows by class property + sampled rows "
                          "row by row vs the C oracle) and the last sweep's gathered changed list + codes vs the oracle's predicate / translate"}
        if not parity["ok"]:
            sys.stderr.write(f"[rank {rank}] PARITY FAILURE: {json.dumps({'select': sel, 'status': st})}\n")
    else:
        assert int((best_sets[last_par] == -7).sum().item()) == 0, "assignment vector has unwritten rows"

    # ---- weak-scaling probe (N > 1): every rank selects over a full P-row shard (N*P pods in total) --------
    weak = None
    if world > 1 and not args.no_weak_probe:
        wp = synth.make_pods(P, row0=rank * P)
        d_wp = {k: torch.from_numpy(v).to(dev) for k, v in wp.items()}
        w_full = torch.empty(world * P, dtype=torch.int32, device=dev)
        w_mine = w_full[rank * P:(rank + 1) * P]

        def weak_step():
            eng.select_device(d_wp, w_mine)
            dist.all_gather_into_tensor(w_full, w_mine)

        for _ in range(3):
            weak_step()
        barrier()
        wsteps = min(args.steps, 10)
        we = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        we[0].record()
        for _ in range(wsteps):
            weak_step()
        we[1].record()
        barrier()
        wt = torch.tensor([we[0].elapsed_time(we[1]) / wsteps], dtype=torch.float64, device=dev)
        dist.all_reduce(wt, op=dist.ReduceOp.MAX)
        weak = {"pods_total": world * P, "offers": G, "ms_per_step": float(wt.item()), "value": world * P * G / (float(wt.item()) * 1e-3),
                "unit": UNIT, "note": "per-GPU work fixed at P rows (select + NCCL all-gather of the N*P-entry vector, no status sweep, no "
                                      "L2 flush); the headline `value` above is the strong-scaling C4 figure"}
        del d_wp, w_full

    # ---- end to end through the host C-ABI: rank 0 drives all N GPUs from one ctx ---------------------
    e2e, k2, streaming = None, None, None
    barrier()
    if rank == 0:
        if not args.no_k2_sweep:
            k2 = run_k2_sweep(eng, synth, dev, args)
        if not args.no_e2e:
            e2e = run_e2e(pkg, synth, offers, P, G, NS, world, args)
        if args.stream_seconds > 0:
            streaming = run_streaming(pkg, synth, world, args)
    if world > 1:
        dist.barrier(group=host_group)  # ranks > 0 wait on the CPU while rank 0 drives every GPU from one ctx
    barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        sys.exit(0 if (parity is None or parity["ok"]) else 3)

    peak, peak_src = measured_peaks()
    k1_ms = select_ms / args.steps  # the select launches: classify + scatter (a few %) + the grid kernel (with its fused push at N > 1)
    achieved = MODEL_BYTES_PER_SCORE * (P / world) * G / (k1_ms * 1e-3) / 1e9
    traffic = None
    prof = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.exists(prof):
        try:
            traffic = json.load(open(prof)).get("dram_bytes_per_launch")
        except Exception:
            pass
    sm_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
    stats = eng.stats()
    kind = stats["select_kernel_kind"]
    if kind == 4:
        # bit-sliced kernel: per (row, 32-offer chunk) one 4-byte mask word per CONSTRAINING column comes out of shared
        # memory (mem always; vcpu / ram only if the row's request exceeds the smallest offer value).  The persistent
        # kernel fetches the words of four chunks with one LDS.128 whose lanes share addresses: measured 2 LSU cycles per
        # warp instruction (tools/microbench/lds_probe.cu) = 64 (row, chunk) words per clock per SM.
        ov, orr = offers.get("vcpu"), offers.get("ram_gb")
        need_v = pods_np["req_vcpu"] > (ov.min() if ov is not None and len(ov) else 0)
        need_r = pods_np["req_ram_gb"] > (orr.min() if orr is not None and len(orr) else 0)
        words = float(np.mean(1.0 + need_v + need_r))
        true_peak = 148 * sm_hz * (64.0 / words) * 32
        true_model = (f"shared-memory return path: 148 SMs x 64 mask words/clk (LDS.128 with shared addresses: 2 cycles per warp instruction, "
                      f"measured) x sm_clock x 32 pairs / {words:.2f} mask words per (row, chunk) (rank-0 row mix: 1 word for mem + 1 per "
                      "constraining vcpu/ram request)")
        true_bound = "shared-memory bandwidth (LDS return path)"
    else:
        ipc = {3: 2.5, 2: 3.0}.get(kind, 4.0)
        true_peak, true_model = 148 * 4 * 32 * sm_hz / ipc, f"148 SMs x 4 SMSPs x 32 lanes x sm_clock / {ipc} instructions per offer-score"
        true_bound = "warp-instruction issue (INT/ALU pipes)"
    onchip = {"bound": true_bound, "achieved": (P / world) * G / (k1_ms * 1e-3), "unit": "offer-scores/s per GPU",
              "peak": true_peak, "frac": (P / world) * G / (k1_ms * 1e-3) / true_peak, "model": true_model,
              "note": "THE limit that binds K1: the kernel keeps its stage of the offer table in shared memory, so HBM sees only the "
                      "compulsory pod-side columns; read this fraction, not the HBM yardstick below"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u32 bit masks over rank-compressed int32 columns + f64 price compare", "data": "synthetic",
        "config": {"workload": f"C4: P={P} pending pods x G={G} offers, full grid (every pair evaluated), pod rows sharded over "
                               f"{world} GPU(s) + all-gather of the assignment vector ({gather_mode}); "
                               f"one status sweep over N={NS} tracked slots (1% mutate per step) runs concurrently on a second stream"
                               + (", its changed list exchanged between all ranks" if p2p else ""),
                   "pods": P, "offers": G, "status_slots": NS, "gather": gather_mode,
                   "fence": ("signal AND wait folded into the last pusher of each kernel (rpk_peer_inline_wait); results double-buffered (even/odd steps)" if p2p else "n/a"),
                   "l2": "flushed between timed iterations (256 MiB write)",
                   "streams": "select on a high-priority stream, the status sweep on a default-priority side stream",
                   "launch": ("one CUDA graph replay per step (captured from the same C-ABI device entry points)" if launch_mode == "graph"
                              else "eager C-ABI calls" if launch_mode == "eager" else launch_mode),
                   "launch_trial": launch_trial,
                   "select_kernel": {1: "generic int32 compare", 2: "packed rank fields + select", 3: "packed rank fields + embedded position (min)",
                                     4: "bit-sliced threshold masks, persistent kernel on the transposed view (32 pairs per mask word, 4 chunks per LDS.128)"}.get(kind),
                   "packed_bits": stats["packed_bits"], "table": "SURVEY 8d tie-heavy offers, mixed pod profile"},
        "clocks": clocks,
        "gpu_launches": launches,
        "wall_s_timed_region": wall,
        "parity": parity,
        "breakdown_ms_per_step": {"select_kernels": select_ms / args.steps, "status_diff_overlapped_on_side_stream": status_ms / args.steps,
                                  "step_total_incl_gather": ms_per_step,
                                  **({"note": "select_kernels / status_diff were timed in a separate eager pass (timing events cannot sit inside "
                                              "a captured graph, and at N > 1 with rpk_peer_wait as a launch of its own so that the kernel times hold no "
                                              "launch skew between ranks); step_total is the graph-replayed step `value` is computed from",
                                      "eager_step_total_rank0": eager_ms_per_step} if launch_mode == "graph" else {})},
        "reconcile": {"metric": "pods reconciled/sec", "value": NS / (status_ms / args.steps * 1e-3), "unit": "pods/s",
                      "changed_last_step": n_changed, "gathered": bool(p2p),
                      "note": f"N={NS} slots x 40 B is launch/latency-bound at this size; see roofline_status_diff for the HBM-bound sweep"},
        "roofline_onchip": onchip,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_source": peak_src,
                     "model": "north-star YARDSTICK only (SURVEY 8d streaming model: 16 algorithmic bytes per offer-score, one 4xint32 offer view "
                              "per score).  The kernel stages offer segments in shared memory, so real DRAM traffic is only the compulsory "
                              "pod-side columns (see traffic, ncu) and frac exceeds 1 by construction; it says nothing about kernel quality -- "
                              "roofline_onchip is the bound that binds K1, roofline_status_diff the HBM-bound kernel of this path."},
    }
    if k2:
        for k in k2.values():
            k["peak"], k["peak_source"] = peak, peak_src
            k["frac"] = k["achieved"] / peak
        line["roofline_status_diff"] = k2["stride32"]
        line["roofline_status_diff16"] = k2["stride16"]
    if weak:
        line["weak_scaling_probe"] = weak
    if e2e:
        line["e2e"] = e2e
    if streaming:
        line["streaming"] = streaming
    if not args.no_cpu_baseline and world == 1:
        import oracle

        threads = host_threads()
        v, desc, _, _ = cpu_select_sample(offers, G, 15.0, threads, synth, oracle)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": desc + "; C restatement of runpod_client.go:465-509 (Go toolchain absent)"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    bad = (parity is not None and not parity["ok"]) or (e2e is not None and not e2e.get("parity_ok", True)) or \
        (streaming is not None and not all(s["assignments_ok"] for s in streaming["runs"]))
    sys.exit(3 if bad else 0)


def run_k2_sweep(eng, synth, dev, args):
    """K2 alone at an HBM-bound size: N slots device-resident, 1 % of the slots change per sweep, codes emitted."""
    import torch

    out = {}
    N = args.k2_slots
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for stride in (32, 16):
        base = synth.make_status_records(1 << 20, 0, stride=stride)
        reps = (N + (1 << 20) - 1) >> 20
        a = torch.from_numpy(base).to(dev).repeat(reps, 1)[:N].contiguous()
        b = a.clone()
        rows = torch.arange(0, N, 100, device=dev)          # every 100th slot takes its neighbour's record
        b[rows] = a[(rows + 1) % N]
        tabs = [a.reshape(-1), b.reshape(-1)]
        hash_prev = torch.zeros(N, dtype=torch.int64, device=dev)
        changed = torch.empty(N, dtype=torch.int32, device=dev)
        code = torch.empty(N, dtype=torch.int16, device=dev)
        nchg = torch.zeros(1, dtype=torch.int32, device=dev)
        for i in range(3):
            eng.status_diff_device(tabs[i & 1], stride, hash_prev, changed, nchg, d_changed_code=code)
        torch.cuda.synchronize()
        iters, ms, n_changed = 5, 0.0, 0
        for i in range(iters):
            flush.fill_(i)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            eng.status_diff_device(tabs[(i + 1) & 1], stride, hash_prev, changed, nchg, d_changed_code=code)
            e1.record()
            torch.cuda.synchronize()
            ms += e0.elapsed_time(e1)
            n_changed = int(nchg.item())
        ms /= iters
        algo = N * (stride + 8) + n_changed * 14  # slot + previous hash read; hash + index + code written per changed slot
        out[f"stride{stride}"] = {"kernel": f"k_status_stream<{stride}>", "bound": "hbm", "achieved": algo / (ms * 1e-3) / 1e9, "unit": "GB/s", "slots": N,
                                  "changed_per_sweep": n_changed, "us_per_launch": ms * 1e3, "pods_reconciled_per_s": N / (ms * 1e-3),
                                  "algorithmic_bytes": algo, "l2": "flushed between launches", "traffic": None}
        del a, b, tabs, hash_prev, changed, code
    return out


def run_e2e(pkg, synth, offers, P, G, NS, world, args):
    """Host C-ABI path: pinned host columns -> ONE rpk_tick (selection + status sweep) on one ctx over all N GPUs."""
    import torch

    import oracle

    def pinned(a):
        t = torch.empty(a.shape, dtype=torch.from_numpy(a).dtype, pin_memory=True)
        t.numpy()[...] = a
        return t

    eng = pkg.Engine(world, device_ids=list(range(world)))
    eng.upload_offers(offers)
    pods = synth.make_pods(P, row0=0)
    keep = {k: pinned(v) for k, v in pods.items()}
    pods_pin = {k: t.numpy() for k, t in keep.items()}
    best_t = torch.empty(P, dtype=torch.int32, pin_memory=True)
    best = best_t.numpy()
    stride = 16  # every RunPod status fits the 16-byte slot: the sweep uploads 16 B per tracked pod
    tabs = [synth.make_status_records(NS, 0, stride=stride), synth.make_status_records(NS, 1, 0.01, stride=stride)]
    recs = [pinned(t) for t in tabs]
    steps = min(args.steps, 5)
    idx = codes = None
    for i in range(2):
        eng.tick(pods_pin, recs[i & 1].numpy(), out_best=best)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        _, _, idx, codes = eng.tick(pods_pin, recs[i & 1].numpy(), out_best=best)
    dt = (time.perf_counter() - t0) / steps
    last = (steps - 1) & 1
    sel = check_select_parity(best, offers, pods, oracle, max(1, host_threads()), sample=1000) if not args.no_parity else {"ok": True}
    st = check_status_parity(idx, codes, tabs[last ^ 1], tabs[last], oracle) if not args.no_parity else {"ok": True}
    h2d = sum(v.nbytes for v in pods_pin.values()) + NS * stride
    d2h = best.nbytes + 4 * world + 6 * len(idx)
    out = {"value": P * G / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "ms_per_step": dt * 1e3, "steps": steps, "timing": "host wall clock around rpk_tick (synchronous; selection and sweep enqueued together)",
           "api": f"rpk_tick = rpk_select + rpk_status_diff_codes, one ctx over {world} GPU(s) (one host thread per extra GPU), pinned host buffers, "
                  f"{stride}-byte status slots; the changed list comes back through mapped pinned memory",
           "parity_ok": bool(sel["ok"] and st["ok"]), "parity": {"select": sel, "status_sweep": st}}
    eng.close()
    return out


def run_streaming(pkg, synth, world, args):
    """BASELINE config 5: 10^4 pods/s churn for `--stream-seconds` per policy; every assignment checked against the oracle."""
    import oracle

    stream = __import__("importlib").import_module("k8s-runpod-kubelet_b200.stream")
    offers = synth.make_offers(10_000)
    runs = []
    for policy in ("window", "eager"):
        engines = [pkg.Engine(1, device_ids=[g]) for g in range(world)]
        res, pods_all, best, top5 = stream.run_stream(engines, offers, seconds=args.stream_seconds, policy=policy)
        for e in engines:
            e.close()
        ob, ot = oracle.select(offers, pods_all, want_top5=True, n_threads=max(1, host_threads()))
        res["assignments_checked"] = int(len(best))
        res["assignments_ok"] = bool(np.array_equal(best, ob) and np.array_equal(top5, ot))
        runs.append(res)
    return {"config": "C5 streaming reconcile: 10^4 pods/s Poisson churn, G = 10^4 offers, 10^5 tracked slots with a sweep every 10 ms",
            "api": "rpk_select (top-5) + rpk_status_diff through the host C-ABI, single host thread, micro-batches round-robined over the GPUs",
            "runs": runs}


if __name__ == "__main__":
    main()
