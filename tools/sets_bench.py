"""Offer-set selection on one B200: set build cost and restricted select cost against the plain select.

  python tools/sets_bench.py [--G 100000] [--P 1000000] [--iters 20] [--out FILE]

Measures, in one process on cuda:0:
  * rpk_offer_sets_upload at G offers for n_sets in {1, 8, 64} non-empty sets (host clock, --iters calls; the call
    synchronises itself) and the device memory those sets take (free memory before / after the first upload);
  * rpk_select_sets_device at P rows x G offers with 8 sets and 0 / 10 / 100 % restricted rows, and rpk_select_device on
    the same rows, alternating the two: host clock around call + stream synchronise, after warm-up, with L2 overwritten
    (256 MiB write) before every timed call;
  * parity of each restricted result: every row through the class property (all rows of one (pod class, set id) share the
    oracle's answer on that set's sub-table) plus sampled rows' best and top-5 against the oracle.
Prints one JSON line (GPU name and power limit included) and writes it to --out if given.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

sys.path.insert(0, os.path.join(ROOT, "tests"))
import rpk  # noqa: E402
from sets_restatement import oracle_select_sets  # noqa: E402  (the contract restated on the C oracle)

SET_ALL = 0xFFFF
POD_COLS = ("req_mem_gb", "req_vcpu", "req_ram_gb", "max_price", "cloud")


def gpu_identity():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        power, clk = [x.strip() for x in q.stdout.strip().split(",")]
    except Exception:
        power, clk = "unknown", "unknown"
    return {"gpu": name, "power_limit": power, "sm_clock_max": clk}


def check_parity(best, top5, offers, pods, members, ids, threads, sample=1500):
    key = np.zeros(len(ids), np.int64)
    radix = 1
    for col in [pods[c] for c in POD_COLS] + [ids]:
        _, inv = np.unique(col, return_inverse=True)
        key += inv.reshape(-1).astype(np.int64) * radix
        radix *= int(inv.max()) + 1
    _, first, inv = np.unique(key, return_index=True, return_inverse=True)
    reps = {k: np.ascontiguousarray(v[first]) for k, v in pods.items()}
    want_class, _ = oracle_select_sets(offers, reps, members, ids[first], n_threads=threads)
    bad_class = int((best != want_class[inv.reshape(-1)]).sum())
    rows = np.random.default_rng(20261017).choice(len(ids), min(sample, len(ids)), replace=False)
    sub = {k: np.ascontiguousarray(v[rows]) for k, v in pods.items()}
    ob, ot = oracle_select_sets(offers, sub, members, ids[rows], n_threads=threads)
    bad_rows = int((best[rows] != ob).sum()) + int((top5[rows] != ot).any(axis=1).sum())
    return {"rows_checked": len(ids), "classes": int(len(first)), "rows_wrong_by_class": bad_class, "sampled_rows": int(len(rows)),
            "sampled_rows_wrong": bad_rows, "ok": bad_class == 0 and bad_rows == 0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--G", type=int, default=100_000)
    ap.add_argument("--P", type=int, default=1_000_000)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("sets_bench: no CUDA device (this measures the GPU path only)")
    threads = max(1, min(32, os.cpu_count() or 1))
    G, P, synth = args.G, args.P, rpk.synth
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    offers = synth.make_offers(G, correlated=True)
    pods = synth.make_pods(P)
    out = {"tool": "sets_bench", **gpu_identity(), "G": G, "P": P, "iters": args.iters, "warmup": args.warmup,
           "clock": "host perf_counter around call + synchronise", "l2": "256 MiB write before every timed call"}
    eng = rpk.Engine(1)
    eng.upload_offers(offers)

    # ---- set build: non-empty sets only (sizes cycle one offer, 1 %, 10 %, 50 %, all; n_sets = 1 is one 10 % set) ----
    upload = {}
    pool = synth.make_offer_sets(G, 6 * 64)
    pool = pool[pool.sum(axis=1) > 0]
    for n_sets in (1, 8, 64):
        members = pool[2:3] if n_sets == 1 else pool[:n_sets]
        eng.upload_offer_sets(np.zeros((0, G), bool))  # no sets resident: the memory delta below is these sets' own
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info(0)[0]
        eng.upload_offer_sets(members)  # warm-up (allocations)
        free1 = torch.cuda.mem_get_info(0)[0]
        ts = []
        for _ in range(args.iters):
            t0 = time.perf_counter()
            eng.upload_offer_sets(members)
            ts.append((time.perf_counter() - t0) * 1e3)
        upload[str(n_sets)] = {"ms_median": statistics.median(ts), "ms_min": min(ts), "calls": len(ts),
                               "members": int(members.sum()), "set_sizes": [int(x) for x in members.sum(axis=1)],
                               "device_bytes": int(free0 - free1)}
    out["offer_sets_upload"] = upload

    # ---- restricted select vs plain select ----
    n_sets = 8
    members = synth.make_offer_sets(G, n_sets)
    eng.upload_offer_sets(members)
    out["sets"] = {"n_sets": n_sets, "sizes": [int(x) for x in members.sum(axis=1)]}
    d = {k: torch.from_numpy(v).to(dev) for k, v in pods.items()}
    d_best = torch.empty(P, dtype=torch.int32, device=dev)
    d_plain = torch.empty(P, dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream()
    runs = {}
    parity_ok = True
    for frac in (0.0, 0.1, 1.0):
        ids = synth.make_set_ids(P, n_sets, frac)
        d_ids = torch.from_numpy(ids.view(np.int16)).to(dev)
        calls = {"select_sets_device": lambda: eng.select_sets_device(d, d_ids, d_best),
                 "select_device": lambda: eng.select_device(d, d_plain)}
        for _ in range(args.warmup):
            for fn in calls.values():
                fn()
        torch.cuda.synchronize()
        times = {k: [] for k in calls}
        for i in range(args.iters):
            for name, fn in (calls.items() if i % 2 == 0 else reversed(list(calls.items()))):
                flush.fill_(i & 0xFF)
                st.synchronize()
                t0 = time.perf_counter()
                fn()
                st.synchronize()
                times[name].append((time.perf_counter() - t0) * 1e6)
        # parity (outside the timed region): the restricted result, with top-5, against the oracle
        d_top5 = torch.empty(P * 5, dtype=torch.int32, device=dev)
        eng.select_sets_device(d, d_ids, d_best, d_top5)
        torch.cuda.synchronize()
        par = check_parity(d_best.cpu().numpy(), d_top5.cpu().numpy().reshape(P, 5), offers, pods, members, ids, threads)
        parity_ok = parity_ok and par["ok"]
        runs[f"{int(frac * 100)}%"] = {
            "restricted_rows": int((ids != SET_ALL).sum()),
            **{f"{k}_us_median": statistics.median(v) for k, v in times.items()},
            **{f"{k}_us_min": min(v) for k, v in times.items()},
            "parity": par}
    out["select_1m"] = runs
    out["parity"] = "ok" if parity_ok else "FAILED"
    eng.close()
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")
    sys.exit(0 if parity_ok else 3)


if __name__ == "__main__":
    main()
