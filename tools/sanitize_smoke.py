"""Small end-to-end run for compute-sanitizer (memcheck / racecheck / synccheck): every kernel kind, top-5,
the latency and the pipelined host paths, both status kernels, offer sets.  Usage on the GPU box:
    compute-sanitizer --tool memcheck python tools/sanitize_smoke.py
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle  # noqa: E402
import rpk  # noqa: E402

ONLY_MULTI = os.environ.get("RPK_SANITIZE_ONLY_MULTI") == "1"  # the 2-GPU part alone (a 2-GPU box is charged twice)
ONLY_SETS = os.environ.get("RPK_SANITIZE_ONLY_SETS") == "1"    # the offer-set part alone


def sets_part():
    """Offer sets: set build (compact / gather / ingest / remap) with empty, one-offer and full sets, and rpk_select_sets
    on the host and device entry points (partition, per-set selects, un-permute), top-5 included, against the oracle."""
    import torch

    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
    import sets_restatement as sr

    es = rpk.Engine(1)
    G = 5000
    so = rpk.synth.make_offers(G, correlated=True, seed=4)
    members = rpk.synth.make_offer_sets(G, 7, seed=4)
    es.upload_offers(so)
    es.upload_offer_sets(members)
    for P in (37, 20_001):  # fused kernel per bin / persistent kernel for the large bins
        pods = rpk.synth.make_pods(P, seed=P)
        ids = rpk.synth.make_set_ids(P, 7, 0.6, seed=P)
        ob, ot = sr.oracle_select_sets(so, pods, members, ids)
        b, t = es.select_sets(pods, ids, want_top5=True)
        assert np.array_equal(b, ob) and np.array_equal(t, ot), ("sets host", P)
        d = {k: torch.from_numpy(v).cuda() for k, v in pods.items()}
        d_best = torch.empty(P, dtype=torch.int32, device="cuda")
        d_top5 = torch.empty(P * 5, dtype=torch.int32, device="cuda")
        es.select_sets_device(d, torch.from_numpy(ids.view(np.int16)).cuda(), d_best, d_top5)
        torch.cuda.synchronize()
        assert np.array_equal(d_best.cpu().numpy(), ob) and np.array_equal(d_top5.cpu().numpy().reshape(P, 5), ot), ("sets device", P)
    es.close()
    print("sanitize_smoke offer-set part ok")


if ONLY_SETS:
    sets_part()
    print("sanitize_smoke ok")
    sys.exit(0)
eng = rpk.Engine(1)
offers = rpk.synth.make_offers(20_000, correlated=True)
for force in () if ONLY_MULTI else (None, "bitmap_grouped", "bitmap_grid", "packed_pos", "packed", "generic"):
    os.environ.pop("RPK_FORCE_KERNEL", None)
    if force:
        os.environ["RPK_FORCE_KERNEL"] = force
    eng.upload_offers(offers)
    for P in (37, 5000, 140_000):  # latency path, one sub-batch, two pipelined sub-batches
        pods = rpk.synth.make_pods(P, seed=P)
        best, t5 = eng.select(pods, want_top5=True)
        ob, ot = oracle.select(offers, pods, n_threads=8)
        assert np.array_equal(best, ob) and np.array_equal(t5, ot), (force, P)
os.environ.pop("RPK_FORCE_KERNEL", None)
for stride in () if ONLY_MULTI else (16, 32, 64):
    tab = oracle.StatusTable(30_000, stride)
    e2 = rpk.Engine(1)
    for sweep, frac in enumerate([0.0, 0.2, 1.0]):
        recs = rpk.synth.make_status_records(30_000, sweep, frac, stride=stride)
        got, codes, hashes = e2.status_diff(recs, want_hashes=True, want_codes=True)
        want = tab.diff(recs)
        assert np.array_equal(got, want) and np.array_equal(hashes, oracle.record_hashes(recs))
        assert np.array_equal(codes, oracle.record_codes(recs)[want])
    e2.status_seed_slots(np.array([5, 77], np.uint32), np.ascontiguousarray(recs[[5, 77]]))
    e2.close()
# the big-table build of the stream kernel (>= 4M slots), ragged last unit
for stride in () if ONLY_MULTI else (32, 16):
    N = (1 << 22) + 37
    e2 = rpk.Engine(1)
    base = rpk.synth.make_status_records(N, 0, stride=stride)
    e2.status_seed(base)
    nxt = rpk.synth.make_status_records(N, 2, 0.01, stride=stride)
    got, codes, _ = e2.status_diff(nxt, want_codes=True)
    tab = oracle.StatusTable(N, stride)
    tab.diff(base)
    want = tab.diff(nxt)
    assert np.array_equal(got, want) and np.array_equal(codes, oracle.record_codes(nxt)[want]), stride
    e2.close()
# one tick: selection and sweep enqueued together
e3 = rpk.Engine(1)
e3.upload_offers(offers)
pods = rpk.synth.make_pods(50_000, seed=3)
recs = rpk.synth.make_status_records(20_000, 0, stride=16)
tb, _, idx, codes = e3.tick(pods, recs)
ob, _ = oracle.select(offers, pods, want_top5=False, n_threads=8)
assert np.array_equal(tb, ob) and len(idx) == 20_000
e3.close()
# device entry points: two output vectors on one GPU (k_gather_push copies local -> local), twice on one scratch
import torch  # noqa: E402

eng.upload_offers(offers)
dev = torch.device("cuda", 0)
for P in (20_001, 70_003):
    pods = rpk.synth.make_pods(P, seed=P)
    d_pods = {k: torch.from_numpy(v).to(dev) for k, v in pods.items()}
    va, vb = torch.full((P + 3,), -9, dtype=torch.int32, device=dev), torch.full((P + 3,), -9, dtype=torch.int32, device=dev)
    ob, _ = oracle.select(offers, pods, want_top5=False, n_threads=8)
    for _ in range(2):
        eng.select_device_gather(d_pods, [va.data_ptr(), vb.data_ptr()], 3)  # slice starts 12 bytes into the vectors
        torch.cuda.synchronize()
        assert np.array_equal(va[3:].cpu().numpy(), ob) and np.array_equal(vb[3:].cpu().numpy(), ob), P
        assert int((va[:3] != -9).sum()) == 0 and int((vb[:3] != -9).sum()) == 0
eng.close()

if not ONLY_MULTI:
    sets_part()

# two GPUs: the fused push + signal + wait, and the sharded sweep's exchange (racecheck / memcheck see peer stores)
if torch.cuda.device_count() >= 2:
    e4 = rpk.Engine(2)
    e4.upload_offers(offers)
    pods = rpk.synth.make_pods(90_001, seed=9)
    ob, _ = oracle.select(offers, pods, want_top5=False, n_threads=8)
    for _ in range(2):
        b, _ = e4.select(pods)
        assert np.array_equal(b, ob)
    tab = oracle.StatusTable(50_001, 16)
    for sweep, frac in enumerate([0.0, 0.3]):
        recs = rpk.synth.make_status_records(50_001, sweep, frac, stride=16)
        got, codes, _ = e4.status_diff(recs, want_codes=True)
        want = tab.diff(recs)
        assert np.array_equal(got, want) and np.array_equal(codes, oracle.record_codes(recs)[want])
    e4.close()
    print("sanitize_smoke 2-GPU part ok")
print("sanitize_smoke ok")
