"""Offer sets (``runpod.io/gpu-type-ids``): a pod restricted to a set gets GetGPUTypes over the set's sub-table.

CPU part: the two restatements (sets_restatement.py) against the hand-derived golden vectors and against each other;
the membership packing and the synthetic set generators.  GPU part (``-m gpu``): rpk_offer_sets_upload /
rpk_select_sets / rpk_select_sets_device through the C-ABI, bit-exact against the oracle over table flavours, set
counts and sizes, row mixes, every kernel path and the batch-size boundaries, plus the call-order contract."""
import json
import os

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

import oracle
import rpk
import sets_restatement as sr
from test_oracle import CLOUD, kat_offers
from test_oracle_property import tables

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ALL = sr.SET_ALL
pack_offer_sets = rpk._pkg.engine.pack_offer_sets


def kat_sets():
    kat, offers = kat_offers()
    names = [o["id"] for o in kat["offers"]]
    cases = json.load(open(os.path.join(GOLD, "select_sets_kat.json")))["cases"]
    lists = [c["set"] for c in cases if c["set"] != "ALL"]
    members = np.array([[n in lst for n in names] for lst in lists], bool)
    pods = {"req_mem_gb": np.array([c["minMem"] for c in cases], np.int32),
            "max_price": np.array([c["maxPrice"] for c in cases], np.float64),
            "cloud": np.array([CLOUD.get(c["cloud"], 7) for c in cases], np.uint8)}
    set_id, k = [], 0
    for c in cases:
        if c["set"] == "ALL":
            set_id.append(ALL)
        else:
            set_id.append(k)
            k += 1
    want = np.array([c["top5"] + [-1] * (5 - len(c["top5"])) for c in cases], np.int32)
    return offers, pods, members, np.array(set_id, np.uint16), want


# ---- CPU --------------------------------------------------------------------------------------------------------

def test_kat_restatements():
    offers, pods, members, set_id, want = kat_sets()
    for b, t in (sr.oracle_select_sets(offers, pods, members, set_id), sr.np_select_sets(offers, pods, members, set_id)):
        assert np.array_equal(t, want) and np.array_equal(b, want[:, 0])


@st.composite
def tables_with_sets(draw):
    offers, pods = draw(tables())
    G = len(offers["mem_gb"])
    P = len(pods["req_mem_gb"])
    n_sets = draw(st.integers(0, 5))
    members = np.array(draw(st.lists(st.lists(st.booleans(), min_size=G, max_size=G), min_size=n_sets, max_size=n_sets)), bool).reshape(n_sets, G)
    ids = draw(st.lists(st.one_of(st.integers(0, n_sets + 2), st.just(ALL)), min_size=P, max_size=P))
    return offers, pods, members, np.array(ids, np.uint16)


@settings(max_examples=300, deadline=None)
@given(tables_with_sets())
def test_restatements_agree(t):
    offers, pods, members, set_id = t
    b0, t0 = sr.oracle_select_sets(offers, pods, members, set_id, n_threads=1)
    b1, t1 = sr.np_select_sets(offers, pods, members, set_id)
    assert np.array_equal(b0, b1) and np.array_equal(t0, t1)
    for p in range(len(b0)):  # a restricted row only ever lists members of its set
        s = int(set_id[p])
        ids = [i for i in t0[p] if i >= 0]
        if s != ALL:
            assert all(s < len(members) and members[s][i] for i in ids)


def test_unrestricted_rows_equal_select():
    for seed in (1, 2, 3):
        offers = rpk.synth.make_offers(300, seed=seed, correlated=seed == 2)
        assert sr.unrestricted_equals_select(offers, rpk.synth.make_pods(200, seed=seed))


def test_synthetic_sets_on_larger_tables():
    offers = rpk.synth.make_offers(2000, correlated=True)
    pods = rpk.synth.make_pods(300)
    members = rpk.synth.make_offer_sets(2000, 7)
    set_id = rpk.synth.make_set_ids(300, 7, 0.7)
    b0, t0 = sr.oracle_select_sets(offers, pods, members, set_id)
    b1, t1 = sr.np_select_sets(offers, pods, members, set_id)
    assert np.array_equal(b0, b1) and np.array_equal(t0, t1)
    assert (b0 >= 0).any() and (b0 < 0).any()


def test_pack_offer_sets_layout():
    G = 70
    m = np.zeros((3, G), bool)
    m[0, [0, 31, 32, 69]] = True
    m[2, :] = True
    w = pack_offer_sets(m)
    assert w.dtype == np.uint32 and w.shape == (3, 3)
    assert w[0].tolist() == [(1 << 0) | (1 << 31), 1, 1 << 5]
    assert w[1].tolist() == [0, 0, 0]
    assert w[2].tolist() == [0xFFFFFFFF, 0xFFFFFFFF, (1 << 6) - 1]
    assert pack_offer_sets(np.zeros((0, G), bool)).shape == (0, 3)


def test_synth_sets_are_deterministic_and_sized():
    G = 100_000
    m = rpk.synth.make_offer_sets(G, 12)
    assert np.array_equal(m, rpk.synth.make_offer_sets(G, 12))
    sizes = m.sum(axis=1)
    assert sizes[0] == 0 and sizes[1] == 1 and sizes[5] == G and sizes[6] == 0 and sizes[7] == 1
    assert 700 < sizes[2] < 1300 and 9000 < sizes[3] < 11000 and 48000 < sizes[4] < 52000
    ids = rpk.synth.make_set_ids(50_000, 8, 0.5)
    assert np.array_equal(ids, rpk.synth.make_set_ids(50_000, 8, 0.5))
    assert np.array_equal(ids[1000:2000], rpk.synth.make_set_ids(1000, 8, 0.5, row0=1000))
    restricted = ids != ALL
    assert 0.45 < restricted.mean() < 0.55
    assert ((ids >= 8) & restricted).any() and (ids[restricted] < 8 + 7).all()
    assert (rpk.synth.make_set_ids(1000, 8, 0.0) == ALL).all()
    assert (rpk.synth.make_set_ids(1000, 0, 1.0) != ALL).all()


# ---- GPU --------------------------------------------------------------------------------------------------------

FORCES = [None, "bitmap_grouped", "bitmap_grid", "packed_pos", "packed", "generic"]
FLAVOURS = {"tie_heavy": {}, "tie_free": {"tie_free": True}, "correlated": {"correlated": True},
            "no_ext": {"with_ext": False, "correlated": True}}
P_SIZES = (1, 4096, 4097, 16385, 200_000)  # small-batch, fused and persistent boundaries


def upload_forced(engine, offers, members, force):
    old = os.environ.pop("RPK_FORCE_KERNEL", None)
    if force:
        os.environ["RPK_FORCE_KERNEL"] = force
    try:
        engine.upload_offers(offers)  # the kernel choice is made here and kept for the sets built on this table
    finally:
        os.environ.pop("RPK_FORCE_KERNEL", None)
        if old is not None:
            os.environ["RPK_FORCE_KERNEL"] = old
    engine.upload_offer_sets(members)


def row_mix(name, P, n_sets, seed):
    if name == "all":
        return np.full(P, ALL, np.uint16)
    if name == "none":
        return rpk.synth.make_set_ids(P, n_sets, 1.0, seed=seed)
    if name == "mixed":
        return rpk.synth.make_set_ids(P, n_sets, 0.5, seed=seed)
    return (n_sets + np.arange(P) % 9).astype(np.uint16)  # "oob": only ids of sets that do not exist


@pytest.mark.gpu
@pytest.mark.parametrize("n_sets", [1, 3, 40])
@pytest.mark.parametrize("flavour", list(FLAVOURS))
def test_parity_matrix(engine, flavour, n_sets):
    G = 3000
    offers = rpk.synth.make_offers(G, seed=17 + n_sets, **FLAVOURS[flavour])
    members = rpk.synth.make_offer_sets(G, n_sets, seed=5 + n_sets)
    if n_sets == 1:
        members[0] = rpk.synth.make_offer_sets(G, 4, seed=5)[3]  # one 10 % set (the generator's first set is empty)
    pods = rpk.synth.make_pods(max(P_SIZES), seed=23)
    pods["max_price"][::3] = 4.0  # longer top-5 lists inside the sets
    want = {}
    for mix in ("all", "none", "mixed", "oob"):
        set_id = row_mix(mix, max(P_SIZES), n_sets, seed=31 + n_sets)
        want[mix] = (set_id, sr.oracle_select_sets(offers, pods, members, set_id))
    assert (want["mixed"][1][0] >= 0).any() and (want["none"][1][0] < 0).any()
    for force in FORCES:
        upload_forced(engine, offers, members, force)
        for mix, (set_id, (ob, ot)) in want.items():
            for P in P_SIZES:
                sub = {k: v[:P] for k, v in pods.items()}
                best, t5 = engine.select_sets(sub, np.ascontiguousarray(set_id[:P]), want_top5=True)
                tag = f"[{flavour} n_sets={n_sets} {force} {mix} P={P}]"
                assert np.array_equal(best, ob[:P]), f"{tag} best differs at rows {np.nonzero(best != ob[:P])[0][:10]}"
                assert np.array_equal(t5, ot[:P]), f"{tag} top5 differs at rows {np.nonzero((t5 != ot[:P]).any(axis=1))[0][:10]}"
    upload_forced(engine, offers, members, None)


@pytest.mark.gpu
def test_kat_through_abi(engine):
    offers, pods, members, set_id, want = kat_sets()
    engine.upload_offers(offers)
    engine.upload_offer_sets(members)
    best, t5 = engine.select_sets(pods, set_id, want_top5=True)
    assert np.array_equal(t5, want) and np.array_equal(best, want[:, 0])


@pytest.mark.gpu
def test_empty_and_full_sets_and_set_sizes(engine):
    """Set sizes from empty through one offer to the whole table, on a table above one 16k-offer segment."""
    G, P = 20_000, 30_000
    offers = rpk.synth.make_offers(G, correlated=True, seed=3)
    members = rpk.synth.make_offer_sets(G, 6, seed=3)  # empty, one, 1 %, 10 %, 50 %, all
    pods = rpk.synth.make_pods(P, seed=4)
    set_id = rpk.synth.make_set_ids(P, 6, 0.8, seed=4)
    engine.upload_offers(offers)
    engine.upload_offer_sets(members)
    best, t5 = engine.select_sets(pods, set_id, want_top5=True)
    ob, ot = sr.oracle_select_sets(offers, pods, members, set_id)
    assert np.array_equal(best, ob) and np.array_equal(t5, ot)
    assert (best[set_id == 0] == -1).all()
    full = set_id == 5  # the full set is the unrestricted table
    b_all, _ = engine.select({k: np.ascontiguousarray(v[full]) for k, v in pods.items()})
    assert np.array_equal(best[full], b_all)


@pytest.mark.gpu
def test_device_entry_matches_host(engine):
    import torch

    G, P = 5000, 50_000
    offers = rpk.synth.make_offers(G, correlated=True, seed=8)
    members = rpk.synth.make_offer_sets(G, 9, seed=8)
    pods = rpk.synth.make_pods(P, seed=9)
    set_id = rpk.synth.make_set_ids(P, 9, 0.6, seed=9)
    engine.upload_offers(offers)
    engine.upload_offer_sets(members)
    hb, ht = engine.select_sets(pods, set_id, want_top5=True)
    dev = {k: torch.from_numpy(v).cuda() for k, v in pods.items()}
    d_set = torch.from_numpy(set_id.view(np.int16)).cuda()
    d_best = torch.full((P,), -7, dtype=torch.int32, device="cuda")
    d_top5 = torch.full((P * 5,), -7, dtype=torch.int32, device="cuda")
    engine.select_sets_device(dev, d_set, d_best, d_top5)
    torch.cuda.synchronize()
    assert np.array_equal(d_best.cpu().numpy(), hb) and np.array_equal(d_top5.cpu().numpy().reshape(P, 5), ht)
    # NULL set_id: the plain select's result, without touching sets
    engine.select_sets_device(dev, None, d_best, d_top5)
    torch.cuda.synchronize()
    sb, stp = engine.select(pods, want_top5=True)
    assert np.array_equal(d_best.cpu().numpy(), sb) and np.array_equal(d_top5.cpu().numpy().reshape(P, 5), stp)


@pytest.mark.gpu
def test_null_set_id_is_select(engine):
    offers = rpk.synth.make_offers(4000, correlated=True, seed=12)
    engine.upload_offers(offers)
    for P in (100, 20_000, 150_000):
        pods = rpk.synth.make_pods(P, seed=P)
        sb, st5 = engine.select(pods, want_top5=True)
        b, t5 = engine.select_sets(pods, None, want_top5=True)  # no sets uploaded for this table: not needed
        assert np.array_equal(b, sb) and np.array_equal(t5, st5)


@pytest.mark.gpu
def test_select_and_resident_vector_unchanged_by_sets(engine):
    import torch

    peer = __import__("importlib").import_module("k8s-runpod-kubelet_b200.peer")
    G, P = 6000, 60_000
    offers = rpk.synth.make_offers(G, correlated=True, seed=21)
    pods = rpk.synth.make_pods(P, seed=21)
    engine.upload_offers(offers)
    b0, t0 = engine.select(pods, want_top5=True)
    resident = peer.as_int32_tensor(engine.best_device_ptr(0), P, torch.device("cuda", 0)).clone()
    assert np.array_equal(resident.cpu().numpy(), b0)
    engine.upload_offer_sets(rpk.synth.make_offer_sets(G, 12, seed=21))
    engine.select_sets(pods, rpk.synth.make_set_ids(P, 12, 0.9, seed=21), want_top5=True)
    now = peer.as_int32_tensor(engine.best_device_ptr(0), P, torch.device("cuda", 0))
    assert torch.equal(now, resident)
    b1, t1 = engine.select(pods, want_top5=True)
    assert np.array_equal(b0, b1) and np.array_equal(t0, t1)


@pytest.mark.gpu
def test_call_order_and_argument_errors():
    E = rpk._ffi
    offers = rpk.synth.make_offers(500, seed=2)
    pods = rpk.synth.make_pods(64, seed=2)
    ids = rpk.synth.make_set_ids(64, 3, 0.5, seed=2)
    with rpk.Engine(1) as eng:
        with pytest.raises(rpk.RpkError) as ei:
            eng.upload_offer_sets(np.ones((1, 500), bool))
        assert ei.value.code == E.RPK_ESTATE  # no table yet
        eng.upload_offers(offers)
        with pytest.raises(rpk.RpkError) as ei:
            eng.select_sets(pods, ids)
        assert ei.value.code == E.RPK_ESTATE  # no sets yet
        with pytest.raises(rpk.RpkError) as ei:
            eng.upload_offer_sets(np.ones((257, 500), bool))
        assert ei.value.code == E.RPK_EINVAL
        with pytest.raises(rpk.RpkError) as ei:
            eng.upload_offer_sets(np.ones((2, 499), bool))
        assert ei.value.code == E.RPK_EINVAL  # G differs from the table's
        members = rpk.synth.make_offer_sets(500, 3, seed=2)
        members[0, :50] = True
        eng.upload_offer_sets(members)
        b, t = eng.select_sets(pods, ids, want_top5=True)
        ob, ot = sr.oracle_select_sets(offers, pods, members, ids)
        assert np.array_equal(b, ob) and np.array_equal(t, ot)
        eng.upload_offers(offers)  # a new table makes the sets stale
        with pytest.raises(rpk.RpkError) as ei:
            eng.select_sets(pods, ids)
        assert ei.value.code == E.RPK_ESTATE
        eng.upload_offer_sets(np.zeros((0, 500), bool))  # n_sets = 0: no sets, every restricted row gets nothing
        b, _ = eng.select_sets(pods, ids)
        sb, _ = eng.select(pods)
        assert (b[ids != ALL] == -1).all() and np.array_equal(b[ids == ALL], sb[ids == ALL])
        assert eng.select_sets({"req_mem_gb": np.zeros(0, np.int32)}, np.zeros(0, np.uint16))[0].size == 0


@pytest.mark.gpu
def test_offer_scores_count_the_evaluated_grid():
    G, P = 1000, 5000
    offers = rpk.synth.make_offers(G, seed=6)
    members = rpk.synth.make_offer_sets(G, 6, seed=6)
    pods = rpk.synth.make_pods(P, seed=6)
    ids = rpk.synth.make_set_ids(P, 6, 0.7, seed=6)
    with rpk.Engine(1) as eng:
        eng.upload_offers(offers)
        eng.upload_offer_sets(members)
        s0 = eng.stats()
        eng.select_sets(pods, ids)
        s1 = eng.stats()
    sizes = members.sum(axis=1)
    want = sum(int((ids == s).sum()) * int(sizes[s]) for s in range(6)) + int((ids == ALL).sum()) * G
    assert s1["offer_scores"] - s0["offer_scores"] == want
    assert s1["select_calls"] - s0["select_calls"] == 1


@pytest.mark.gpu
def test_two_gpu_ctx():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    G, P = 8000, 90_001
    offers = rpk.synth.make_offers(G, correlated=True, seed=14)
    members = rpk.synth.make_offer_sets(G, 10, seed=14)
    pods = rpk.synth.make_pods(P, seed=14)
    ids = rpk.synth.make_set_ids(P, 10, 0.5, seed=14)
    with rpk.Engine(2) as eng:
        eng.upload_offers(offers)
        eng.upload_offer_sets(members)
        b, t = eng.select_sets(pods, ids, want_top5=True)
    ob, ot = sr.oracle_select_sets(offers, pods, members, ids)
    assert np.array_equal(b, ob) and np.array_equal(t, ot)
