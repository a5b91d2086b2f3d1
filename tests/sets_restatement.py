"""Two independent restatements of selection restricted to offer sets (``runpod.io/gpu-type-ids``).

``oracle_select_sets`` states the contract literally -- a restricted pod gets what ``GetGPUTypes``
(runpod_client.go:465-509) returns when the GraphQL answer holds only the set's members, in table order -- by running
the C oracle on each set's sub-table and mapping the sub-table indices back to table indices.
``np_select_sets`` is the filter-loop reading instead: the whole table, one more membership test in the predicate
of :478.  The two must agree on every input.
"""
import numpy as np

import np_restatement as npr
import oracle

SET_ALL = 0xFFFF


def sub_table(offers, idx):
    return {k: (np.ascontiguousarray(v[idx]) if v is not None else None) for k, v in offers.items()}


def oracle_select_sets(offers, pods, members, set_id, n_threads=8):
    """-> (best[P], top5[P,5]).  members: bool (n_sets, G); set_id: uint16[P] or None (= every row SET_ALL)."""
    P = int(pods["req_mem_gb"].shape[0])
    if set_id is None:
        return oracle.select(offers, pods, want_top5=True, n_threads=n_threads)
    n_sets = members.shape[0]
    best = np.full(P, -1, np.int32)
    top5 = np.full((P, 5), -1, np.int32)
    for sid in np.unique(set_id):
        rows = np.nonzero(set_id == sid)[0]
        sub_pods = {k: (np.ascontiguousarray(v[rows]) if v is not None else None) for k, v in pods.items()}
        if sid == SET_ALL:
            b, t = oracle.select(offers, sub_pods, want_top5=True, n_threads=n_threads)
        elif sid < n_sets:
            idx = np.nonzero(members[sid])[0]
            b, t = oracle.select(sub_table(offers, idx), sub_pods, want_top5=True, n_threads=n_threads)
            b = np.where(b >= 0, idx[np.maximum(b, 0)] if idx.size else -1, -1).astype(np.int32)
            t = np.where(t >= 0, idx[np.maximum(t, 0)] if idx.size else -1, -1).astype(np.int32)
        else:  # no such set: nothing feasible
            continue
        best[rows] = b
        top5[rows] = t
    return best, top5


def np_select_sets(offers, pods, members, set_id):
    """runpod_client.go:465-509 per pod with ``member(g)`` added to the filter (numpy, vectorised over offers)."""
    P = int(pods["req_mem_gb"].shape[0])
    G = int(offers["mem_gb"].shape[0])
    n_sets = members.shape[0]
    best = np.full(P, -1, np.int32)
    top5 = np.full((P, 5), -1, np.int32)
    names = {0: "SECURE", 1: "COMMUNITY"}
    for p in range(P):
        sid = SET_ALL if set_id is None else int(set_id[p])
        if sid == SET_ALL:
            member = np.ones(G, bool)
        elif sid < n_sets:
            member = members[sid]
        else:
            continue
        cloud = names.get(int(pods["cloud"][p]) if pods.get("cloud") is not None else 0, "OTHER")
        if cloud == "SECURE":
            price, ok = offers["secure_price"], (offers["flags"] & 1).astype(bool)
        elif cloud == "COMMUNITY":
            price, ok = offers["community_price"], (offers["flags"] & 2).astype(bool)
        else:
            continue
        mp = float(pods["max_price"][p]) if pods.get("max_price") is not None else 0.5
        rv = int(pods["req_vcpu"][p]) if pods.get("req_vcpu") is not None else 0
        rr = int(pods["req_ram_gb"][p]) if pods.get("req_ram_gb") is not None else 0
        vcpu = np.zeros(G, np.int64) if offers.get("vcpu") is None else offers["vcpu"].astype(np.int64)
        ram = np.zeros(G, np.int64) if offers.get("ram_gb") is None else offers["ram_gb"].astype(np.int64)
        with np.errstate(invalid="ignore"):
            keep = member & ok & (price > 0) & (price < mp) & (offers["mem_gb"].astype(np.int64) >= int(pods["req_mem_gb"][p]))
        keep &= (vcpu >= rv) & (ram >= rr)
        idx = np.nonzero(keep)[0]
        ids = idx[np.argsort(price[idx], kind="stable")][:5]
        top5[p, : len(ids)] = ids
        if len(ids):
            best[p] = ids[0]
    return best, top5


def unrestricted_equals_select(offers, pods):
    """set_id = SET_ALL everywhere is rpk_select's contract, row for row (used by the CPU tests)."""
    P = int(pods["req_mem_gb"].shape[0])
    b0, t0 = oracle.select(offers, pods, want_top5=True)
    b1, t1 = oracle_select_sets(offers, pods, np.zeros((0, len(offers["mem_gb"])), bool), np.full(P, SET_ALL, np.uint16))
    b2, t2 = npr.select(offers, pods)
    return np.array_equal(b0, b1) and np.array_equal(t0, t1) and np.array_equal(b0, b2) and np.array_equal(t0, t2)
