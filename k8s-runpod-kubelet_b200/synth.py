"""Deterministic synthetic pod / offer / status tables (SURVEY.md 8d).

``r(col, row) = splitmix64(seed + (col << 40) + row)``, seed ``0x52504B31``
("RPK1").  Everything is a pure function of (seed, row), so any slice of a table
can be generated on any rank without generating the rest -- the pod-row shards of
the multi-GPU bench rely on this.

Offer rows follow ``GPUType`` (reference runpod_client.go:83-95); pod rows are the
(minRAMPerGPU, cloudType, maxPrice) triple that parameterises ``GetGPUTypes``
(runpod_client.go:1261-1281) plus the two extension columns; status rows are the
(``InstanceInfo.Status``, ``InstanceInfo.PortsExposed``) pair compared by the sweep
(kubelet.go:870-871).
"""
from __future__ import annotations

import numpy as np

SEED = 0x52504B31
MEM_SET = np.array([8, 12, 16, 20, 24, 32, 40, 48, 80, 94, 141, 180, 192], np.int32)
VCPU_SET = np.array([4, 8, 16, 32, 64, 128], np.int32)
RAM_SET = np.array([16, 32, 64, 128, 256, 512], np.int32)
REQ_MEM_SET = np.array([2, 8, 16, 24, 40, 48, 80], np.int32)
MAX_PRICE_SET = np.array([0.25, 1.0, 2.0, 4.0], np.float64)
# PodStatus enum, runpod_client.go:55-64, with the sweep weights of SURVEY.md 8d
STATUS_SET = [b"RUNNING", b"STARTING", b"EXITED", b"TERMINATING", b"TERMINATED", b"NOT_FOUND"]
STATUS_WEIGHTS = np.array([700, 150, 80, 30, 30, 10], np.int64)  # per-mille
UNKNOWN_STATUS = [b"PAUSED", b"CREATED", b"RESTARTING", b"DEAD"]  # "arbitrary unknown strings", kubelet.go:1967
DEFAULT_MAX_PRICE = 0.5  # runpod_client.go:48
DEFAULT_REQ_MEM = 16     # runpod_client.go:1182


def splitmix64(x: np.ndarray) -> np.ndarray:
    with np.errstate(over="ignore"):
        z = x.astype(np.uint64) + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def r(col: int, rows: np.ndarray, seed: int = SEED) -> np.ndarray:
    with np.errstate(over="ignore"):
        return splitmix64(np.uint64(seed) + (np.uint64(col) << np.uint64(40)) + rows.astype(np.uint64))


def _pick(rnd: np.ndarray, table: np.ndarray) -> np.ndarray:
    return table[(rnd % np.uint64(len(table))).astype(np.int64)]


def make_offers(G: int, seed: int = SEED, tie_free: bool = False, with_ext: bool = True, correlated: bool = False) -> dict:
    """G offers.  ``tie_free``: distinct prices (result independent of Go's unstable sort.Slice tie
    order).  ``with_ext=False``: no vcpu/ram columns, exactly the reference's GPUType.  ``correlated``:
    price grows with memory/vcpu/ram (plus noise), so the argmin differs from pod to pod instead of
    collapsing onto the few globally cheapest offers -- the discriminating table for parity tests."""
    rows = np.arange(G, dtype=np.uint64)
    mem = _pick(r(0, rows, seed), MEM_SET)
    secure_cloud = (r(1, rows, seed) % np.uint64(100)) < np.uint64(75)
    community_cloud = (r(2, rows, seed) % np.uint64(100)) < np.uint64(50)
    if tie_free:
        # rank of a random key = a permutation of 0..G-1 -> G distinct prices in (0, 4]
        perm = np.argsort(np.argsort(r(3, rows, seed), kind="stable"), kind="stable").astype(np.float64)
        secure = (perm + 1.0) * 4.0 / float(G)
        community = 0.6 * secure
    else:
        cents = (np.uint64(5) + r(3, rows, seed) % np.uint64(395)).astype(np.int64)
        if correlated:
            rk = lambda col, tab: np.searchsorted(tab, _pick(r(col, rows, seed), tab)).astype(np.int64)  # noqa: E731
            cents = 5 + rk(0, MEM_SET) * 22 + rk(5, VCPU_SET) * 9 + rk(6, RAM_SET) * 9 + (r(3, rows, seed) % np.uint64(48)).astype(np.int64)
        cents[(r(4, rows, seed) % np.uint64(100)) < np.uint64(2)] = 0  # exercises `price > 0`
        secure = cents.astype(np.float64) / 100.0  # float64(c)/100.0, what Go would hold after JSON decode
        community = ((cents * 6) // 10).astype(np.float64) / 100.0
    out = {
        "mem_gb": mem.astype(np.int32),
        "secure_price": np.ascontiguousarray(secure, np.float64),
        "community_price": np.ascontiguousarray(community, np.float64),
        "flags": (secure_cloud.astype(np.uint8) | (community_cloud.astype(np.uint8) << 1)).astype(np.uint8),
        "vcpu": None,
        "ram_gb": None,
    }
    if with_ext:
        out["vcpu"] = _pick(r(5, rows, seed), VCPU_SET).astype(np.int32)
        out["ram_gb"] = _pick(r(6, rows, seed), RAM_SET).astype(np.int32)
    return out


def make_pods(P: int, seed: int = SEED, reference_exact: bool = False, row0: int = 0) -> dict:
    """Pod rows [row0, row0+P).  ``reference_exact``: max_price = 0.5 for all, vcpu = ram = 0 -- the only
    profile with true reference semantics (runpod_client.go:1281 passes the constant)."""
    rows = np.arange(row0, row0 + P, dtype=np.uint64)
    req_mem = _pick(r(17, rows, seed), REQ_MEM_SET)
    req_mem[(r(16, rows, seed) % np.uint64(100)) < np.uint64(40)] = DEFAULT_REQ_MEM
    cloud = ((r(18, rows, seed) % np.uint64(100)) >= np.uint64(90)).astype(np.uint8)  # 90 % SECURE(0)
    max_price = _pick(r(20, rows, seed), MAX_PRICE_SET)
    max_price[(r(19, rows, seed) % np.uint64(100)) < np.uint64(80)] = DEFAULT_MAX_PRICE
    req_vcpu = _pick(r(22, rows, seed), VCPU_SET)
    req_vcpu[(r(21, rows, seed) % np.uint64(100)) < np.uint64(70)] = 0
    req_ram = _pick(r(24, rows, seed), RAM_SET)
    req_ram[(r(23, rows, seed) % np.uint64(100)) < np.uint64(70)] = 0
    if reference_exact:
        max_price[:] = DEFAULT_MAX_PRICE
        req_vcpu[:] = 0
        req_ram[:] = 0
    return {
        "req_mem_gb": req_mem.astype(np.int32),
        "req_vcpu": req_vcpu.astype(np.int32),
        "req_ram_gb": req_ram.astype(np.int32),
        "max_price": np.ascontiguousarray(max_price, np.float64),
        "cloud": cloud,
    }


SET_ALL = 0xFFFF  # RPK_SET_ALL: an unrestricted row
# offer-set sizes, cycled over the set index: empty, one offer, 1 %, 10 %, 50 %, every offer
SET_FRACTIONS = (0.0, None, 0.01, 0.10, 0.50, 1.0)


def make_offer_sets(G: int, n_sets: int, seed: int = SEED) -> np.ndarray:
    """bool ``(n_sets, G)`` membership of ``n_sets`` offer sets (the ``runpod.io/gpu-type-ids`` lists of a batch).
    Set s has the size class ``SET_FRACTIONS[s % 6]``: empty, a single offer (drawn per set), or each offer
    independently with that probability (all offers for 1.0)."""
    rows = np.arange(G, dtype=np.uint64)
    out = np.zeros((n_sets, G), bool)
    for s in range(n_sets):
        f = SET_FRACTIONS[s % len(SET_FRACTIONS)]
        if f is None:
            if G:
                out[s, int(r(300 + s, np.zeros(1, np.uint64), seed)[0] % np.uint64(G))] = True
        elif f >= 1.0:
            out[s] = True
        elif f > 0.0:
            out[s] = (r(300 + s, rows, seed) % np.uint64(1_000_000)) < np.uint64(int(f * 1_000_000))
    return out


def make_set_ids(P: int, n_sets: int, frac_restricted: float, seed: int = SEED, row0: int = 0) -> np.ndarray:
    """uint16 set id per pod row [row0, row0+P): a row is restricted with probability ``frac_restricted`` (to a set drawn
    uniformly), else ``SET_ALL``; 1 % of the restricted rows carry an id >= n_sets (no such set: nothing feasible)."""
    rows = np.arange(row0, row0 + P, dtype=np.uint64)
    restricted = (r(50, rows, seed) % np.uint64(1_000_000)) < np.uint64(int(frac_restricted * 1_000_000))
    ids = (r(51, rows, seed) % np.uint64(max(n_sets, 1))).astype(np.int64)
    unknown = ((r(52, rows, seed) % np.uint64(100)) < np.uint64(1)) | (n_sets == 0)
    ids = np.where(unknown, n_sets + (r(53, rows, seed) % np.uint64(7)).astype(np.int64), ids)
    return np.where(restricted, ids, SET_ALL).astype(np.uint16)


def encode_record(status: bytes, ports_exposed: bool, stride: int = 32, msg_error: bool = False) -> np.ndarray:
    """Canonical slot ``[b0][status][0x00][ports][pad]``, b0 = len | flag << 7, len = len(status)+2 <= min(stride-1, 127);
    the flag bit ("statusMessage contains error/fail", kubelet.go:1907) is not a compared field and is not hashed."""
    body = status + b"\x00" + (b"\x01" if ports_exposed else b"\x00")
    if len(body) > stride - 1 or len(body) > 127:
        raise ValueError("status too long for the record slot")
    rec = np.zeros(stride, np.uint8)
    rec[0] = len(body) | (0x80 if msg_error else 0)
    rec[1 : 1 + len(body)] = np.frombuffer(body, np.uint8)
    return rec


_STATUS_LUT_CACHE: dict = {}


def _status_lut(stride: int) -> np.ndarray:
    if stride not in _STATUS_LUT_CACHE:
        names = STATUS_SET + UNKNOWN_STATUS
        lut = np.zeros((len(names), 2, 2, stride), np.uint8)
        for i, s in enumerate(names):
            for p in (0, 1):
                for f in (0, 1):
                    lut[i, p, f] = encode_record(s, bool(p), stride, bool(f))
        _STATUS_LUT_CACHE[stride] = lut
    return _STATUS_LUT_CACHE[stride]


def _status_draw(rnd: np.ndarray, rnd_unknown: np.ndarray) -> np.ndarray:
    cum = np.cumsum(STATUS_WEIGHTS)
    sid = np.searchsorted(cum, (rnd % np.uint64(1000)).astype(np.int64), side="right").astype(np.int64)
    unk = (rnd_unknown % np.uint64(1000)) < np.uint64(1)  # 0.1 % unknown strings
    sid[unk] = len(STATUS_SET) + (rnd_unknown[unk] >> np.uint64(20)).astype(np.int64) % len(UNKNOWN_STATUS)
    return sid


def make_status_records(N: int, sweep: int = 0, mutate_frac: float = 0.0, seed: int = SEED, stride: int = 32,
                        row0: int = 0) -> np.ndarray:
    """Record table for sweep number ``sweep``.  Sweep 0 is the base state; in sweep s>0 a row takes a
    fresh draw iff its per-sweep coin < mutate_frac, else it keeps its sweep-0 state (so the changed
    set between consecutive sweeps is non-trivial but reproducible)."""
    rows = np.arange(row0, row0 + N, dtype=np.uint64)
    sid = _status_draw(r(32, rows, seed), r(33, rows, seed))
    ports = (r(34, rows, seed) % np.uint64(100)) < np.uint64(85)
    if sweep > 0 and mutate_frac > 0.0:
        coin = (r(40 + 4 * sweep, rows, seed) % np.uint64(1_000_000)).astype(np.float64) / 1e6
        m = coin < mutate_frac
        sid2 = _status_draw(r(41 + 4 * sweep, rows, seed), r(42 + 4 * sweep, rows, seed))
        ports2 = (r(43 + 4 * sweep, rows, seed) % np.uint64(100)) < np.uint64(85)
        sid = np.where(m, sid2, sid)
        ports = np.where(m, ports2, ports)
    # the message flag is drawn per (row, sweep): it moves between sweeps on rows whose (status, ports) do not, and must
    # never make a row report (it is not a compared field)
    flag = (r(200 + sweep, rows, seed) % np.uint64(100)) < np.uint64(30)
    return np.ascontiguousarray(_status_lut(stride)[sid, ports.astype(np.int64), flag.astype(np.int64)])
