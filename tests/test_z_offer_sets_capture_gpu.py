"""rpk_select_sets_device with set ids synchronises its stream once (per-set row counts), so it cannot be captured in a
CUDA graph: on a capturing stream it must refuse with RPK_ESTATE before enqueuing anything, leaving the capture valid.
(Sorts after the parity suites, like the other graph-capture tests.)"""
import numpy as np
import pytest

import rpk

pytestmark = pytest.mark.gpu


def test_capturing_stream_is_refused_and_capture_stays_valid(engine):
    import torch

    G, P = 2000, 3000
    offers = rpk.synth.make_offers(G, correlated=True, seed=41)
    engine.upload_offers(offers)
    engine.upload_offer_sets(rpk.synth.make_offer_sets(G, 4, seed=41))
    pods = rpk.synth.make_pods(P, seed=41)
    ids = rpk.synth.make_set_ids(P, 4, 0.5, seed=41)
    d = {k: torch.from_numpy(v).cuda() for k, v in pods.items()}
    d_ids = torch.from_numpy(ids.view(np.int16)).cuda()
    d_best = torch.full((P,), -7, dtype=torch.int32, device="cuda")
    x = torch.zeros(16, device="cuda")
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    err = None
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            x.add_(1)
            try:
                engine.select_sets_device(d, d_ids, d_best, stream=s.cuda_stream)
            except rpk.RpkError as e:
                err = e
            x.add_(1)
    assert err is not None and err.code == rpk._ffi.RPK_ESTATE and "captured" in str(err)
    g.replay()
    torch.cuda.synchronize()
    assert float(x[0]) == 2.0  # the capture was not invalidated
    assert int((d_best != -7).sum()) == 0  # nothing was enqueued
    # outside a capture the same call works
    engine.select_sets_device(d, d_ids, d_best)
    torch.cuda.synchronize()
    hb, _ = engine.select_sets(pods, ids)
    assert np.array_equal(d_best.cpu().numpy(), hb)
