"""Runs the C++ tests of runpod.io/gpu-type-ids in the Provider mirror (k8s-runpod-kubelet_b200/host/sets_test.cc):
the annotation parser and column producer on the CPU, DeployBatch through rpk_select_sets on the GPU."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "k8s-runpod-kubelet_b200", "host")
BIN = os.path.join(HOST, "sets_test")


def run(arg):
    if not os.path.exists(BIN):
        subprocess.check_call(["make", "-C", HOST, "-s"])
    out = subprocess.run([BIN, arg], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout[-4000:] + out.stderr[-2000:]
    assert out.stdout.strip().splitlines()[-1].startswith("ok:")
    return out.stdout


def test_gpu_type_ids_parser_and_columns():
    """strings.Split + TrimSpace like runpod.io/datacenter-ids; pod -> owner Job fallback; empty elements kept"""
    assert "0 failed" in run("--cpu")


@pytest.mark.gpu
def test_deploy_batch_restricts_to_listed_gpu_types():
    """restricted pods get only listed types cheapest first, Job fallback, unknown-only lists deploy nothing, a batch
    without the annotation issues the plain rpk_select, resident sets reused, more than 256 lists split over calls"""
    out = run("--gpu")
    assert "(gpu)" in out and "0 failed" in out
