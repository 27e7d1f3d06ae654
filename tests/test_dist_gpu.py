"""-m gpu: sharded ID-only path == single-GPU engine (world 1 always; world 2 over NCCL when two GPUs are visible)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def test_sharded_world1_equals_engine():
    r = subprocess.run([sys.executable, os.path.join(HERE, "dist_gpu_check.py")], capture_output=True, text=True, timeout=300)
    assert "DIST_CHECK_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_sharded_demand_world1_equals_engine():
    """demand-driven step (last layer on the batch's neighbourhood only, row-sparse user gradient) == the dense single-GPU engine"""
    r = subprocess.run([sys.executable, os.path.join(HERE, "dist_gpu_check.py")], capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, LLMREC_DIST_DEMAND="1"))
    assert "DIST_CHECK_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_sharded_demand_world2_equals_engine():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29521", os.path.join(HERE, "dist_gpu_check.py")], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, LLMREC_DIST_DEMAND="1"))
    assert "DIST_CHECK_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_sharded_world2_equals_engine():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29517", os.path.join(HERE, "dist_gpu_check.py")], capture_output=True, text=True, timeout=600)
    assert "DIST_CHECK_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


# ---- promoted from the round-1 "experimental" gate after passing on 2 x B200 (round 2, gpurun_out/r2b) -----------------------------
def test_item_sharded_exchange_world2_equals_engine():
    """dist.ShardedHotPath(item_sharded=True): reduce-scatter / row-local / all-gather form == single-GPU engine."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    here = HERE
    env = dict(os.environ, LLMREC_DIST_ITEM_SHARDED="1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29519", os.path.join(here, "dist_gpu_check.py")], capture_output=True, text=True, timeout=600, env=env)
    assert "DIST_CHECK_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.parametrize("world", [1, 2])
def test_sharded_feature_path_equals_engine(world):
    """dist_feat.ShardedFeatureHotPath (side features, users and item tables sharded) == engine.HotPath."""
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    here = HERE
    cmd = [sys.executable, os.path.join(here, "dist_feat_gpu_check.py")] if world == 1 else \
        [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
         "--master-port", "29523", os.path.join(here, "dist_feat_gpu_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert "DIST_FEAT_CHECK_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
