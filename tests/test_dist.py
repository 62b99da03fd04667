"""N>1 path: world_size-2 gloo test on CPU (host logic + DP identity), torchrun NCCL test on >= 2 GPUs."""
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


def _torchrun(mode, nproc, port, env=None):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(HERE, "dist_worker.py"), mode]
    return subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, **(env or {})))


def test_data_parallel_identity_gloo_world2():
    r = _torchrun("gloo", 2, 29611)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]


@pytest.mark.gpu
@pytest.mark.parametrize("exchange,env", [("peer-memory", {}), ("nccl", {"TCR_P2P": "0"})])
def test_gradient_exchange_matches_oracle(exchange, env):
    """Both exchanges of the data-parallel step: the update kernel summing the ranks' gradients from peer memory (default on
    one node) and the ncclAllReduce fallback; 4 steps, averaged gradient vs the oracle's shard-wise mean, identical replicas."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = _torchrun("nccl", min(torch.cuda.device_count(), 8), 29612 if exchange == "nccl" else 29613, env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "replicas bit-identical" in r.stdout and f"exchange={exchange}" in r.stdout, r.stdout[-500:]


@pytest.mark.gpu
def test_sync_bn_flag_equals_single_device_global_batch():
    """tcr_comm_set_sync_bn (parity-test flag, SURVEY.md 8(e)): with BatchNorm statistics all-reduced over the ranks, every rank's
    step equals the oracle's single-device step on the concatenated global batch."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = _torchrun("syncbn", 2, 29614)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "syncbn world=2" in r.stdout, r.stdout[-500:]


@pytest.mark.gpu
def test_trainer_data_parallel_two_ranks_checkpoints(tmp_path):
    """train_audio.py --data_parallel under torchrun (2 GPUs, synthetic data): the loop runs to the end with a checkpoint every 5
    steps written by rank 0 only (every rank used to write the same tmp path and die at the first save), every rank leaves the
    loop at the same global step, and the checkpoint loads."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(HERE)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29615", os.path.join(root, "tc-resnet_b200", "train_audio.py"),
           "--dataset_path", "synthetic:1024", "--dataset_split_name", "train", "--output_name", "output/softmax", "--num_classes", "12",
           "--train_dir", str(tmp_path), "--augmentation_method", "anchored_slice_or_pad_with_shift", "--preprocess_method", "mfcc",
           "--num_mfccs", "40", "--clip_duration_ms", "1000", "--window_size_ms", "40", "--window_stride_ms", "20", "--batch_size", "64",
           "--boundaries", "1000", "--max_step_from_restore", "23", "--lr_list", "0.1", "0.01", "--absolute_schedule",
           "--no-boundaries_epoch", "--step_save_checkpoint", "5", "--step_evaluation", "100000", "--step_save_summaries", "100000",
           "--step_save_first_n_summaries", "0", "--max_to_keep", "3", "--optimizer", "mom", "--momentum", "0.9", "--data_parallel",
           "TCResNet8Model", "--weight_decay", "0.001", "--width_multiplier", "1.0"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    sys.path.insert(0, os.path.join(root, "tc-resnet_b200"))
    import tcresnet_b200  # noqa: F401
    from tcresnet_b200.common import checkpoint as ckpt
    latest = ckpt.latest_checkpoint(str(tmp_path))
    assert latest is not None and latest.rstrip("/").endswith("-23"), latest
    values = ckpt.load(latest)
    assert len(values) > 10 and int(values["global_step"]) == 23
    leftovers = [f for f in os.listdir(tmp_path) if f.startswith(".") and ".tmp" in f]
    assert not leftovers, leftovers
