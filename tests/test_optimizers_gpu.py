"""Adam / RMSProp / EMA in the fused training step on the B200: the update against the fp64 rule on the reported gradient at the
flagship shapes in every TCR_RESIDENT mode, bitwise determinism, the host-feed and CUDA-graph paths, checkpoint resume, the
trainer CLI with --optimizer adam, and two GPUs."""
import os
import shlex
import subprocess
import sys

import numpy as np
import pytest

from optim_cases import run_optimizer_case

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def backend():
    from tcr_harness import TorchBackend
    return TorchBackend()


RULES = [("mom", False), ("adam", False), ("rmsprop", False), ("adam", True)]


@pytest.mark.parametrize("mode", ["0", "1", "2", "3"])
@pytest.mark.parametrize("kind,ema", RULES, ids=["mom", "adam", "rmsprop", "adam-ema"])
@pytest.mark.parametrize("shape", [dict(model="TCResNet8", wm=1.0, n=512), dict(model="TCResNet14", wm=1.5, n=1024)],
                         ids=["r8-n512", "r14x1.5-n1024"])
def test_update_matches_the_rule_on_the_reported_gradient(backend, monkeypatch, mode, kind, ema, shape):
    """5 steps; the first step's gradient against the fp64 oracle (with the CUDA path's ReLU decisions), every step's update
    against the fp64 rule carried forward on the reported gradients; then apply_update = 0 changes nothing."""
    monkeypatch.setenv("TCR_RESIDENT", mode)
    run_optimizer_case(backend, kind, ema, steps=5, grad_steps=(0,), force_masks=True, **shape)


def _engine_and_batches(n=256, k=3):
    import torch
    from oracle import tcr_oracle as O
    from tcresnet_b200.engine import Engine
    eng = Engine(max_batch=n)
    wavs, hots = [], []
    for i in range(k):
        w, h = O.synthetic_batch(n, seed_wav=100 + i, seed_label=200 + i)
        wavs.append(torch.from_numpy(w))
        hots.append(torch.from_numpy(h))
    return eng, wavs, hots


def _state_tensors(params, st, moving):
    out = [params, moving, st.slots] + [t for t in (st.slots2, st.scalars, st.ema) if t is not None]
    return [t.clone() for t in out]


def test_adam_step_is_bitwise_deterministic():
    import torch
    from tcresnet_b200.engine import Optimizer
    eng, wavs, hots = _engine_and_batches()
    opt = Optimizer.adam(ema_decay=0.999)
    runs = []
    for _ in range(2):
        p, _, m = eng.new_variables(seed=3)
        st = eng.new_optimizer_state(opt, p)
        for i in range(3):
            eng.train_step(wavs[i].cuda(), hots[i].cuda(), p, None, m, 0.01, weight_decay=1e-3, dropout_seed=i, optimizer=opt, state=st)
        torch.cuda.synchronize()
        runs.append(_state_tensors(p, st, m))
    assert all(torch.equal(a, b) for a, b in zip(*runs))
    assert runs[0][4].tolist() == [np.float32(np.float32(np.float32(0.9) * np.float32(0.9)) * np.float32(0.9)) * np.float32(0.9),
                                   np.float32(np.float32(np.float32(0.999) * np.float32(0.999)) * np.float32(0.999)) * np.float32(0.999)]
    eng.close()


@pytest.mark.parametrize("kind", ["adam", "rmsprop"])
def test_host_feed_equals_device_steps_bitwise(kind):
    """tcr_train_step_host copies the step arguments: the optimizer fields reach the step, and the result is the device path's."""
    import torch
    from tcresnet_b200.engine import HostFeed, Optimizer
    eng, wavs, hots = _engine_and_batches()
    opt = Optimizer.adam(ema_decay=0.999) if kind == "adam" else Optimizer.rmsprop(momentum=0.5, ema_decay=0.999)
    h_wavs, h_hots = [w.pin_memory() for w in wavs], [h.pin_memory() for h in hots]   # alive until the copies have run
    res = []
    for host in (False, True):
        p, _, m = eng.new_variables(seed=4)
        st = eng.new_optimizer_state(opt, p)
        feed = HostFeed(eng, lag=2)
        for i in range(6):
            if host:
                feed.submit(h_wavs[i % 3], h_hots[i % 3], p, None, m, 0.01, weight_decay=1e-3, dropout_seed=i, optimizer=opt, state=st)
            else:
                eng.train_step(wavs[i % 3].cuda(), hots[i % 3].cuda(), p, None, m, 0.01, weight_decay=1e-3, dropout_seed=i,
                               optimizer=opt, state=st)
        feed.flush()
        torch.cuda.synchronize()
        res.append(_state_tensors(p, st, m))
    assert all(torch.equal(a, b) for a, b in zip(*res))
    eng.close()


def test_cuda_graph_replay_advances_the_beta_powers(monkeypatch):
    """4 Adam steps replayed from one captured step == 4 eager steps, bit for bit: the powers live in a device buffer that the
    update launch itself advances.  Per-layer kernels (TCR_RESIDENT=0): the resident kernels' grid barrier takes a host-side
    target per call, so a captured resident step cannot be replayed (DESIGN.md section 4g)."""
    import torch
    from tcresnet_b200.engine import Optimizer
    monkeypatch.setenv("TCR_RESIDENT", "0")
    eng, wavs, hots = _engine_and_batches(k=1)
    opt = Optimizer.adam(ema_decay=0.999)
    x, y = wavs[0].cuda(), hots[0].cuda()
    p, _, m = eng.new_variables(seed=5)
    st = eng.new_optimizer_state(opt, p)
    for i in range(4):
        eng.train_step(x, y, p, None, m, 0.01, weight_decay=1e-3, dropout_seed=7, optimizer=opt, state=st)
    torch.cuda.synchronize()
    eager = _state_tensors(p, st, m)
    p2, _, m2 = eng.new_variables(seed=5)
    st2 = eng.new_optimizer_state(opt, p2)
    saved = _state_tensors(p2, st2, m2)
    losses = torch.empty(2, device=eng.device)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):                      # warm-up outside capture (lazy per-kernel attributes), then restore the state
            eng.train_step(x, y, p2, None, m2, 0.01, weight_decay=1e-3, dropout_seed=7, optimizer=opt, state=st2, losses=losses)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    for t, v in zip([p2, m2, st2.slots, st2.slots2, st2.scalars, st2.ema], saved):
        t.copy_(v)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        eng.train_step(x, y, p2, None, m2, 0.01, weight_decay=1e-3, dropout_seed=7, optimizer=opt, state=st2, losses=losses)
    for t, v in zip([p2, m2, st2.slots, st2.slots2, st2.scalars, st2.ema], saved):   # capture does not run the kernels
        assert torch.equal(t, v)
    for _ in range(4):
        g.replay()
    torch.cuda.synchronize()
    replayed = _state_tensors(p2, st2, m2)
    assert all(torch.equal(a, b) for a, b in zip(eager, replayed))
    assert st2.scalars[0].item() == pytest.approx(0.9 ** 5, rel=1e-6)
    eng.close()


def _model(tmp_path, extra=""):
    from tcresnet_b200 import train_audio
    from tcresnet_b200.factory import audio_nets
    args = train_audio.parse_arguments(shlex.split(
        f"--dataset_path synthetic:64 --dataset_split_name train --output_name output/softmax --num_classes 12 --train_dir {tmp_path} "
        "--augmentation_method anchored_slice_or_pad --preprocess_method mfcc --num_mfccs 40 --clip_duration_ms 1000 --window_size_ms 40 --window_stride_ms 20 --batch_size 128 "
        f"--optimizer adam {extra} TCResNet8Model --weight_decay 0.001 --width_multiplier 1.0"))
    m = audio_nets.TCResNet8Model(args)
    m.build_inference(None)
    return m


def test_resume_of_adam_with_ema_is_bitwise(tmp_path):
    """2k steps == k steps, checkpoint (TF tensor bundle), restore into a fresh model, k steps: params, m, v, the beta powers,
    the shadows and the BN moving statistics all bit for bit."""
    import torch
    from tcresnet_b200.common import checkpoint as ckpt
    from tcresnet_b200.engine import Optimizer
    from oracle import tcr_oracle as O
    opt = Optimizer.adam(ema_decay=0.999)
    batches = [tuple(torch.from_numpy(a).cuda() for a in O.synthetic_batch(128, seed_wav=300 + i, seed_label=400 + i)) for i in range(6)]
    k = 3

    def steps(m, lo, hi):
        for i in range(lo, hi):
            m.engine.train_step(batches[i][0], batches[i][1], m.params, None, m.moving, 0.01, weight_decay=1e-3, dropout_seed=i,
                                optimizer=m.optimizer, state=m.opt_state)
        torch.cuda.synchronize()
    a = _model(tmp_path / "a")
    a.set_optimizer(opt)
    init = a.get_variables()
    steps(a, 0, 2 * k)
    straight = a.get_variables()
    b = _model(tmp_path / "b")
    b.set_optimizer(opt)
    b.set_variables(init)
    steps(b, 0, k)
    path = ckpt.save(tmp_path, "TCResNet8Model", k, b.get_variables(), 2, fmt="tf")
    c = _model(tmp_path / "c")
    c.set_optimizer(opt)
    c.set_variables(ckpt.load(path))
    steps(c, k, 2 * k)
    resumed = c.get_variables()
    assert set(resumed) == set(straight) and "beta1_power" in resumed and "TCResNet8/fc/weights/ExponentialMovingAverage" in resumed
    for name, v in straight.items():
        assert np.array_equal(resumed[name], v), name
    for m in (a, b, c):
        m.engine.close()


def test_trainer_with_adam_runs_at_the_host_feed_rate(tmp_path):
    """train_audio.train with --optimizer adam --use_ema on synthetic data (host-buffer step): >= 200 steps, per-step wall time
    within 1.3x of the same Adam steps driven directly through engine.HostFeed; the checkpoint holds Adam's and EMA's state."""
    import time
    import torch
    from tcresnet_b200 import train_audio
    from tcresnet_b200.common import checkpoint as ckpt
    from tcresnet_b200.engine import HostFeed
    common = ("--dataset_path synthetic:4096 --output_name output/softmax --num_classes 12 --preprocess_method mfcc --num_mfccs 40 "
              "--clip_duration_ms 1000 --window_size_ms 40 --window_stride_ms 20 ")
    steps = 260
    args = train_audio.parse_arguments(shlex.split(
        common + f"--dataset_split_name train --train_dir {tmp_path} --augmentation_method anchored_slice_or_pad_with_shift "
        f"--batch_size 512 --boundaries 100000 --max_step_from_restore {steps} --lr_list 0.001 0.0001 --absolute_schedule "
        "--no-boundaries_epoch --step_save_checkpoint 100000 --step_evaluation 100000 --step_save_summaries 100000 "
        "--step_save_first_n_summaries 0 --optimizer adam --use_ema TCResNet8Model --weight_decay 0.001 --width_multiplier 1.0"))
    trainer = train_audio.train(args)
    model = trainer.model
    assert model.global_step == steps and np.isfinite(model._feed_last[1])
    values = ckpt.load(ckpt.latest_checkpoint(tmp_path))
    assert "TCResNet8/fc/weights/Adam_1" in values and "TCResNet8/fc/weights/ExponentialMovingAverage" in values
    assert values["beta1_power"] == pytest.approx(0.9 ** (steps + 1), rel=1e-4)
    fetch = {"step_op": trainer.train_op, "global_step": trainer.global_step, "total_loss": model.total_loss, "model_loss": model.model_loss}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(200):
        trainer.session.run(fetch)
    model.flush_feed()
    torch.cuda.synchronize()
    trainer_ms = (time.perf_counter() - t0) / 200 * 1e3
    feed = HostFeed(model.engine, lag=2)
    batches = [model.dataset.next_batch_pinned() for _ in range(8)]
    run = lambda i: feed.submit(batches[i % 8][0], batches[i % 8][1], model.params, None, model.moving, 1e-3, weight_decay=1e-3,
                                dropout_seed=i, optimizer=model.optimizer, state=model.opt_state)
    for i in range(20):
        run(i)
    feed.flush()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(200):
        run(i)
    feed.flush()
    torch.cuda.synchronize()
    direct_ms = (time.perf_counter() - t0) / 200 * 1e3
    print(f"trainer loop (adam + ema) {trainer_ms:.3f} ms/step, HostFeed directly {direct_ms:.3f} ms/step")
    assert trainer_ms <= 1.3 * direct_ms + 0.05
    assert torch.isfinite(model.params).all() and torch.isfinite(model.opt_state.ema).all()


@pytest.mark.parametrize("exchange,env,port", [("peer-memory", {}, 29621), ("nccl", {"TCR_P2P": "0"}, 29622)])
def test_two_gpus_adam_replicas_identical(exchange, env, port):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(HERE, "dist_optim_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, **env))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "replicas bit-identical" in r.stdout and f"exchange={exchange}" in r.stdout, r.stdout[-500:]
