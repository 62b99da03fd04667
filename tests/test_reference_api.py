"""The reference's Python surface (SURVEY.md 8b): the recipes' exact command lines parse, the registries expose the
reference's names, and (GPU) a short train -> checkpoint -> evaluate run works through train_audio / evaluate_audio."""
import os
import shlex

import numpy as np
import pytest

import tcresnet_b200  # noqa: F401
from tcresnet_b200 import evaluate_audio, train_audio
from tcresnet_b200.common import checkpoint as ckpt
from tcresnet_b200.datasets import preprocessor_factory
from tcresnet_b200.factory import audio_nets
from tcresnet_b200.helper.trainer import piecewise_constant
from tcresnet_b200.runtime import Node, Session

RECIPES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_recipes.txt")

# verbatim copies of the TC-ResNet recipe lines (scripts/commands/TCResNet8Model-1.0_mfcc_40_3010_0.001_mom_l1.sh:3,5,7)
TRAIN_LINE = ("--dataset_path google_speech_commands/splitted_data --dataset_split_name train --output_name output/softmax "
              "--num_classes 12 --train_dir work/v1/TCResNet8Model-1.0/mfcc_40_3010_0.001_mom_l1 --num_silent 1854 "
              "--augmentation_method anchored_slice_or_pad_with_shift --preprocess_method mfcc --num_mfccs 40 "
              "--clip_duration_ms 1000 --window_size_ms 30 --window_stride_ms 10 --batch_size 100 --boundaries 10000 20000 "
              "--max_step_from_restore 30000 --lr_list 0.1 0.01 0.001 --absolute_schedule --no-boundaries_epoch --max_to_keep 20 "
              "--step_save_checkpoint 500 --step_evaluation 500 --optimizer mom --momentum 0.9 TCResNet8Model --weight_decay 0.001 "
              "--width_multiplier 1.0")
EVAL_LINE = ("--dataset_path google_speech_commands/splitted_data --dataset_split_name valid --output_name output/softmax "
             "--num_classes 12 --checkpoint_path work/v1/TCResNet8Model-1.0/mfcc_40_3010_0.001_mom_l1 --num_silent 258 "
             "--augmentation_method anchored_slice_or_pad --preprocess_method mfcc --num_mfccs 40 --clip_duration_ms 1000 "
             "--window_size_ms 30 --window_stride_ms 10 --background_frequency 0.0 --background_max_volume 0.0 "
             "--max_step_from_restore 30000 --batch_size 3 --no-shuffle --valid_type loop TCResNet8Model --weight_decay 0.001 "
             "--width_multiplier 1.0")


def test_recipe_command_lines_parse():
    a = train_audio.parse_arguments(shlex.split(TRAIN_LINE))
    assert (a.model, a.weight_decay, a.width_multiplier, a.batch_size) == ("TCResNet8Model", 0.001, 1.0, 100)
    assert a.lr_list == [0.1, 0.01, 0.001] and a.boundaries == [10000, 20000] and a.relative is False
    assert a.boundaries_epoch is False and a.optimizer == "mom" and a.momentum == 0.9
    assert (a.window_size_ms, a.window_stride_ms, a.num_mfccs, a.num_mel_bins) == (30.0, 10.0, 40, 64)
    e = evaluate_audio.parse_arguments(shlex.split(EVAL_LINE))
    assert (e.model, e.valid_type, e.batch_size, e.shuffle) == ("TCResNet8Model", "loop", 3, False)


def test_every_reference_recipe_parses():
    n = 0
    for line in open(RECIPES):
        if line.startswith("python train_audio.py"):
            train_audio.parse_arguments(shlex.split(line)[2:])
            n += 1
        elif line.startswith("python evaluate_audio.py"):
            evaluate_audio.parse_arguments(shlex.split(line)[2:])
            n += 1
    assert n >= 40


def test_registries_expose_the_reference_names():
    ref = ["KWSModel", "Res8Model", "Res8NarrowModel", "Res15Model", "Res15NarrowModel", "DSCNNSModel", "DSCNNMModel",
           "DSCNNLModel", "TCResNet8Model", "TCResNet14Model", "ResNet2D8Model", "ResNet2D8PoolModel"]
    assert audio_nets._available_nets == ref                      # factory/audio_nets.py:19-32
    for name in ref:
        assert hasattr(audio_nets, name)
    assert set(preprocessor_factory._available_preprocessors) == {"log_mel_spectrogram", "mfcc", "no_preprocessing"}
    with pytest.raises(NotImplementedError):
        preprocessor_factory.factory("nope", "s", "n")
    pre = preprocessor_factory.factory("mfcc", "input/audio/preprocessing", "input/audio/preprocessed")
    node = pre.preprocess(Node("wav", [None, 16000, 1]), 480, 160, False, num_mfccs=40, num_mel_bins=64, sample_rate=16000)
    assert node.shape == [None, 98, 40, 1] and pre.preprocessed_node is node


@pytest.mark.parametrize("fmt", ["tf", "npz"])
def test_learning_rate_schedule_and_checkpoints(tmp_path, fmt):
    assert [piecewise_constant(s, [10000, 20000], [0.1, 0.01, 0.001]) for s in (0, 10000, 10001, 20001)] == [0.1, 0.1, 0.01, 0.001]
    var = {"TCResNet8/conv0/weights": np.arange(6, dtype=np.float32).reshape(3, 1, 2, 1)}
    for step in (500, 1000, 1500):
        path = ckpt.save(tmp_path, "TCResNet8Model", step, var, max_to_keep=2, fmt=fmt)
    assert ckpt.checkpoint_step(path) == 1500 and ckpt.latest_checkpoint(tmp_path) == path
    assert len(list(tmp_path.glob("*.npz" if fmt == "npz" else "*.index"))) == 2      # max_to_keep
    assert not list(tmp_path.glob("*-500*"))
    back = ckpt.load(path)
    assert int(back["global_step"]) == 1500
    np.testing.assert_array_equal(back["TCResNet8/conv0/weights"], var["TCResNet8/conv0/weights"])
    assert next(ckpt.checkpoints_iterator(tmp_path, timeout=0)) == path
    (tmp_path / ".TCResNet8Model-9999.123.tmp").write_bytes(b"partial")              # an in-progress save is never picked up
    assert ckpt.latest_checkpoint(tmp_path) == path


def test_concurrent_saves_into_one_directory_do_not_collide(tmp_path):
    """Several processes saving the same step (a mis-configured data-parallel run) must not trip over each other's temporary files."""
    import multiprocessing as mp
    var = {"v": np.arange(1000, dtype=np.float32)}
    ctx = mp.get_context("fork")
    procs = [ctx.Process(target=lambda: [ckpt.save(tmp_path, "M", s, var, fmt="tf") for s in range(1, 11)]) for _ in range(4)]
    [p.start() for p in procs]
    [p.join() for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    np.testing.assert_array_equal(ckpt.load(ckpt.latest_checkpoint(tmp_path))["v"], var["v"])


def test_session_requires_a_bound_model():
    with pytest.raises(RuntimeError):
        Session().run({"x": Node("total_loss")})
    assert Session().run(Node("noop")) is None


@pytest.mark.gpu
def test_train_then_evaluate_through_the_reference_cli(tmp_path):
    common = (f"--dataset_path synthetic:96 --output_name output/softmax --num_classes 12 --preprocess_method mfcc "
              f"--num_mfccs 40 --clip_duration_ms 1000 --window_size_ms 30 --window_stride_ms 10 ")
    train_args = train_audio.parse_arguments(shlex.split(
        common + f"--dataset_split_name train --train_dir {tmp_path} --augmentation_method anchored_slice_or_pad_with_shift "
        "--batch_size 32 --boundaries 10 20 --max_step_from_restore 12 --lr_list 0.1 0.01 0.001 --absolute_schedule "
        "--no-boundaries_epoch --step_save_checkpoint 6 --step_evaluation 6 --optimizer mom --momentum 0.9 "
        "TCResNet8Model --weight_decay 0.001 --width_multiplier 1.0"))
    trainer = train_audio.train(train_args)
    assert trainer.model.global_step == 12
    saved = ckpt.latest_checkpoint(tmp_path)
    assert saved is not None and ckpt.checkpoint_step(saved) == 12
    names = set(ckpt.load(saved))
    assert "TCResNet8/block0/conv0_0/BatchNorm/moving_variance" in names and "TCResNet8/fc/weights/Momentum" in names
    eval_args = evaluate_audio.parse_arguments(shlex.split(
        common + f"--dataset_split_name valid --checkpoint_path {tmp_path} --augmentation_method anchored_slice_or_pad "
        "--batch_size 3 --no-shuffle --valid_type once TCResNet8Model --weight_decay 0.001 --width_multiplier 1.0"))
    results = evaluate_audio.main(eval_args)
    assert len(results) == 1 and 0.0 <= results[0]["accuracy"] <= 1.0 and np.isfinite(results[0]["total_loss"])
    assert (tmp_path / "valid" / "accuracy").is_dir()              # best-checkpoint directory the test recipe reads


@pytest.mark.gpu
def test_trainer_loop_runs_at_the_host_feed_rate(tmp_path):
    """train_audio.train on `synthetic:` data goes through the C ABI's host-buffer step (tcr_train_step_host): its per-step wall
    time must stay within 1.3x of the same steps driven directly through engine.HostFeed (what bench.py's e2e measures)."""
    import time
    import torch
    from tcresnet_b200.engine import HostFeed
    common = ("--dataset_path synthetic:4096 --output_name output/softmax --num_classes 12 --preprocess_method mfcc --num_mfccs 40 "
              "--clip_duration_ms 1000 --window_size_ms 40 --window_stride_ms 20 ")
    steps = 260
    args = train_audio.parse_arguments(shlex.split(
        common + f"--dataset_split_name train --train_dir {tmp_path} --augmentation_method anchored_slice_or_pad_with_shift "
        f"--batch_size 512 --boundaries 100000 --max_step_from_restore {steps} --lr_list 0.1 0.01 --absolute_schedule --no-boundaries_epoch "
        "--step_save_checkpoint 100000 --step_evaluation 100000 --step_save_summaries 100000 --step_save_first_n_summaries 0 "
        "--optimizer mom --momentum 0.9 TCResNet8Model --weight_decay 0.001 --width_multiplier 1.0"))
    trainer = train_audio.train(args)                                        # warm-up run (also exercises the final flush + checkpoint)
    model = trainer.model
    assert model.global_step == steps and np.isfinite(model._feed_last[1])
    fetch = {"step_op": trainer.train_op, "global_step": trainer.global_step, "total_loss": model.total_loss, "model_loss": model.model_loss}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(200):
        trainer.session.run(fetch)
    model.flush_feed()
    torch.cuda.synchronize()
    trainer_ms = (time.perf_counter() - t0) / 200 * 1e3
    eng, feed = model.engine, HostFeed(model.engine, lag=2)
    batches = [model.dataset.next_batch_pinned() for _ in range(8)]
    for i in range(20):
        feed.submit(batches[i % 8][0], batches[i % 8][1], model.params, model.slots, model.moving, 0.1, 0.9, 1e-3, dropout_seed=i)
    feed.flush()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(200):
        feed.submit(batches[i % 8][0], batches[i % 8][1], model.params, model.slots, model.moving, 0.1, 0.9, 1e-3, dropout_seed=i)
    feed.flush()
    torch.cuda.synchronize()
    direct_ms = (time.perf_counter() - t0) / 200 * 1e3
    print(f"trainer loop {trainer_ms:.3f} ms/step, HostFeed directly {direct_ms:.3f} ms/step")
    assert trainer_ms <= 1.3 * direct_ms + 0.05


@pytest.mark.gpu
def test_deployable_model_batch1_inference(tmp_path):
    """build_deployable_model(include_preprocess=True / False): wav -> softmax for one clip, equal to the evaluation forward of the
    engine, eagerly and when the launch sequence is replayed from a CUDA graph (third call onwards)."""
    import argparse
    args = argparse.Namespace(width_multiplier=1.0, num_classes=12, sample_rate=16000, clip_duration_ms=1000, window_size_ms=40.0,
                              window_stride_ms=20.0, num_mel_bins=64, num_mfccs=40, lower_edge_hertz=80.0, upper_edge_hertz=7600.0,
                              preprocess_method="mfcc", batch_size=1, input_batch_size=1, dropout_keep_prob=0.5, output_name="output/softmax",
                              weight_decay=1e-3, height=-1, width=-1, channels=-1)
    model = audio_nets.TCResNet8Model(args, None)
    inputs, deployed = model.build_deployable_model(include_preprocess=True)
    assert inputs[0].shape == [1, 16000, 1]
    rng = np.random.default_rng(0)
    clips = rng.uniform(-1, 1, (5, 16000)).astype(np.float32)
    import torch
    ref = np.concatenate([model.engine.forward(torch.from_numpy(c[None]).cuda(), model.params, model.moving)["probs"].cpu().numpy()
                          for c in clips])                                 # the engine was sized for batch 1
    got = np.concatenate([deployed(c) for c in clips])                     # calls 3-5 replay the captured graph
    assert deployed._graph is not None
    np.testing.assert_allclose(got, ref, rtol=0, atol=1e-6)
    assert np.array_equal(got.argmax(1), ref.argmax(1))
    args.height, args.width, args.channels = 49, 40, 1
    _, deployed_f = model.build_deployable_model(include_preprocess=False)
    feat = model.engine.mfcc(torch.from_numpy(clips[:1]).cuda()).cpu().numpy()
    np.testing.assert_allclose(deployed_f(feat), ref[:1], rtol=0, atol=1e-6)
