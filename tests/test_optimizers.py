"""Adam / RMSProp / EMA on a CPU box: the NumPy restatements of the update rules pinned against torch.optim and hand-computed
values, the update kernel compiled against the test emulator (tests/emu) against those restatements, and the host logic
(trainer flags, checkpoint names, the --use_ema restore)."""
import shlex
import types

import numpy as np
import pytest
import torch

import tcresnet_b200  # noqa: F401
from oracle import optim_oracle as OO
from oracle import tcr_oracle as O
from optim_cases import run_optimizer_case
from tcr_harness import NumpyBackend
from tcresnet_b200 import engine as E
from tcresnet_b200 import train_audio
from tcresnet_b200.common import checkpoint as ckpt
from tcresnet_b200.factory import audio_nets
from tcresnet_b200.helper.trainer import TrainerBase


# ---------------------------------------------------------------- restatements of the rules
def _problem(seed=0):
    rng = np.random.RandomState(seed)
    params = {"a": rng.randn(3, 4), "b": rng.randn(5)}
    grads = [{k: rng.randn(*v.shape) for k, v in params.items()} for _ in range(5)]
    return params, grads


def test_adam_without_epsilon_equals_torch_adam():
    """TF puts epsilon outside the bias correction of v, torch inside: with eps = 0 the two rules are the same function."""
    params, grads = _problem()
    lr, b1, b2 = 0.01, 0.9, 0.999
    tp = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in params.items()}
    opt = torch.optim.Adam(list(tp.values()), lr=lr, betas=(b1, b2), eps=0.0)
    p, st = dict(params), OO.adam_state(params, b1, b2)
    for g in grads:
        for k in tp:
            tp[k].grad = torch.tensor(g[k])
        opt.step()
        p, st = OO.adam_update(p, g, st, lr, b1, b2, 0.0)
        for k in tp:
            np.testing.assert_allclose(p[k], tp[k].detach().numpy(), rtol=1e-12, atol=1e-14)
    assert st["beta1_power"] == pytest.approx(b1 ** 6) and st["beta2_power"] == pytest.approx(b2 ** 6)


def test_rmsprop_equals_torch_rmsprop_with_ones_initialised_square_average():
    """torch.optim.RMSprop with square_avg preset to ones (TF's ms initialiser) and eps = 0 (torch adds it outside the sqrt,
    TF inside): mom = momentum*mom + lr*g/sqrt(ms) in both; torch keeps the buffer without lr, which is a constant factor."""
    params, grads = _problem(1)
    lr, decay, mom = 0.01, 0.9, 0.5
    tp = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in params.items()}
    opt = torch.optim.RMSprop(list(tp.values()), lr=lr, alpha=decay, eps=0.0, momentum=mom)
    for t in tp.values():
        opt.state[t] = {"step": torch.tensor(0.0, dtype=torch.float64), "square_avg": torch.ones_like(t).detach(),
                        "momentum_buffer": torch.zeros_like(t).detach()}
    p, st = dict(params), OO.rmsprop_state(params)
    for g in grads:
        for k in tp:
            tp[k].grad = torch.tensor(g[k])
        opt.step()
        p, st = OO.rmsprop_update(p, g, st, lr, decay, mom, 0.0)
        for k in tp:
            np.testing.assert_allclose(p[k], tp[k].detach().numpy(), rtol=1e-12, atol=1e-14)


def test_rmsprop_two_steps_by_hand():
    p, st = {"w": np.array([1.0])}, OO.rmsprop_state({"w": np.array([1.0])})
    p, st = OO.rmsprop_update(p, {"w": np.array([2.0])}, st, lr=0.1, decay=0.9, momentum=0.5, epsilon=0.0)
    # ms = 1 + (4 - 1) * 0.1 = 1.3 ; mom = 0.2 / sqrt(1.3) ; w = 1 - mom
    m1 = 0.2 / np.sqrt(1.3)
    assert st["ms"]["w"][0] == pytest.approx(1.3) and p["w"][0] == pytest.approx(1 - m1)
    p, st = OO.rmsprop_update(p, {"w": np.array([-1.0])}, st, lr=0.1, decay=0.9, momentum=0.5, epsilon=0.0)
    # ms = 1.3 + (1 - 1.3) * 0.1 = 1.27 ; mom = 0.5 * m1 - 0.1 / sqrt(1.27)
    m2 = 0.5 * m1 - 0.1 / np.sqrt(1.27)
    assert st["ms"]["w"][0] == pytest.approx(1.27) and p["w"][0] == pytest.approx(1 - m1 - m2)


def test_adam_first_step_by_hand():
    p, st = {"w": np.array([0.5, -0.5])}, OO.adam_state({"w": np.zeros(2)})
    p, st = OO.adam_update(p, {"w": np.array([3.0, -1e-3])}, st, lr=0.1)
    # alpha = 0.1 * sqrt(0.001) / 0.1 ; m = 0.1 g ; v = 0.001 g^2 -> step = alpha * m / (sqrt(v) + eps) ~ 0.1 * sign(g)
    alpha, g = 0.1 * np.sqrt(0.001) / 0.1, np.array([3.0, -1e-3])
    step = alpha * 0.1 * g / (np.sqrt(0.001) * np.abs(g) + 1e-8)
    np.testing.assert_allclose(p["w"], [0.5, -0.5] - step, rtol=1e-12)
    np.testing.assert_allclose(step, [0.1, -0.1], rtol=1e-3)        # epsilon is visible only for the tiny gradient


def test_ema_by_hand():
    s = {"w": np.array([1.0, 2.0])}
    s = OO.ema_update(s, {"w": np.array([3.0, 0.0])}, decay=0.9)
    np.testing.assert_allclose(s["w"], [1.0 - (1.0 - 3.0) * 0.1, 2.0 - 2.0 * 0.1])
    s = OO.ema_update(s, {"w": np.array([3.0, 0.0])}, decay=0.9)
    np.testing.assert_allclose(s["w"], [1.2 + 1.8 * 0.1, 1.8 - 1.8 * 0.1])


# ---------------------------------------------------------------- the update kernel, emulated
@pytest.fixture(scope="module")
def backend():
    return NumpyBackend()


@pytest.mark.parametrize("kind,ema", [("adam", False), ("adam", True), ("rmsprop", False), ("rmsprop", True), ("mom", True)])
def test_emulated_update_matches_the_rule_on_the_reported_gradient(backend, kind, ema):
    """TCResNet8 at n=5, 3 steps, state kept in place between steps; then an apply_update = 0 step leaves everything as it was."""
    run_optimizer_case(backend, kind, ema, steps=3, n=5)


@pytest.mark.parametrize("mode", ["0", "2"])
def test_emulated_adam_through_the_resident_kernels(backend, monkeypatch, mode):
    """TCR_RESIDENT 2 reduces the gradient inside the resident backward kernel; the update launch is the same."""
    monkeypatch.setenv("TCR_RESIDENT", mode)
    run_optimizer_case(backend, "adam", True, steps=2, n=4)


def test_rules_are_validated(backend):
    import ctypes as C
    from optim_cases import OptimizerRun
    run = OptimizerRun(backend, "adam", n=2)
    try:
        wav, hot = O.synthetic_batch(2)
        inp, oh = backend.upload(wav), backend.upload(hot)
        for field, bad, msg in (("opt_scalars", None, b"opt_scalars"), ("slots2", None, b"slots2"), ("optimizer", 7, b"unknown optimizer")):
            a = run.args(inp, oh)
            setattr(a, field, bad)
            assert run.eng.lib.tcr_train_step(run.eng.h, C.byref(a), None) == 1
            assert msg in run.eng.lib.tcr_last_error()
            assert run.eng.lib.tcr_train_step_host(run.eng.h, C.byref(a), 0, None, None, None) == 1
        a = run.args(inp, oh, apply_update=False)
        a.slots2 = a.opt_scalars = None                    # gradients only: the rule's buffers are not needed
        assert run.eng.lib.tcr_train_step(run.eng.h, C.byref(a), None) == 0
    finally:
        run.close()


# ---------------------------------------------------------------- host logic
def _trainer(**flags):
    t = TrainerBase.__new__(TrainerBase)
    t.log = types.SimpleNamespace(info=lambda *a: None, error=lambda *a: None)
    t.args = types.SimpleNamespace(use_ema=False, ema_decay=0.999, **flags)
    return t


def test_build_optimizer_maps_the_reference_flags():
    t = _trainer()
    assert t.build_optimizer("mom", None, momentum=0.9) == E.Optimizer("mom", momentum=0.9)
    assert t.build_optimizer("mom", None) == E.Optimizer("mom", momentum=0.0)
    assert t.build_optimizer("gd", None, momentum=0.9).kind == "gd"
    assert t.build_optimizer("adam", None) == E.Optimizer("adam", beta1=0.9, beta2=0.999, epsilon=1e-8)
    assert t.build_optimizer("adam", None, epsilon=1e-4).epsilon == 1e-4
    assert t.build_optimizer("adam", None, momentum=0.0, decay=0.0).kind == "adam"        # falsy flags are not forwarded
    with pytest.raises(TypeError, match="momentum"):
        t.build_optimizer("adam", None, momentum=0.9)
    with pytest.raises(TypeError, match="decay"):
        t.build_optimizer("adam", None, decay=0.95)
    r = t.build_optimizer("rmsprop", None)
    assert (r.kind, r.decay, r.momentum, r.epsilon) == ("rmsprop", 0.9, 0.0, 1e-10)
    r = t.build_optimizer("rmsprop", None, momentum=0.5, decay=0.95, epsilon=1e-6)
    assert (r.decay, r.momentum, r.epsilon) == (0.95, 0.5, 1e-6)
    with pytest.raises(NotImplementedError):
        t.build_optimizer("lbfgs", None)


class _CpuEngine(E.Engine):
    """The engine's host-side variable plumbing (TF names <-> flat buffers) on CPU tensors, its table from the oracle's spec."""

    def __init__(self, spec):
        self.device = torch.device("cpu")
        self.table, off = [], 0
        for n in spec.var_names:
            sz = int(np.prod(spec.var_shapes[n]))
            self.table.append(dict(name=n, trainable=True, shape=spec.var_shapes[n], offset=off, numel=sz))
            off += sz
        self.num_trainable, off = off, 0
        for n in O.moving_names(spec):
            c = spec.var_shapes[n.split("/BatchNorm/")[0] + "/weights"][3]
            self.table.append(dict(name=n, trainable=False, shape=(c,), offset=off, numel=c))
            off += c
        self.num_moving = off

    def close(self):
        pass


def _cpu_model(seed=0):
    spec = O.build_spec("TCResNet8", 1.0, 49)
    m = audio_nets.TCResNet8Model(types.SimpleNamespace())
    m.engine = _CpuEngine(spec)
    rng = np.random.RandomState(seed)
    m.params = torch.from_numpy(rng.randn(m.engine.num_trainable).astype(np.float32))
    m.moving = torch.from_numpy(rng.rand(m.engine.num_moving).astype(np.float32))
    m.slots = torch.zeros_like(m.params)
    m.opt_state = E.OptimizerState(slots=m.slots)
    return spec, m


@pytest.mark.parametrize("kind,ema", [("adam", True), ("rmsprop", False), ("mom", True)])
def test_optimizer_state_checkpoint_names_round_trip_through_tf_bundle(tmp_path, kind, ema):
    spec, m = _cpu_model()
    opt = {"adam": E.Optimizer.adam(), "rmsprop": E.Optimizer.rmsprop(), "mom": E.Optimizer("mom")}[kind]
    if ema:
        import dataclasses
        opt = dataclasses.replace(opt, ema_decay=0.999)
    m.set_optimizer(opt)
    st = m.opt_state
    if kind == "rmsprop":
        assert torch.all(st.slots == 1) and torch.all(st.slots2 == 0)      # ms initialised to ones
    if kind == "adam":
        assert st.scalars.tolist() == pytest.approx([0.9, 0.999])
    if ema:
        assert torch.equal(st.ema, m.params)
    for buf in (st.slots, st.slots2, st.ema):                               # something to save
        if buf is not None:
            buf.copy_(torch.randn_like(buf))
    if st.scalars is not None:
        st.scalars.copy_(torch.tensor([0.729, 0.997003]))
    values = m.get_variables()
    w = "TCResNet8/fc/weights"
    expect = {"adam": [w + "/Adam", w + "/Adam_1", "beta1_power", "beta2_power"], "rmsprop": [w + "/RMSProp", w + "/RMSProp_1"],
              "mom": [w + "/Momentum"]}[kind] + ([w + "/ExponentialMovingAverage"] if ema else [])
    for name in expect:
        assert name in values, name
    n_var = len(spec.var_names)
    assert len(values) == n_var + len(O.moving_names(spec)) + n_var * (len(audio_nets.SLOT_SUFFIXES[kind]) + ema) \
        + 2 * (kind == "adam")
    if kind == "adam":
        assert values["beta1_power"].shape == () and values["beta1_power"] == np.float32(0.729)
    path = ckpt.save(tmp_path, "TCResNet8Model", 7, values, 2, fmt="tf")
    back = ckpt.load(path)
    _, fresh = _cpu_model(seed=1)
    fresh.set_optimizer(opt)
    fresh.set_variables(back)
    got = fresh.get_variables()
    for k, v in values.items():
        np.testing.assert_array_equal(got[k], v, err_msg=k)


def test_optimizer_state_missing_from_a_checkpoint_keeps_its_initial_value():
    _, m = _cpu_model()
    values = m.get_variables(with_slots=False)                            # e.g. a momentum checkpoint's model variables
    _, fresh = _cpu_model(seed=3)
    fresh.set_optimizer(E.Optimizer.rmsprop(ema_decay=0.999))
    ema0 = fresh.opt_state.ema.clone()
    fresh.set_variables(values)
    assert torch.all(fresh.opt_state.slots == 1) and torch.all(fresh.opt_state.slots2 == 0)
    assert torch.equal(fresh.opt_state.ema, ema0)
    assert torch.equal(fresh.params, m.params)


def test_use_ema_restore_takes_trainables_from_their_shadows():
    """evaluate_audio.py --use_ema: trainables <- `<var>/ExponentialMovingAverage`, moving statistics under their own names."""
    from tcresnet_b200.helper.evaluator import Evaluator
    spec, m = _cpu_model()
    m.set_optimizer(E.Optimizer("mom", ema_decay=0.999))
    m.opt_state.ema.copy_(torch.randn_like(m.params))
    values = m.get_variables()
    _, ev_model = _cpu_model(seed=5)
    ev = Evaluator.__new__(Evaluator)
    ev.model, ev.args = ev_model, types.SimpleNamespace(use_ema=True, ignore_missing_vars=False, max_step_from_restore=10 ** 9,
                                                       save_best_keeper=False)
    ev.setup_dataset_iterator = lambda: None
    ev.run_evaluation = lambda step, is_training: {}
    ev.metric_manager = types.SimpleNamespace(filter_best_keep_metric=lambda m: {}, log_metrics=lambda *a: None)
    ev.log = types.SimpleNamespace(info=lambda *a: None)
    import tcresnet_b200.helper.evaluator as evmod
    orig = evmod.ckpt.load
    evmod.ckpt.load = lambda path: values
    try:
        ev.evaluate_once("model-12")
    finally:
        evmod.ckpt.load = orig
    assert torch.equal(ev_model.params, m.opt_state.ema) and torch.equal(ev_model.moving, m.moving)
    del values["TCResNet8/fc/weights/ExponentialMovingAverage"]                # a shadow missing: strict restore fails
    with pytest.raises(KeyError):
        ev_model.set_variables_from_ema(values, strict=True)


def test_default_recipe_with_adam_parses_and_builds_a_trainer():
    """The TC-ResNet recipe with --optimizer adam (its --momentum dropped: AdamOptimizer has no such argument) parses, and the
    trainer's optimizer / train-op construction hands the model Adam with EMA when --use_ema is given."""
    line = ("--dataset_path google_speech_commands/splitted_data --dataset_split_name train --output_name output/softmax "
            "--num_classes 12 --train_dir work/v1/TCResNet8Model-1.0/mfcc_40_3010_0.001_adam_l1 --num_silent 1854 "
            "--augmentation_method anchored_slice_or_pad_with_shift --preprocess_method mfcc --num_mfccs 40 "
            "--clip_duration_ms 1000 --window_size_ms 30 --window_stride_ms 10 --batch_size 100 --boundaries 10000 20000 "
            "--max_step_from_restore 30000 --lr_list 0.1 0.01 0.001 --absolute_schedule --no-boundaries_epoch --max_to_keep 20 "
            "--step_save_checkpoint 500 --step_evaluation 500 --optimizer adam --use_ema TCResNet8Model --weight_decay 0.001 "
            "--width_multiplier 1.0")
    a = train_audio.parse_arguments(shlex.split(line))
    assert a.optimizer == "adam" and a.momentum is None and a.use_ema and a.ema_decay == 0.999
    _, m = _cpu_model()
    t = TrainerBase.__new__(TrainerBase)
    TrainerBase.__init__(t, m, None, a, None, "train", "AudioTrainer")
    opt = t.build_optimizer(a.optimizer, None, momentum=a.momentum, decay=a.optimizer_decay, epsilon=a.optimizer_epsilon)
    t.build_train_op(None, opt, a.trainable_scopes, None)
    assert m.optimizer == E.Optimizer.adam(ema_decay=0.999)
    assert m.opt_state.slots2 is not None and m.opt_state.scalars is not None and m.opt_state.ema is not None
    with pytest.raises(TypeError):
        t.build_optimizer("adam", None, momentum=0.9)                     # the recipe's own --momentum 0.9 with adam
