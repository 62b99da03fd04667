"""Optimizer parity cases shared by the emulator (CPU) and GPU tests: the Adam / RMSProp / momentum update and the EMA shadows
of the CUDA step, driven through the C ABI with state buffers that stay in place across steps.

Tolerance (DESIGN.md section 2, "Update rules"): the gradient the step reports is checked against the fp64 oracle as in
parity_cases.py; the update is checked by applying the fp64 restatement of the rule (oracle/optim_oracle.py) to THAT gradient
and to the state from before the step, carried forward over the steps.  Adam's first step is ~lr*sign(g): an fp32 round-off
gradient near zero may flip sign between the two paths, so the rule must not be fed the oracle's own gradient.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from oracle import optim_oracle as OO
from oracle import tcr_oracle as O
from parity_cases import TOL_STATE, cuda_relu_masks, perturbed_variables
from tcr_harness import Engine, rel_err
from tcresnet_b200 import _lib as L

KINDS = {"mom": L.TCR_OPT_MOMENTUM, "adam": L.TCR_OPT_ADAM, "rmsprop": L.TCR_OPT_RMSPROP}
HYPER = {"mom": dict(momentum=0.9), "adam": dict(beta1=0.9, beta2=0.999, epsilon=1e-8),
         "rmsprop": dict(decay=0.9, momentum=0.0, epsilon=1e-10)}


def initial_state(kind, spec, params, ema, dtype=np.float64):
    """The optimizer state a fresh model starts from, as fp64 dicts by variable name."""
    if kind == "adam":
        st = OO.adam_state(params, HYPER["adam"]["beta1"], HYPER["adam"]["beta2"], dtype)
    elif kind == "rmsprop":
        st = OO.rmsprop_state(params, dtype)
    else:
        rng = np.random.RandomState(7)
        st = dict(slots={k: 0.01 * rng.randn(*v.shape) for k, v in params.items()})
    if ema:
        st["ema"] = {k: np.asarray(v, dtype).copy() for k, v in params.items()}
    return st


class OptimizerRun:
    """One handle + device-resident params / moving / slots / slots2 / powers / shadows, stepped in place."""

    def __init__(self, backend, kind, ema=False, model="TCResNet8", wm=1.0, n=4, max_batch=None, keep=1.0, lr=0.01, wd=1e-3,
                 ema_decay=0.999, window=640, stride=320, hyper=None):
        self.b, self.kind, self.ema, self.n, self.lr, self.wd, self.ema_decay = backend, kind, ema, n, lr, wd, ema_decay
        self.hyper = dict(HYPER[kind], **(hyper or {}))
        t = O.num_frames(16000, window, stride)
        self.spec = O.build_spec(model, wm, t)
        self.eng = Engine(backend, model=int(model[len("TCResNet"):]), width_multiplier=wm, max_batch=max_batch or max(n, 8),
                          dropout_keep_prob=keep, window_size_samples=window, window_stride_samples=stride)
        self.keep = keep
        params, moving = perturbed_variables(self.spec)
        st = initial_state(kind, self.spec, params, ema)
        fl = lambda d: O.flatten_vars(self.spec, d)
        b = backend
        self.params, self.moving = b.upload(fl(params)), b.upload(O.flatten_moving(self.spec, moving))
        if kind == "adam":
            self.slots, self.slots2 = b.upload(fl(st["m"])), b.upload(fl(st["v"]))
            self.scalars = b.upload(np.array([st["beta1_power"], st["beta2_power"]], np.float32))
        elif kind == "rmsprop":
            self.slots, self.slots2, self.scalars = b.upload(fl(st["ms"])), b.upload(fl(st["mom"])), None
        else:
            self.slots, self.slots2, self.scalars = b.upload(fl(st["slots"])), None, None
        self.shadow = b.upload(fl(st["ema"])) if ema else None
        self.window, self.stride = window, stride
        self.grads = b.empty(self.eng.info.num_trainable)
        self.losses, self.logits = b.empty(2), b.empty(n, self.eng.cfg.num_classes)

    def close(self):
        self.eng.close()

    def args(self, inp, onehot, seed=0, mask=None, apply_update=True):
        b, h = self.b, self.hyper
        a = L.TcrStepArgs()
        a.input, a.input_is_features, a.onehot, a.n = b.ptr(inp), 0, b.ptr(onehot), self.n
        a.params, a.slots, a.moving = b.ptr(self.params), b.ptr(self.slots), b.ptr(self.moving)
        a.learning_rate, a.momentum, a.weight_decay = self.lr, h.get("momentum", 0.0), self.wd
        a.dropout_seed, a.dropout_mask = seed, b.ptr(mask)
        a.losses, a.logits, a.grads, a.apply_update = b.ptr(self.losses), b.ptr(self.logits), b.ptr(self.grads), int(apply_update)
        a.optimizer, a.slots2, a.opt_scalars = KINDS[self.kind], b.ptr(self.slots2), b.ptr(self.scalars)
        a.beta1, a.beta2 = h.get("beta1", 0.0), h.get("beta2", 0.0)
        a.epsilon, a.rms_decay = h.get("epsilon", 0.0), h.get("decay", 0.0)
        a.ema, a.ema_decay = b.ptr(self.shadow), self.ema_decay if self.ema else 0.0
        return a

    def step(self, inp, onehot, seed=0, mask=None, apply_update=True):
        a = self.args(inp, onehot, seed, mask, apply_update)
        L.check(self.eng.lib, self.eng.lib.tcr_train_step(self.eng.h, C.byref(a), self.b.stream), "tcr_train_step")
        self.b.sync()

    def state(self):
        """Everything the step updates, downloaded (fp32 NumPy)."""
        d = self.b.download
        out = dict(params=d(self.params), moving=d(self.moving), slots=d(self.slots))
        if self.slots2 is not None:
            out["slots2"] = d(self.slots2)
        if self.scalars is not None:
            out["scalars"] = d(self.scalars)
        if self.shadow is not None:
            out["ema"] = d(self.shadow)
        return out

    # ---- fp64 restatement of the update on the reported gradient
    def oracle_state(self, s):
        """fp64 oracle state (rule-specific dicts) from a downloaded state()."""
        un = lambda f: O.unflatten_vars(self.spec, f)
        if self.kind == "adam":
            st = dict(m=un(s["slots"]), v=un(s["slots2"]), beta1_power=np.float64(s["scalars"][0]),
                      beta2_power=np.float64(s["scalars"][1]))
        elif self.kind == "rmsprop":
            st = dict(ms=un(s["slots"]), mom=un(s["slots2"]))
        else:
            st = dict(slots=un(s["slots"]))
        if self.ema:
            st["ema"] = un(s["ema"])
        return un(s["params"]), st

    def oracle_update(self, params, st, grads_flat):
        g = O.unflatten_vars(self.spec, grads_flat)
        p1, st1 = OO.apply_rule(self.kind, params, g, st, self.lr, self.hyper)
        if self.ema:
            st1["ema"] = OO.ema_update(st["ema"], p1, self.ema_decay)
        return p1, st1

    def compare(self, got, params_ref, st_ref):
        """rel_err of every state buffer against the carried fp64 state."""
        fl = lambda d: O.flatten_vars(self.spec, d, np.float64)
        r = {"params": rel_err(got["params"], fl(params_ref))}
        if self.kind == "adam":
            r["m"], r["v"] = rel_err(got["slots"], fl(st_ref["m"])), rel_err(got["slots2"], fl(st_ref["v"]))
            r["powers"] = rel_err(got["scalars"], np.array([st_ref["beta1_power"], st_ref["beta2_power"]]))
        elif self.kind == "rmsprop":
            r["ms"], r["mom"] = rel_err(got["slots"], fl(st_ref["ms"])), rel_err(got["slots2"], fl(st_ref["mom"]))
        else:
            r["slots"] = rel_err(got["slots"], fl(st_ref["slots"]))
        if self.ema:
            r["ema"] = rel_err(got["ema"], fl(st_ref["ema"]))
        return r


def run_optimizer_case(backend, kind, ema=False, steps=3, model="TCResNet8", wm=1.0, n=4, max_batch=None, keep=1.0,
                       grad_steps=None, force_masks=False, lr=0.01):
    """`steps` steps of one rule: every step's gradient against the fp64 oracle (the steps listed in grad_steps, default all),
    every step's update against the fp64 rule carried forward on the reported gradients.  Then one apply_update = 0 step,
    which must leave every state buffer (powers included) bit for bit as it was.  Returns the report."""
    run = OptimizerRun(backend, kind, ema, model=model, wm=wm, n=n, max_batch=max_batch, keep=keep, lr=lr)
    spec = run.spec
    try:
        wav, onehot = O.synthetic_batch(n, adversarial=True)
        feat = O.mfcc(wav, run.window, run.stride)
        inp, hot = backend.upload(wav), backend.upload(onehot)
        rng = np.random.RandomState(11)
        report = {}
        got = run.state()
        p_ref, st_ref = run.oracle_state(got)
        for step in range(steps):
            mask_np = (rng.rand(n, spec.c_last) < keep).astype(np.float32) if keep < 1 else None
            before = got
            run.step(inp, hot, seed=step, mask=backend.upload(mask_np) if mask_np is not None else None)
            got = run.state()
            grads = backend.download(run.grads)
            if grad_steps is None or step in grad_steps:
                p = O.unflatten_vars(spec, before["params"])
                mv = O.unflatten_moving(spec, before["moving"])
                forced = cuda_relu_masks(run.eng, spec, n) if force_masks else None
                _, mv1, _, ref = O.train_step(spec, p, mv, O.zeros_like_vars(spec), feat, onehot, run.lr, 0.0, run.wd, keep,
                                              mask_np, 0.0, forced_masks=forced)
                report[f"grads{step}"] = rel_err(grads, O.flatten_vars(spec, ref["grads"], np.float64))
                report[f"moving{step}"] = rel_err(got["moving"], O.flatten_moving(spec, mv1, np.float64))
                assert report[f"grads{step}"] <= TOL_STATE, report
                assert report[f"moving{step}"] <= TOL_STATE, report
            p_ref, st_ref = run.oracle_update(p_ref, st_ref, grads)
            for k, v in run.compare(got, p_ref, st_ref).items():
                report[f"{k}{step}"] = v
                assert v <= TOL_STATE, (k, step, report)
        # gradients only: nothing moves, the powers included
        run.step(inp, hot, seed=99, apply_update=False)
        after = run.state()
        for k in got:
            assert np.array_equal(after[k], got[k]), k
        return report
    finally:
        run.close()
