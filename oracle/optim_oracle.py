"""Update rules of the reference's other optimizers and of --use_ema, restated in NumPy (fp64 or fp32, the dtype of the inputs).

TF 1.13 semantics (no TF here; unpinned, restated from the kernels' documented arithmetic):
  * tf.train.AdamOptimizer(lr, beta1, beta2, epsilon) — ApplyAdam, then `_finish` advances the non-slot beta powers;
  * tf.train.RMSPropOptimizer(lr, decay, momentum, epsilon), not centered — ApplyRMSProp;
  * tf.train.ExponentialMovingAverage(decay).apply(trainables) after the train op (helper/trainer.py:213-217),
    assign_moving_average with zero_debias=False and no num_updates.
The gradient `g` is the total-loss gradient (weight decay included), as tcr_oracle.backward returns it or as the CUDA step
reports it.  tcr_oracle.train_step (momentum) is left as it is; these functions take the gradient so the update can be
checked on the gradient the step itself reports (DESIGN.md section 2).
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np


def adam_state(params: Dict[str, np.ndarray], beta1=0.9, beta2=0.999, dtype=np.float64):
    """Slots `<var>/Adam` (m) and `<var>/Adam_1` (v) at zero, powers at beta1 / beta2."""
    return dict(m={k: np.zeros(v.shape, dtype) for k, v in params.items()},
                v={k: np.zeros(v.shape, dtype) for k, v in params.items()},
                beta1_power=dtype(beta1), beta2_power=dtype(beta2))


def adam_update(params, grads, state, lr, beta1=0.9, beta2=0.999, epsilon=1e-8):
    """One ApplyAdam per variable + _finish.  Returns (new params, new state); the inputs are not modified."""
    dt = np.asarray(state["beta1_power"]).dtype.type
    b1p, b2p = dt(state["beta1_power"]), dt(state["beta2_power"])
    alpha = dt(lr) * np.sqrt(dt(1) - b2p) / (dt(1) - b1p)
    new_p, m_out, v_out = {}, {}, {}
    for k in params:
        g = np.asarray(grads[k], dt)
        m = state["m"][k] + (g - state["m"][k]) * (dt(1) - dt(beta1))
        v = state["v"][k] + (g * g - state["v"][k]) * (dt(1) - dt(beta2))
        new_p[k] = params[k] - (m * alpha) / (np.sqrt(v) + dt(epsilon))
        m_out[k], v_out[k] = m, v
    return new_p, dict(m=m_out, v=v_out, beta1_power=b1p * dt(beta1), beta2_power=b2p * dt(beta2))


def rmsprop_state(params: Dict[str, np.ndarray], dtype=np.float64):
    """Slots `<var>/RMSProp` (ms) initialised to ONES and `<var>/RMSProp_1` (mom) to zeros."""
    return dict(ms={k: np.ones(v.shape, dtype) for k, v in params.items()},
                mom={k: np.zeros(v.shape, dtype) for k, v in params.items()})


def rmsprop_update(params, grads, state, lr, decay=0.9, momentum=0.0, epsilon=1e-10):
    """One ApplyRMSProp per variable: ms += (g^2 - ms)(1 - decay); mom = mom*momentum + g*lr/sqrt(ms + eps); w -= mom."""
    dt = next(iter(state["ms"].values())).dtype.type
    new_p, ms_out, mom_out = {}, {}, {}
    for k in params:
        g = np.asarray(grads[k], dt)
        ms = state["ms"][k] + (g * g - state["ms"][k]) * (dt(1) - dt(decay))
        mom = state["mom"][k] * dt(momentum) + (g * dt(lr)) / np.sqrt(ms + dt(epsilon))
        new_p[k] = params[k] - mom
        ms_out[k], mom_out[k] = ms, mom
    return new_p, dict(ms=ms_out, mom=mom_out)


def momentum_update(params, grads, slots, lr, momentum=0.9):
    """ApplyMomentum on a given gradient (the arithmetic of tcr_oracle.train_step's update): m = mom*m + g; w -= lr*m."""
    new_p, new_s = {}, {}
    for k in params:
        dt = params[k].dtype.type
        m = slots[k] * dt(momentum) + np.asarray(grads[k], params[k].dtype)
        new_p[k], new_s[k] = params[k] - dt(lr) * m, m
    return new_p, new_s


def ema_update(shadows, params, decay=0.999):
    """ExponentialMovingAverage.apply on the UPDATED weights: s -= (s - w) * (1 - decay) (fixed decay, no zero-debias)."""
    out = {}
    for k in shadows:
        dt = shadows[k].dtype.type
        out[k] = shadows[k] - (shadows[k] - np.asarray(params[k], shadows[k].dtype)) * (dt(1) - dt(decay))
    return out


def apply_rule(kind: str, params, grads, state, lr, hyper: Optional[dict] = None):
    """Dispatch on the trainer's optimizer kind ("mom", "gd", "adam", "rmsprop").  `state`: {"slots": ...} for momentum,
    adam_state() / rmsprop_state() otherwise.  Returns (new params, new state)."""
    h = dict(hyper or {})
    if kind in ("mom", "gd"):
        p, s = momentum_update(params, grads, state["slots"], lr, h.get("momentum", 0.9) if kind == "mom" else 0.0)
        return p, dict(slots=s)
    if kind == "adam":
        return adam_update(params, grads, state, lr, h.get("beta1", 0.9), h.get("beta2", 0.999), h.get("epsilon", 1e-8))
    if kind == "rmsprop":
        return rmsprop_update(params, grads, state, lr, h.get("decay", 0.9), h.get("momentum", 0.0), h.get("epsilon", 1e-10))
    raise ValueError(kind)
