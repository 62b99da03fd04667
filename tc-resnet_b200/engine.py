"""Host-side engine: one C-ABI handle + torch CUDA tensors as buffer carriers.

This is the object the reference-facing shims (factory/audio_nets.py, helper/trainer.py, helper/evaluator.py)
drive; it maps the reference's `args` flags onto tcr_config and exposes the three calls a `session.run`
of the reference amounts to: front-end, forward (eval / training-graph) and one full training step.
There is no CPU path: constructing an Engine without a CUDA device or without libtcr_b200.so raises.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib as L

_MODELS = {"TCResNet8": 8, "TCResNet8Model": 8, "TCResNet14": 14, "TCResNet14Model": 14, 8: 8, 14: 14}
_FEATURES = {"mfcc": L.TCR_FEATURE_MFCC, "log_mel_spectrogram": L.TCR_FEATURE_LOG_MEL}
_RULES = {"mom": L.TCR_OPT_MOMENTUM, "gd": L.TCR_OPT_MOMENTUM, "adam": L.TCR_OPT_ADAM, "rmsprop": L.TCR_OPT_RMSPROP}


@dataclass
class Optimizer:
    """The update rule of a training step and its hyper-parameters (what helper/trainer.py:build_optimizer chose).
    kind: "mom" (tf.train.MomentumOptimizer), "gd" (momentum 0), "adam" (tf.train.AdamOptimizer) or "rmsprop"
    (tf.train.RMSPropOptimizer, not centered).  ema_decay not None: tf.train.ExponentialMovingAverage after every step
    (--use_ema).  The defaults are TF 1.13's."""
    kind: str = "mom"
    momentum: float = 0.9          # mom; rmsprop (default 0.0 there, see rmsprop())
    beta1: float = 0.9
    beta2: float = 0.999
    epsilon: float = 1e-8          # adam 1e-8, rmsprop 1e-10
    decay: float = 0.9             # rmsprop
    ema_decay: Optional[float] = None

    def __post_init__(self):
        if self.kind not in _RULES:
            raise NotImplementedError(f"optimizer {self.kind!r}")

    @classmethod
    def rmsprop(cls, decay=0.9, momentum=0.0, epsilon=1e-10, ema_decay=None):
        return cls("rmsprop", momentum=momentum, epsilon=epsilon, decay=decay, ema_decay=ema_decay)

    @classmethod
    def adam(cls, beta1=0.9, beta2=0.999, epsilon=1e-8, ema_decay=None):
        return cls("adam", beta1=beta1, beta2=beta2, epsilon=epsilon, ema_decay=ema_decay)


@dataclass
class OptimizerState:
    """Device buffers of an update rule, by role.  slots: `<var>/Momentum` | `<var>/Adam` (m) | `<var>/RMSProp` (ms);
    slots2: `<var>/Adam_1` (v) | `<var>/RMSProp_1` (mom); scalars: [beta1_power, beta2_power] (Adam);
    ema: `<var>/ExponentialMovingAverage` shadows.  Unused roles are None."""
    slots: torch.Tensor
    slots2: Optional[torch.Tensor] = None
    scalars: Optional[torch.Tensor] = None
    ema: Optional[torch.Tensor] = None


def _set_rule(a: "L.TcrStepArgs", ptr, slots, momentum: float, optimizer: Optional[Optimizer], state: Optional[OptimizerState]):
    """Fills the update-rule fields of tcr_step_args.  optimizer None: the momentum step with `momentum` (the v5 call)."""
    opt = optimizer if optimizer is not None else Optimizer("mom", momentum=momentum)
    if slots is None:
        if state is None:
            raise ValueError("train step needs `slots` or an OptimizerState")
        slots = state.slots
    a.slots = ptr(slots)
    a.optimizer = _RULES[opt.kind]
    a.momentum = 0.0 if opt.kind in ("gd", "adam") else float(opt.momentum)
    if opt.kind in ("adam", "rmsprop"):
        if state is None or state.slots2 is None or (opt.kind == "adam" and state.scalars is None):
            raise ValueError(f"optimizer {opt.kind!r} needs its OptimizerState (Engine.new_optimizer_state)")
        a.slots2, a.opt_scalars = ptr(state.slots2), ptr(state.scalars)
        a.beta1, a.beta2, a.epsilon, a.rms_decay = float(opt.beta1), float(opt.beta2), float(opt.epsilon), float(opt.decay)
    if opt.ema_decay is not None:
        if state is None or state.ema is None:
            raise ValueError("EMA needs the shadow buffer of an OptimizerState (Engine.new_optimizer_state)")
        a.ema, a.ema_decay = ptr(state.ema), float(opt.ema_decay)


class Engine:
    def __init__(self, model="TCResNet8", width_multiplier=1.0, num_classes=12, sample_rate=16000,
                 clip_duration_ms=1000, window_size_ms=40.0, window_stride_ms=20.0, num_mel_bins=64, num_mfccs=40,
                 lower_edge_hertz=80.0, upper_edge_hertz=7600.0, preprocess_method="mfcc", max_batch=512,
                 dropout_keep_prob=0.5, label_smoothing=0.0, bn_decay=0.997, bn_epsilon=1e-3,
                 device: Optional[int] = None):
        if not torch.cuda.is_available():
            raise L.TcrError("tcresnet_b200.Engine needs a CUDA device (there is no CPU fallback)")
        if model not in _MODELS:
            raise NotImplementedError(f"{model}: only TCResNet8/TCResNet14 are on the accelerated path")
        if preprocess_method not in _FEATURES:
            raise NotImplementedError(f"preprocess_method {preprocess_method}")
        self.lib = L.load()
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        c = L.TcrConfig()
        L.check(self.lib, self.lib.tcr_config_default(C.byref(c)), "tcr_config_default")
        c.model = _MODELS[model]
        c.width_multiplier = float(width_multiplier)
        c.num_classes = int(num_classes)
        c.sample_rate = int(sample_rate)
        # the reference's integer truncations (factory/audio_nets.py:63-64, :89)
        c.clip_samples = int(sample_rate * clip_duration_ms / 1000)
        c.window_size_samples = int(sample_rate * window_size_ms / 1000)
        c.window_stride_samples = int(sample_rate * window_stride_ms / 1000)
        c.num_mel_bins, c.num_mfccs = int(num_mel_bins), int(num_mfccs)
        c.lower_edge_hertz, c.upper_edge_hertz = float(lower_edge_hertz), float(upper_edge_hertz)
        c.feature_kind = _FEATURES[preprocess_method]
        c.max_batch = int(max_batch)
        c.bn_decay, c.bn_epsilon = float(bn_decay), float(bn_epsilon)
        c.dropout_keep_prob, c.label_smoothing = float(dropout_keep_prob), float(label_smoothing)
        c.device = self.device.index
        self.cfg = c
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            L.check(self.lib, self.lib.tcr_create(C.byref(c), C.byref(self._h)), "tcr_create")
        self.info = L.TcrInfo()
        L.check(self.lib, self.lib.tcr_get_info(self._h, C.byref(self.info)), "tcr_get_info")
        self.num_trainable = int(self.info.num_trainable)
        self.num_moving = int(self.info.num_moving)
        self.frames, self.features = int(self.info.frames), int(self.info.features)
        self.num_classes = int(num_classes)
        self.table = self._read_table()
        self.world_size = 1

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_h", None):
            self.lib.tcr_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _read_table(self):
        descs = C.POINTER(L.TcrParamDesc)()
        n = C.c_int32()
        L.check(self.lib, self.lib.tcr_param_table(self._h, C.byref(descs), C.byref(n)), "tcr_param_table")
        return [dict(name=descs[i].name.decode(), kind=L.KIND_NAMES[descs[i].kind], trainable=descs[i].kind < 3,
                     shape=tuple(descs[i].shape[:descs[i].rank]), offset=int(descs[i].offset),
                     numel=int(descs[i].numel)) for i in range(n.value)]

    def _f32(self, *shape):
        return torch.empty(shape, dtype=torch.float32, device=self.device)

    @staticmethod
    def _ptr(t, dtype=torch.float32):
        if t is None:
            return None
        assert t.is_cuda and t.dtype == dtype and t.is_contiguous(), f"expected contiguous {dtype} CUDA tensor"
        return t.data_ptr()

    def _input(self, inputs, input_is_features):
        """(pointer, TCR_INPUT_* kind): fp32 wav, precomputed features, or int16 PCM (decode_wav scaling on device)."""
        n = inputs.shape[0]
        if input_is_features:
            return self._ptr(inputs), L.TCR_INPUT_FEATURES
        inputs = inputs.reshape(n, -1)
        if inputs.dtype == torch.int16:
            return self._ptr(inputs, torch.int16), L.TCR_INPUT_WAV_PCM16
        return self._ptr(inputs), L.TCR_INPUT_WAV_F32

    # ------------------------------------------------------------------ variables
    def new_variables(self, seed: int = 0):
        """(params, slots, moving): Xavier-uniform / gamma=1 / beta=0 / moving (0,1) / slots 0."""
        params, slots, moving = self._f32(self.num_trainable), self._f32(self.num_trainable), self._f32(self.num_moving)
        L.check(self.lib, self.lib.tcr_init_variables(self._h, self._ptr(params), self._ptr(slots), self._ptr(moving),
                                                      seed, self._stream), "tcr_init_variables")
        return params, slots, moving

    def new_optimizer_state(self, optimizer: Optimizer, params: torch.Tensor, slots: Optional[torch.Tensor] = None) -> OptimizerState:
        """The state `optimizer` starts from, as TF initialises it: momentum accumulators, Adam m / v at zero and the beta powers at
        beta1 / beta2, RMSProp ms at ONES and mom at zero, EMA shadows a copy of `params`.  `slots` (e.g. from new_variables) is
        reused as the first slot buffer when given."""
        n = params.numel()
        new = lambda v: torch.full((n,), float(v), dtype=torch.float32, device=params.device)
        first = slots if slots is not None else new(0.0)
        st = OptimizerState(slots=first)
        if optimizer.kind == "adam":
            first.zero_()
            st.slots2 = new(0.0)
            st.scalars = torch.tensor([optimizer.beta1, optimizer.beta2], dtype=torch.float32, device=params.device)
        elif optimizer.kind == "rmsprop":
            first.fill_(1.0)
            st.slots2 = new(0.0)
        if optimizer.ema_decay is not None:
            st.ema = params.detach().clone()
        return st

    def variables_to_dict(self, params: torch.Tensor, moving: Optional[torch.Tensor] = None) -> Dict[str, np.ndarray]:
        """{TF variable name: ndarray} — the reference's `var_names_to_values` form (helper/trainer.py:145-154)."""
        p = params.detach().cpu().numpy()
        m = moving.detach().cpu().numpy() if moving is not None else None
        out = {}
        for d in self.table:
            src = p if d["trainable"] else m
            if src is not None:
                out[d["name"]] = src[d["offset"]:d["offset"] + d["numel"]].reshape(d["shape"]).copy()
        return out

    def variables_from_dict(self, values: Dict[str, np.ndarray], params: torch.Tensor, moving: Optional[torch.Tensor] = None,
                            strict: bool = True):
        p = params.detach().cpu().numpy().copy()
        m = moving.detach().cpu().numpy().copy() if moving is not None else None
        for d in self.table:
            if d["name"] not in values:
                if strict:
                    raise KeyError(d["name"])
                continue
            dst = p if d["trainable"] else m
            if dst is None:
                continue
            v = np.asarray(values[d["name"]], np.float32)
            if v.size != d["numel"]:
                raise ValueError(f"{d['name']}: expected {d['shape']}, got {v.shape}")
            dst[d["offset"]:d["offset"] + d["numel"]] = v.ravel()
        params.copy_(torch.from_numpy(p))
        if moving is not None:
            moving.copy_(torch.from_numpy(m))

    # ------------------------------------------------------------------ the three calls
    def mfcc(self, wav: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        wav = wav.reshape(wav.shape[0], -1)
        n = wav.shape[0]
        out = out if out is not None else self._f32(n, self.frames, self.features)
        if wav.dtype == torch.int16:
            L.check(self.lib, self.lib.tcr_mfcc_forward_pcm16(self._h, self._ptr(wav, torch.int16), self._ptr(out), n, self._stream),
                    "tcr_mfcc_forward_pcm16")
        else:
            L.check(self.lib, self.lib.tcr_mfcc_forward(self._h, self._ptr(wav), self._ptr(out), n, self._stream),
                    "tcr_mfcc_forward")
        return out

    def augment(self, pcm: torch.Tensor, clips: torch.Tensor, background: Optional[torch.Tensor] = None,
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Device input stage (datasets/augmentation_factory.py): int16 clips [n, stride] + per-clip draws -> fp32 wav
        [n, clip_samples].  `clips`: uint8 CUDA tensor holding n packed tcr_augment_clip records (24 bytes each, see
        include/tcr_b200.h); `background`: the background recordings concatenated (fp32) or None."""
        n = pcm.shape[0]
        assert pcm.is_cuda and pcm.dtype == torch.int16 and pcm.is_contiguous()
        assert clips.is_cuda and clips.dtype == torch.uint8 and clips.numel() == 24 * n
        out = out if out is not None else self._f32(n, self.cfg.clip_samples)
        L.check(self.lib, self.lib.tcr_augment_pcm16(self._h, pcm.data_ptr(), pcm.shape[1], clips.data_ptr(), self._ptr(background),
                                                     self._ptr(out), n, self._stream), "tcr_augment_pcm16")
        return out

    def forward(self, inputs: torch.Tensor, params: torch.Tensor, moving: Optional[torch.Tensor] = None,
                is_training: bool = False, onehot: Optional[torch.Tensor] = None, weight_decay: float = 0.0,
                dropout_seed: int = 0, dropout_mask: Optional[torch.Tensor] = None, input_is_features: bool = False):
        n = inputs.shape[0]
        in_ptr, in_kind = self._input(inputs, input_is_features)
        logits, probs = self._f32(n, self.num_classes), self._f32(n, self.num_classes)
        losses = self._f32(2) if onehot is not None else None
        L.check(self.lib, self.lib.tcr_forward(self._h, in_ptr, in_kind, self._ptr(params),
                                               self._ptr(moving), n, int(is_training), int(dropout_seed),
                                               self._ptr(dropout_mask), self._ptr(onehot), float(weight_decay),
                                               self._ptr(logits), self._ptr(probs), self._ptr(losses), self._stream),
                "tcr_forward")
        return dict(logits=logits, probs=probs, losses=losses)

    def train_step(self, inputs: torch.Tensor, onehot: torch.Tensor, params: torch.Tensor, slots: torch.Tensor,
                   moving: torch.Tensor, learning_rate: float, momentum: float = 0.9, weight_decay: float = 1e-4,
                   dropout_seed: int = 0, dropout_mask: Optional[torch.Tensor] = None, input_is_features: bool = False,
                   want_outputs: bool = False, want_grads: bool = False, apply_update: bool = True,
                   losses: Optional[torch.Tensor] = None, clips: Optional[torch.Tensor] = None,
                   background: Optional[torch.Tensor] = None, input_resident: bool = False,
                   optimizer: Optional[Optimizer] = None, state: Optional[OptimizerState] = None):
        """optimizer / state: the update rule and its buffers (new_optimizer_state); without them the step is SGD-momentum with
        `momentum` on `slots`.  With a state, `slots` may be None (state.slots is used).
        clips (uint8 CUDA tensor of n packed tcr_augment_clip records) + int16 `inputs` [n, stride]: the step starts with
        the device input stage (decode, shift, background mix, clip) instead of taking decoded fp32 samples.
        input_resident=True: `inputs` is final when the call is made (nothing queued on the current stream writes it); the
        front-end then runs ahead on the library's own stream and overlaps the previous step's tail (tcr_step_args::input_resident)."""
        n = inputs.shape[0]
        a = L.TcrStepArgs()
        if clips is not None:
            assert inputs.dtype == torch.int16 and inputs.is_cuda and inputs.is_contiguous() and clips.numel() == 24 * n
            a.input, a.input_is_features = inputs.data_ptr(), L.TCR_INPUT_WAV_PCM16
            a.clips, a.background, a.pcm_stride = clips.data_ptr(), self._ptr(background), inputs.shape[1]
        else:
            a.input, a.input_is_features = self._input(inputs, input_is_features)
        a.onehot, a.n = self._ptr(onehot), n
        a.params, a.moving = self._ptr(params), self._ptr(moving)
        _set_rule(a, self._ptr, slots, momentum, optimizer, state)
        a.learning_rate, a.weight_decay = float(learning_rate), float(weight_decay)
        a.dropout_seed, a.dropout_mask = int(dropout_seed), self._ptr(dropout_mask)
        losses = losses if losses is not None else self._f32(2)
        out = dict(losses=losses)
        a.losses = self._ptr(losses)
        if want_outputs:
            out["logits"], out["probs"] = self._f32(n, self.num_classes), self._f32(n, self.num_classes)
            a.logits, a.probs = self._ptr(out["logits"]), self._ptr(out["probs"])
        if want_grads:
            out["grads"] = self._f32(self.num_trainable)
            a.grads = self._ptr(out["grads"])
        a.apply_update = int(apply_update)
        a.input_resident = int(bool(input_resident))
        L.check(self.lib, self.lib.tcr_train_step(self._h, C.byref(a), self._stream), "tcr_train_step")
        return out

    def eval_accumulate(self, scores: torch.Tensor, onehot: torch.Tensor, counts: Optional[torch.Tensor] = None, topk: int = 5) -> torch.Tensor:
        """Adds one batch to the device-resident evaluation counts (int64 [C*C + 2]: confusion matrix, top-k hits, samples);
        see tcr_eval_accumulate in include/tcr_b200.h.  metrics.manager.metrics_from_counts turns them into the reference's metrics."""
        n, c = scores.shape[0], self.num_classes
        if counts is None:
            counts = torch.zeros(c * c + 2, dtype=torch.int64, device=self.device)
        assert counts.is_cuda and counts.dtype == torch.int64 and counts.numel() == c * c + 2
        L.check(self.lib, self.lib.tcr_eval_accumulate(self._h, self._ptr(scores), self._ptr(onehot), n, int(topk), counts.data_ptr(),
                                                       self._stream), "tcr_eval_accumulate")
        return counts

    # ------------------------------------------------------------------ data parallel
    def set_sync_bn(self, enable: bool = True):
        """Parity-test flag (SURVEY.md 8(e)): BatchNorm statistics over the global batch of all ranks (= one device with batch
        world * n).  Needs attach_process_group() first; the step then runs on the per-layer kernels with one small NCCL all-reduce
        per BN layer, forward and backward.  The default (local statistics) is what production runs use."""
        L.check(self.lib, self.lib.tcr_comm_set_sync_bn(self._h, int(bool(enable))), "tcr_comm_set_sync_bn")

    def attach_process_group(self):
        """One NCCL communicator per handle; the 128-byte unique id travels through torch.distributed."""
        import torch.distributed as dist
        world, rank = dist.get_world_size(), dist.get_rank()
        if world == 1:
            return
        from .dp import broadcast_bytes
        buf = (C.c_char * 128)()
        if rank == 0:
            L.check(self.lib, self.lib.tcr_comm_unique_id(buf), "tcr_comm_unique_id")
        idbuf = (C.c_char * 128).from_buffer_copy(broadcast_bytes(bytes(buf) if rank == 0 else None))
        with torch.cuda.device(self.device):
            L.check(self.lib, self.lib.tcr_comm_init(self._h, idbuf, rank, world), "tcr_comm_init")
        self.world_size = world
        self.exchange = "nccl"
        # Peer-memory exchange (same node, <= 8 ranks): the update kernel sums the ranks' gradients itself over NVLink
        # (include/tcr_b200.h, tcr_comm_p2p_*).  Every rank must take the same branch, hence the all_gather of the outcome.
        import os
        if world <= 8 and os.environ.get("TCR_P2P", "1") != "0":
            mine = (C.c_char * 128)()
            with torch.cuda.device(self.device):
                ok = self.lib.tcr_comm_p2p_export(self._h, mine) == 0
            gathered = [None] * world
            dist.all_gather_object(gathered, bytes(mine) if ok else None)
            if all(g is not None for g in gathered):
                table = (C.c_char * (128 * world)).from_buffer_copy(b"".join(gathered))
                with torch.cuda.device(self.device):
                    ok = self.lib.tcr_comm_p2p_attach(self._h, table, rank, world) == 0
            else:
                ok = False
            outcome = [None] * world
            dist.all_gather_object(outcome, bool(ok))
            if all(outcome):
                self.exchange = "peer-memory"
            else:                                     # someone could not export / map a peer: everybody stays on NCCL
                with torch.cuda.device(self.device):
                    self.lib.tcr_comm_p2p_detach(self._h)

    # ------------------------------------------------------------------ accounting
    def launch_count(self) -> int:
        n = C.c_uint64()
        self.lib.tcr_launch_count(C.byref(n))
        return int(n.value)

    def profile(self, enable: bool):
        self.lib.tcr_profile_enable(int(enable))

    def profile_read(self):
        stats = C.POINTER(L.TcrKernelStat)()
        n = C.c_int32()
        L.check(self.lib, self.lib.tcr_profile_read(C.byref(stats), C.byref(n)), "tcr_profile_read")
        return {stats[i].name.decode(): (float(stats[i].total_ms), int(stats[i].launches)) for i in range(n.value)}

    def fp32_peak_tflops(self) -> float:
        v = C.c_double()
        L.check(self.lib, self.lib.tcr_measure_fp32_peak(self._h, C.byref(v), self._stream), "tcr_measure_fp32_peak")
        return float(v.value)


class HostFeed:
    """Host-buffer feed around the C ABI's tcr_train_step_host (the `session.run(train_op)` loop of
    helper/trainer.py:132-154 with the input pipeline's prefetch, datasets/data_wrapper_base.py:100-108).

    submit() hands one pinned host batch (fp32 wav, int16 PCM, or features) to the library, which copies it H2D on its
    own copy stream into a staging slot, runs the step behind the copy and reads the two losses back.  The call does
    not wait for the step it submits: it returns (step_index, total_loss, model_loss) of the step `lag` submissions
    earlier (None while the pipeline fills), so copies, launches and compute of neighbouring steps overlap while every
    step's input still crosses the bus and every step's loss reaches the host.  flush() drains what is outstanding.
    """

    def __init__(self, engine: "Engine", lag: int = 2):
        self.eng, self.lag = engine, int(lag)
        self._out = (C.c_float * 2)()
        self._step = C.c_int64(-1)

    def _result(self):
        return None if self._step.value < 0 else (int(self._step.value), float(self._out[0]), float(self._out[1]))

    def submit(self, h_inputs: torch.Tensor, h_onehot: torch.Tensor, params, slots, moving, learning_rate, momentum=0.9,
               weight_decay=1e-4, dropout_seed=0, input_is_features=False, h_clips: Optional[torch.Tensor] = None,
               background: Optional[torch.Tensor] = None, optimizer: Optional[Optimizer] = None,
               state: Optional[OptimizerState] = None):
        """h_clips (pinned uint8 tensor of n packed tcr_augment_clip records, datasets/device_input_stage.py) with int16
        h_inputs [n, stride]: the wav files' samples and the per-clip draws cross the bus; the input stage runs on the device
        (`background`: the CUDA-resident bank).  optimizer / state: as Engine.train_step."""
        eng = self.eng
        assert h_inputs.is_pinned() and h_onehot.is_pinned() and h_inputs.is_contiguous(), "HostFeed needs pinned host tensors"
        a = L.TcrStepArgs()
        a.input = h_inputs.data_ptr()
        a.input_is_features = (L.TCR_INPUT_FEATURES if input_is_features else
                               L.TCR_INPUT_WAV_PCM16 if h_inputs.dtype == torch.int16 else L.TCR_INPUT_WAV_F32)
        a.onehot, a.n = h_onehot.data_ptr(), h_inputs.shape[0]
        if h_clips is not None:
            assert h_clips.is_pinned() and h_clips.dtype == torch.uint8 and h_inputs.dtype == torch.int16
            a.clips, a.background, a.pcm_stride = h_clips.data_ptr(), eng._ptr(background), h_inputs.shape[1]
        a.params, a.moving = eng._ptr(params), eng._ptr(moving)
        _set_rule(a, eng._ptr, slots, momentum, optimizer, state)
        a.learning_rate, a.weight_decay = float(learning_rate), float(weight_decay)
        a.dropout_seed, a.apply_update = int(dropout_seed), 1
        L.check(eng.lib, eng.lib.tcr_train_step_host(eng._h, C.byref(a), self.lag, eng._stream, self._out, C.byref(self._step)),
                "tcr_train_step_host")
        return self._result()

    def flush(self):
        """Drain the pipeline: list of (step_index, total_loss, model_loss) for every outstanding step."""
        out = []
        while True:
            L.check(self.eng.lib, self.eng.lib.tcr_host_flush(self.eng._h, self._out, C.byref(self._step)), "tcr_host_flush")
            r = self._result()
            if r is None:
                return out
            out.append(r)
