"""Model builders with the reference's names and attribute surface (factory/audio_nets.py:19-183, 362-409),
executing on the CUDA engine instead of building a TF graph.

`train_audio.py` / `evaluate_audio.py` look the class up by NAME (`eval(f"audio_nets.{args.model}")`,
train_audio.py:32), call `Model(args, dataset)`, then `model.build(wavs, labels, is_training)` and hand the model
to the trainer / evaluator, which touch only the attributes set here and `session.run`.  TCResNet8Model and
TCResNet14Model are on the accelerated path; the other entries of `_available_nets` (baselines the north star
does not name) are registered so the CLI accepts them but raise NotImplementedError when built.
"""
from __future__ import annotations

from typing import Dict, Optional, Set

import numpy as np
import torch

from ..common import utils
from ..datasets import preprocessor_factory
from ..engine import Engine, Optimizer, OptimizerState
from ..runtime import InvalidArgumentError, Node
from .base import TFModel

# TF names of the per-variable optimizer state: `<var><suffix>` (slot_creator / ExponentialMovingAverage.average_name)
SLOT_SUFFIXES = {"mom": ("/Momentum",), "gd": ("/Momentum",), "adam": ("/Adam", "/Adam_1"), "rmsprop": ("/RMSProp", "/RMSProp_1")}
EMA_SUFFIX = "/ExponentialMovingAverage"

_available_nets = [
    "KWSModel", "Res8Model", "Res8NarrowModel", "Res15Model", "Res15NarrowModel", "DSCNNSModel", "DSCNNMModel",
    "DSCNNLModel", "TCResNet8Model", "TCResNet14Model", "ResNet2D8Model", "ResNet2D8PoolModel",
]


class AudioNetModel(TFModel):
    engine_model: Optional[str] = None      # set by the accelerated subclasses

    def __init__(self, args, dataset=None):
        self.log = utils.get_logger("AudioNetModel")
        self.args, self.dataset = args, dataset
        self.engine: Optional[Engine] = None
        self.global_step = 0
        self.optimizer = Optimizer("mom", momentum=0.9)             # set by the trainer (build_train_op -> set_optimizer)
        self.opt_state: Optional[OptimizerState] = None              # its device buffers (Engine.new_optimizer_state)
        self.lr_schedule = lambda step: getattr(args, "learning_rate", 1e-4)
        self.var_names_to_values = None                            # in-memory weight injection hook (trainer.py:145-154)
        self.endpoints_loss: Dict[str, Node] = {}
        self._last: Dict[str, np.ndarray] = {}
        self._feed, self._feed_last = None, (0, np.float32("nan"), np.float32("nan"))
        self._feed_steps = []                                       # global step numbers of the submitted, not yet reported steps
        self._feed_slots = []
        self._counts = None                                        # device int64 [classes^2 + 2] (tcr_eval_accumulate)

    # ------------------------------------------------------------------ graph-construction API of the reference
    def build(self, wavs, labels, is_training):
        self._audio_original, self.labels, self.is_training = wavs, labels, is_training
        self.preprocess_input()
        self.inputs, self.logits, self._outputs, self.endpoints = self.build_output(
            self.audio, self.is_training, self.args.output_name)
        self._total_loss, self._model_loss, self.endpoints_loss = self.build_loss(self.logits, self.outputs, self.labels)
        self.total_params = self.engine.num_trainable + self.engine.num_moving
        self.log.info(f"{type(self).__name__}: {self.engine.num_trainable} trainable parameters, "
                      f"{self.engine.info.forward_flops_per_utt / 1e6:.3f} MFLOP forward per utterance")
        if self.dataset is not None and getattr(self.dataset, "session", None) is not None:
            self.dataset.session.bind(self)

    def preprocess_input(self, for_deploy=False):
        a = self.args
        window = int(a.sample_rate * a.window_size_ms / 1000)
        stride = int(a.sample_rate * a.window_stride_ms / 1000)
        pre = preprocessor_factory.factory(preprocess_method=a.preprocess_method, scope="input/audio/preprocessing",
                                           preprocessed_node_name="input/audio/preprocessed")
        self._audio = pre.preprocess(self._audio_original, window_size_samples=window, window_stride_samples=stride,
                                     for_deploy=for_deploy, **vars(a))
        self._audio.name = "audio"
        self.log.info(f"Update height/width to {self._audio.shape}")
        a.height, a.width, a.channels = self._audio.shape[1:4]
        self.input_preprocessors_for_tflite = [pre]

    def build_output(self, inputs, is_training, output_name):
        logits, endpoints = self.build_inference(inputs, is_training=is_training)
        return inputs, logits, Node("outputs", [None, self.args.num_classes]), endpoints

    def build_inference(self, inputs, is_training=True):
        if self.engine_model is None:
            raise NotImplementedError(f"{type(self).__name__} is a baseline outside the accelerated TC-ResNet path")
        a = self.args
        self.engine = Engine(model=self.engine_model, width_multiplier=a.width_multiplier, num_classes=a.num_classes,
                             sample_rate=a.sample_rate, clip_duration_ms=a.clip_duration_ms,
                             window_size_ms=a.window_size_ms, window_stride_ms=a.window_stride_ms,
                             num_mel_bins=a.num_mel_bins, num_mfccs=a.num_mfccs, lower_edge_hertz=a.lower_edge_hertz,
                             upper_edge_hertz=a.upper_edge_hertz, preprocess_method=a.preprocess_method,
                             max_batch=max(int(getattr(a, 'batch_size', 1) or 1), int(getattr(a, 'input_batch_size', 1) or 1)),
                             dropout_keep_prob=a.dropout_keep_prob,
                             label_smoothing=getattr(a, "label_smoothing", 0.0))
        self.params, self.slots, self.moving = self.engine.new_variables(seed=getattr(a, "seed", 0) or 0)
        self.opt_state = OptimizerState(slots=self.slots)           # momentum until the trainer says otherwise (set_optimizer)
        if getattr(a, "data_parallel", False):
            self.engine.attach_process_group()
        n = int(getattr(a, 'batch_size', 1) or 1)
        dev = self.engine.device
        self._h_wav = torch.empty(n, self.engine.cfg.clip_samples, dtype=torch.float32).pin_memory()
        self._h_hot = torch.empty(n, a.num_classes, dtype=torch.float32).pin_memory()
        self._d_wav, self._d_hot = self._h_wav.to(dev), self._h_hot.to(dev)
        self._feed_slots = [(torch.empty_like(self._h_wav).pin_memory(), torch.empty_like(self._h_hot).pin_memory()) for _ in range(4)]
        return Node("logits", [None, a.num_classes]), {"ranges": Node("ranges")}

    def build_loss(self, logits, scores, labels):
        return Node("total_loss", []), Node("model_loss", []), {}

    def build_deployable_model(self, include_preprocess=True):
        """The deploy graph of the reference (factory/audio_nets.py:87-125: placeholder [input_batch_size, samples, 1] ->
        preprocessing -> network in inference mode -> softmax) as a callable on the CUDA engine: returns
        ([input node], DeployedModel).  include_preprocess=False takes features [1, height, width, 1] like the profiling graph.
        The front-end is the TRAINING front-end (tf.contrib.signal path, datasets/preprocessors.py:64-96): the reference's deploy
        front-end (audio_ops.mfcc, :98-158) is a different approximation of the same features and is not reproduced; TFLite
        conversion itself (freeze.py) stays out of scope."""
        a = self.args
        n = int(getattr(a, "input_batch_size", 1) or 1)
        if self.engine is None or int(self.engine.cfg.max_batch) < n:
            self.build_inference(None, is_training=False)
        samples = int(a.sample_rate * a.clip_duration_ms / 1000)
        if include_preprocess:
            node = Node("input/audio/before_preprocessing", [n, samples, 1])
        else:
            assert a.height > 0 and a.width > 0 and a.channels > 0
            node = Node("input", [1, a.height, a.width, a.channels])
        return [node], DeployedModel(self, n, include_preprocess)

    # ------------------------------------------------------------------ attribute surface
    @property
    def model_loss(self):
        return self._model_loss

    @property
    def total_loss(self):
        return self._total_loss

    @property
    def audio_original(self):
        return self._audio_original

    @property
    def audio(self):
        return self._audio

    @property
    def outputs(self):
        return self._outputs

    # ------------------------------------------------------------------ optimizer state
    def set_optimizer(self, optimizer: Optimizer):
        """Adopt the trainer's update rule (helper/trainer.py build_train_op) and create its state the way TF initialises it
        (Engine.new_optimizer_state); the existing slot buffer becomes its first slot."""
        self.optimizer = optimizer
        if self.engine is not None:
            self.flush_feed()
            self.opt_state = self.engine.new_optimizer_state(optimizer, self.params, self.slots)
            self.slots = self.opt_state.slots

    def _state_buffers(self):
        """(TF variable-name suffix, flat buffer) of every per-variable slot / shadow of the current rule."""
        st, kind = self.opt_state or OptimizerState(slots=self.slots), self.optimizer.kind
        out = [(s, b) for s, b in zip(SLOT_SUFFIXES[kind], (st.slots, st.slots2)) if b is not None]
        if self.optimizer.ema_decay is not None and st.ema is not None:
            out.append((EMA_SUFFIX, st.ema))
        return out

    # ------------------------------------------------------------------ variables by TF name
    def get_variables(self, with_slots=True) -> Dict[str, np.ndarray]:
        """Model variables, and with_slots=True the optimizer's state under TF's names: `<var>/Momentum`, `<var>/Adam` +
        `<var>/Adam_1` + `beta1_power` / `beta2_power`, `<var>/RMSProp` + `<var>/RMSProp_1`, `<var>/ExponentialMovingAverage`."""
        self.flush_feed()
        out = self.engine.variables_to_dict(self.params, self.moving)
        if with_slots:
            for suffix, buf in self._state_buffers():
                for k, v in self.engine.variables_to_dict(buf).items():
                    out[k + suffix] = v
            st = self.opt_state
            if self.optimizer.kind == "adam" and st is not None and st.scalars is not None:
                powers = st.scalars.detach().cpu().numpy()
                out["beta1_power"], out["beta2_power"] = np.float32(powers[0]).reshape(()), np.float32(powers[1]).reshape(())
        return out

    def set_variables(self, values: Dict[str, np.ndarray], strict=True):
        """Restore by TF name.  Optimizer state the checkpoint does not hold keeps its initial value."""
        self.flush_feed()
        self.engine.variables_from_dict(values, self.params, self.moving, strict=strict)
        for suffix, buf in self._state_buffers():
            slots = {k[:-len(suffix)]: v for k, v in values.items() if k.endswith(suffix)}
            if slots:
                self.engine.variables_from_dict(slots, buf, None, strict=False)
        st = self.opt_state
        if self.optimizer.kind == "adam" and st is not None and st.scalars is not None:
            for i, name in enumerate(("beta1_power", "beta2_power")):
                if name in values:
                    st.scalars[i] = float(np.asarray(values[name], np.float32).reshape(()))

    def set_variables_from_ema(self, values: Dict[str, np.ndarray], strict=True):
        """evaluate_audio.py --use_ema (common/model_loader.py:62-67, ExponentialMovingAverage.variables_to_restore): every
        trainable from its `<var>/ExponentialMovingAverage` shadow, everything else under its own name."""
        mapped = dict(values)
        for d in self.engine.table:
            if d["trainable"]:
                mapped.pop(d["name"], None)
                shadow = d["name"] + EMA_SUFFIX
                if shadow in values:
                    mapped[d["name"]] = values[shadow]
        self.set_variables(mapped, strict=strict)

    def _dropout_seed(self):
        """Counter-RNG seed of this step: distinct per rank under data parallelism (the kernel indexes utterances locally)."""
        world = getattr(self.engine, "world_size", 1)
        rank = getattr(self.dataset, "rank", 0) if world > 1 else 0
        return self.global_step * world + rank

    def read_metric_counts(self, reset: bool = True) -> np.ndarray:
        """Confusion matrix / top-5 hits / sample count accumulated by the forward passes since the last reset (one D2H read)."""
        if self._counts is None:
            return np.zeros(self.args.num_classes ** 2 + 2, np.int64)
        out = self._counts.cpu().numpy()
        if reset:
            self._counts.zero_()
        return out

    # ------------------------------------------------------------------ one session.run
    def _execute_train_fast(self, names: Set[str]) -> Optional[Dict[str, object]]:
        """session.run(train_op) through the host-buffer step of the C ABI (tcr_train_step_host via engine.HostFeed): the batch goes
        H2D on the library's copy stream, the step is queued behind it and the call returns without waiting for it.  The losses
        handed back are those of the step `feed_lag` calls earlier (`loss_global_step` says which), exactly the overlap the
        reference gets from tf.data prefetching + an asynchronous session (helper/trainer.py:312-321).  Used when nothing but
        the train op, losses, step and learning rate is fetched; metric / output fetches take the synchronous path below."""
        if names - {"train_op", "global_step", "total_loss", "model_loss", "learning_rate"}:
            return None
        lag = int(getattr(self.args, "feed_lag", 2))
        if lag <= 0:
            return None
        pinned = self.dataset.next_batch_pinned() if hasattr(self.dataset, "next_batch_pinned") else None
        if pinned is None:
            wav_np, hot_np = self.dataset.next_batch()
            n = wav_np.shape[0]
            if n != self.args.batch_size:
                raise InvalidArgumentError(f"bad batch: {wav_np.shape}")
            slot = self._feed_slots[self.global_step % len(self._feed_slots)]       # reused only after lag + 1 later calls
            slot[0].copy_(torch.from_numpy(wav_np.reshape(n, -1)))
            slot[1].copy_(torch.from_numpy(hot_np))
            pinned = slot
        if self._feed is None:
            from ..engine import HostFeed
            self._feed = HostFeed(self.engine, lag=lag)
        lr = float(self.lr_schedule(self.global_step))
        r = self._feed.submit(pinned[0], pinned[1], self.params, self.slots, self.moving, lr, weight_decay=self.args.weight_decay,
                              dropout_seed=self._dropout_seed(), optimizer=self.optimizer, state=self.opt_state)
        self.global_step += 1
        self._feed_steps.append(self.global_step)
        if r is not None:
            self._feed_last = (self._feed_steps.pop(0), np.float32(r[1]), np.float32(r[2]))
            if not np.isfinite(r[1]):
                raise InvalidArgumentError(f"non-finite loss at step {self._feed_last[0]} (malformed input batch?)")
        step, total, model = self._feed_last
        return {"train_op": None, "learning_rate": np.float32(lr), "global_step": np.int64(self.global_step), "total_loss": total,
                "model_loss": model, "loss_global_step": np.int64(step)}

    def flush_feed(self):
        """Drain the host-feed pipeline (before anything reads the variables: checkpoints, evaluation, get_variables)."""
        if self._feed is not None:
            for r in self._feed.flush():
                self._feed_last = (self._feed_steps.pop(0), np.float32(r[1]), np.float32(r[2]))

    def execute(self, names: Set[str], feed) -> Dict[str, object]:
        if "train_op" in names:
            fast = self._execute_train_fast(names)
            if fast is not None:
                self._last = fast
                return fast
        self.flush_feed()
        wav_np, hot_np = self.dataset.next_batch()
        n = wav_np.shape[0]
        if n != self.args.batch_size:
            raise InvalidArgumentError(f"bad batch: {wav_np.shape}")
        self._h_wav.copy_(torch.from_numpy(wav_np.reshape(n, -1)))
        self._h_hot.copy_(torch.from_numpy(hot_np))
        self._d_wav.copy_(self._h_wav, non_blocking=True)
        self._d_hot.copy_(self._h_hot, non_blocking=True)
        wd = self.args.weight_decay
        vals: Dict[str, object] = {}
        if "train_op" in names:
            lr = float(self.lr_schedule(self.global_step))
            out = self.engine.train_step(self._d_wav, self._d_hot, self.params, self.slots, self.moving, lr,
                                         weight_decay=wd, dropout_seed=self._dropout_seed(),
                                         want_outputs=bool(names & {"outputs", "logits"}), optimizer=self.optimizer,
                                         state=self.opt_state)
            self.global_step += 1
            vals["train_op"], vals["learning_rate"] = None, np.float32(lr)
        else:
            out = self.engine.forward(self._d_wav, self.params, self.moving, is_training=bool(self.is_training),
                                      onehot=self._d_hot, weight_decay=wd, dropout_seed=self._dropout_seed())
            vals["learning_rate"] = np.float32(self.lr_schedule(self.global_step))
        if "metric_counts" in names:                            # evaluation counts stay on the device until read_metric_counts()
            if self._counts is None:
                self._counts = torch.zeros(self.args.num_classes ** 2 + 2, dtype=torch.int64, device=self.engine.device)
            self.engine.eval_accumulate(out["probs"], self._d_hot, self._counts, topk=5)
            vals["metric_counts"] = None
        losses = out["losses"].cpu().numpy()                    # the D2H read synchronises the step
        vals.update(total_loss=losses[0], model_loss=losses[1], global_step=np.int64(self.global_step),
                    labels=hot_np, audio_original=wav_np)
        if "outputs" in names or "logits" in names:
            vals["outputs"], vals["logits"] = out["probs"].cpu().numpy(), out["logits"].cpu().numpy()
        if "audio" in names:
            feat = self.engine.mfcc(self._d_wav)
            vals["audio"] = feat.unsqueeze(-1).cpu().numpy()
        if "ranges" in names:
            vals["ranges"] = None       # dead `fc2` head: its forward is skipped (SURVEY.md 2b C6)
        self._last = vals
        return vals

    @staticmethod
    def add_arguments(parser):
        parser.add_argument("--label_smoothing", default=0.0, type=float)
        parser.add_argument("--feed_lag", default=2, type=int,
                            help="steps a training session.run may run ahead of the losses it reports (host-buffer step of the C ABI; "
                                 "0: synchronous steps, the loss returned is this step's)")


def _tc_flags(parser):
    parser.add_argument("--weight_decay", default=0.0001, type=float)
    parser.add_argument("--dropout_keep_prob", default=0.5, type=float)
    parser.add_argument("--width_multiplier", default=1.0, type=float)


class DeployedModel:
    """Batch-n (default 1) inference entry: wav [n, samples(,1)] or features [n, T, F(,1)] in, softmax outputs [n, classes] out.
    After the first call the launch sequence (front-end + every layer) is replayed from a CUDA graph: at batch 1 the forward is
    launch-latency bound (DESIGN.md section 6), and a graph replay is one submission instead of ~11 launches."""

    def __init__(self, model: "AudioNetModel", batch: int, include_preprocess: bool, use_graph: bool = True):
        self.model, self.batch, self.include_preprocess, self.use_graph = model, int(batch), include_preprocess, use_graph
        eng = model.engine
        shape = (self.batch, eng.cfg.clip_samples) if include_preprocess else (self.batch, eng.frames, eng.features)
        self._in = torch.zeros(shape, dtype=torch.float32, device=eng.device)
        self._graph, self._out, self._calls = None, None, 0

    def _run(self):
        m = self.model
        return m.engine.forward(self._in, m.params, m.moving, is_training=False, input_is_features=not self.include_preprocess)

    def __call__(self, x) -> np.ndarray:
        x = torch.as_tensor(np.asarray(x, np.float32)).reshape(self._in.shape)
        self._in.copy_(x, non_blocking=True)
        if not self.use_graph or self._calls < 2:                  # two eager calls first: lazy per-kernel attributes are set outside capture
            self._out = self._run()
        else:
            if self._graph is None:
                stream = torch.cuda.Stream(device=self._in.device)
                stream.wait_stream(torch.cuda.current_stream(self._in.device))
                with torch.cuda.stream(stream):
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=stream):
                        self._out = self._run()
                torch.cuda.current_stream(self._in.device).wait_stream(stream)
                self._graph = g
            self._graph.replay()
        self._calls += 1
        return self._out["probs"].cpu().numpy()


class TCResNet8Model(AudioNetModel):
    engine_model = "TCResNet8"
    add_arguments = staticmethod(_tc_flags)


class TCResNet14Model(AudioNetModel):
    engine_model = "TCResNet14"
    add_arguments = staticmethod(_tc_flags)


def _baseline(name, flags):
    def add_arguments(parser):
        for flag, default in flags:
            if isinstance(default, str):
                parser.add_argument(flag, default=default, type=str)
            else:
                parser.add_argument(flag, default=default, type=float)
    return type(name, (AudioNetModel,), {"add_arguments": staticmethod(add_arguments), "__doc__":
                "Baseline of the reference registered for CLI compatibility; not on the accelerated path."})


_TC = [("--weight_decay", 0.0001), ("--dropout_keep_prob", 0.5), ("--width_multiplier", 1.0)]
KWSModel = _baseline("KWSModel", [("--architecture", "conv")])
Res8Model = _baseline("Res8Model", [("--weight_decay", 0.00001)])
Res8NarrowModel = _baseline("Res8NarrowModel", [("--weight_decay", 0.00001)])
Res15Model = _baseline("Res15Model", [("--weight_decay", 0.00001)])
Res15NarrowModel = _baseline("Res15NarrowModel", [("--weight_decay", 0.00001)])
DSCNNSModel = _baseline("DSCNNSModel", [("--weight_decay", 0.0)])
DSCNNMModel = _baseline("DSCNNMModel", [("--weight_decay", 0.0)])
DSCNNLModel = _baseline("DSCNNLModel", [("--weight_decay", 0.0)])
ResNet2D8Model = _baseline("ResNet2D8Model", _TC)
ResNet2D8PoolModel = _baseline("ResNet2D8PoolModel", _TC)
