"""Training driver with the reference's class names, flags and loop structure (helper/trainer.py:38-599).

What changes underneath: `build_train_op` does not assemble a gradient graph (slim.learning.create_train_op,
:199-222) — it arms the model so that fetching the train op in `session.run` executes ONE fused CUDA training step
(front-end, forward, backward, optimizer update, BN moving averages).  The learning rate is
tf.train.piecewise_constant(global_step, boundaries, lr_list) (:135) evaluated on the host per step.
Optimizers (:171-197): "mom" (the TC-ResNet recipes), "gd" (= momentum 0), "adam" (the CLI default) and "rmsprop" all run in
the fused step's update kernel; --use_ema adds tf.train.ExponentialMovingAverage(--ema_decay) shadows of the trainables,
updated in the same kernel after the optimizer (:213-217).
"""
from __future__ import annotations

import dataclasses
import sys
import time
from pathlib import Path

from ..common import checkpoint as ckpt
from ..common import utils
from ..engine import Optimizer
from ..metrics.manager import AudioMetricManager
from ..runtime import InvalidArgumentError, Node, no_op
from .base import AudioBase


def piecewise_constant(step, boundaries, values):
    for b, v in zip(boundaries, values):
        if step <= b:
            return v
    return values[-1]


class TrainerBase:
    def __init__(self, model, session, args, dataset, dataset_name, name):
        self.model, self.session, self.args = model, session, args
        self.dataset, self.dataset_name = dataset, dataset_name
        self.log = utils.get_logger(name)
        self.timer = utils.Timer(self.log)
        # data parallel (one process per GPU): every rank steps, rank 0 alone writes checkpoints (the replicas are identical;
        # BN moving statistics are rank 0's) and everybody waits for it, so no rank runs ahead into the next exchange alone
        self.rank, self.world = 0, 1
        if getattr(args, "data_parallel", False):
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                self.rank, self.world = dist.get_rank(), dist.get_world_size()
        self.is_chief = self.rank == 0

    # ---- setup -------------------------------------------------------------------------------
    def setup_essentials(self, max_to_keep=5):
        self.no_op = no_op()
        self.args.checkpoint_path = ckpt.resolve_checkpoint_path(self.args.checkpoint_path)
        self.train_dir_name = (Path.cwd() / Path(self.args.train_dir)).resolve()
        self.global_step_from_checkpoint = ckpt.checkpoint_step(self.args.checkpoint_path) if self.args.checkpoint_path else 0
        self.global_step = Node("global_step")
        self.model.global_step = self.global_step_from_checkpoint
        if self.args.boundaries_epoch:
            boundaries = [b * self.dataset.num_samples // (self.dataset.batch_size * self.world) for b in self.args.boundaries]
        else:
            boundaries = list(self.args.boundaries)
        if self.args.relative:
            self.boundaries = [self.global_step_from_checkpoint + b for b in boundaries]
            self.log.info(f"global_step starts with {self.global_step_from_checkpoint}, boundaries {boundaries} -> {self.boundaries}")
        else:
            self.boundaries = boundaries
        lr_list = list(self.args.lr_list)
        assert len(lr_list) == len(self.boundaries) + 1, "--lr_list needs one more entry than --boundaries"
        self.model.lr_schedule = lambda step: piecewise_constant(step, self.boundaries, lr_list)
        self.learning_rate_placeholder = Node("learning_rate")
        self.max_to_keep = max_to_keep

    def build_optimizer(self, optimizer, learning_rate, momentum=None, decay=None, epsilon=None):
        """The update rule with its hyper-parameters (engine.Optimizer).  Like the reference, momentum / decay / epsilon are
        forwarded to the TF optimizer only when truthy, so AdamOptimizer given --momentum or --optimizer_decay raises the same
        TypeError (it has no such argument); RMSProp takes all three.  "mom" and "gd" ignore the flags they do not use."""
        kwargs = {}
        if momentum:
            kwargs["momentum"] = momentum
        if decay:
            kwargs["decay"] = decay
        if epsilon:
            kwargs["epsilon"] = epsilon
        if optimizer == "mom":
            self.log.info("Use MomentumOptimizer")
            return Optimizer("mom", momentum=momentum if momentum is not None else 0.0)
        if optimizer == "gd":
            self.log.info("Use GradientDescentOptimizer")
            return Optimizer("gd", momentum=0.0)
        if optimizer == "adam":
            for bad in ("momentum", "decay"):
                if bad in kwargs:
                    raise TypeError(f"__init__() got an unexpected keyword argument '{bad}'")
            self.log.info("Use AdamOptimizer")
            return Optimizer.adam(**kwargs)
        if optimizer == "rmsprop":
            self.log.info("Use RMSPropOptimizer")
            return Optimizer.rmsprop(**kwargs)
        self.log.error(f"Unknown optimizer: {optimizer}")
        raise NotImplementedError

    def build_train_op(self, total_loss, optimizer, trainable_scopes, global_step, gradient_multipliers=None):
        if trainable_scopes:
            raise NotImplementedError("--trainable_scopes (partial training) is not supported by the fused step")
        if getattr(self.args, "use_ema", False):
            optimizer = dataclasses.replace(optimizer, ema_decay=float(self.args.ema_decay))
        self.model.set_optimizer(optimizer)
        return Node("train_op")

    def routine_restore_and_initialize(self, checkpoint_path=None):
        checkpoint_path = self.args.checkpoint_path if checkpoint_path is None else checkpoint_path
        values = getattr(self.model, "var_names_to_values", None)
        if values is not None:
            self.model.set_variables(values, strict=False)
            self.log.info("Restore from Memory")
        elif not checkpoint_path:
            self.log.info("Initialize global / local variables")
        else:
            self.model.set_variables(ckpt.load(checkpoint_path), strict=not self.args.ignore_missing_vars)
            self.log.info(f"Restored {checkpoint_path}")

    def setup_trainer(self):
        self.setup_essentials(self.args.max_to_keep)
        self.optimizer = self.build_optimizer(self.args.optimizer, learning_rate=self.learning_rate_placeholder,
                                              momentum=self.args.momentum, decay=self.args.optimizer_decay,
                                              epsilon=self.args.optimizer_epsilon)
        self.train_op = self.build_train_op(total_loss=self.model.total_loss, optimizer=self.optimizer,
                                            trainable_scopes=self.args.trainable_scopes, global_step=self.global_step)
        self.routine_restore_and_initialize()

    # ---- one step ----------------------------------------------------------------------------
    def build_epoch(self, step):
        return (step * self.dataset.batch_size * self.world) / self.dataset.num_samples

    def run_single_step(self, fetch_ops, feed_dict=None):
        t0 = time.perf_counter()
        vals = self.session.run(fetch_ops, feed_dict=feed_dict)
        ms = (time.perf_counter() - t0) * 1e3
        vals["single_step"], vals["single_step_per_instance"] = ms, ms / self.dataset.batch_size
        return vals

    def run_with_logging(self, summary_op, metric_op_dict, feed_dict):
        fetch_ops = {"step_op": self.train_op, "global_step": self.global_step,
                     "total_loss": self.model.total_loss, "model_loss": self.model.model_loss}
        if metric_op_dict:
            fetch_ops.update(metric_op_dict)
        vals = self.run_single_step(fetch_ops, feed_dict)
        global_step = int(vals["global_step"])
        step_from_restore = global_step - self.global_step_from_checkpoint
        epoch_from_restore = self.build_epoch(step_from_restore)
        lstep = int(getattr(self.model, "_last", {}).get("loss_global_step", global_step))   # host-feed pipeline: losses lag the submission
        if self.is_chief and (step_from_restore % max(1, self.args.step_save_summaries) == 0
                              or step_from_restore <= self.args.step_save_first_n_summaries):
            self.log.info(f"[{self.dataset_name}] GlobalStep {global_step:8d} / StepFromRestore {step_from_restore:8d} / "
                          f"EpochFromRestore {epoch_from_restore:3.3f} | "
                          + (f"(losses of step {int(lstep)}) " if lstep != global_step else "")
                          + f"TotalLoss {vals['total_loss']:.5f} / "
                          f"ModelLoss {vals['model_loss']:.5f} | SingleStep(ms) {vals['single_step']:.3f} / "
                          f"SingleStepPerInstance(ms) {vals['single_step_per_instance']:.5f}")
        return vals, global_step, step_from_restore, epoch_from_restore

    def save_checkpoint(self, global_step):
        path = None
        if self.is_chief:
            path = ckpt.save(self.args.train_dir, self.args.model, global_step, self.model.get_variables(), self.args.max_to_keep,
                             fmt=getattr(self.args, "checkpoint_format", "tf"))
            self.log.info(f"save checkpoint: {path}")
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        return path

    def train(self, name: str = "Training"):
        self.log.info(f"{name} started")
        global_step, step_from_restore, epoch_from_restore = 0, 0, 0
        while True:
            try:
                feed_dict = self.get_feed_dict(is_training=True)
                metric_ops = self.metric_tf_op if step_from_restore % self.args.step_evaluation == 0 else None
                _, global_step, step_from_restore, epoch_from_restore = self.run_with_logging(None, metric_ops, feed_dict)
                if step_from_restore % self.args.step_save_checkpoint == 0:
                    self.save_checkpoint(global_step)
                if step_from_restore % self.args.step_evaluation == 0:
                    self.evaluate(epoch_from_restore, step_from_restore, global_step, self.dataset_name)
                if epoch_from_restore >= self.args.max_epoch_from_restore:
                    self.log.info(f"Reached {self.args.max_epoch_from_restore} epochs from restore.")
                    break
                if step_from_restore >= self.args.max_step_from_restore:
                    self.log.info(f"Reached {self.args.max_step_from_restore} steps from restore.")
                    break
            except InvalidArgumentError as e:
                self.log.error(f"Invalid instance is detected: {e}")
                continue
        self.save_checkpoint(global_step)
        self.log.info(f"{name} finished")

    def evaluate(self, epoch_from_restore, step_from_restore, global_step, dataset_name, iters=None):
        """In-training evaluation: runs on the TRAINING graph (batch-statistics BN, dropout on), helper/trainer.py:436-460."""
        iters = self.build_evaluate_iterations(iters)
        with self.timer(f"run_evaluation (iterations: {iters})"):
            eval_dict = self.run_inference(global_step, iters=iters, is_training=True)
            data = self.build_non_tensor_data_from_eval_dict(eval_dict)
            self.metric_manager.evaluate_and_aggregate_metrics(step=global_step, non_tensor_data=data, eval_dict=eval_dict)
        if self.is_chief:
            self.metric_manager.log_metrics(global_step, self.log.info)

    @staticmethod
    def add_arguments(parser, name: str = "TrainerBase"):
        g = parser.add_argument_group(f"({name}) Optimizer Arguments")
        g.add_argument("--optimizer", default="adam", type=str, choices=["gd", "adam", "mom", "rmsprop"])
        g.add_argument("--momentum", default=None, type=float)
        g.add_argument("--optimizer_decay", default=None, type=float)
        g.add_argument("--optimizer_epsilon", default=None, type=float)
        g = parser.add_argument_group(f"({name}) Saver(Restore) Arguments")
        g.add_argument("--trainable_scopes", default="", type=str)
        g = parser.add_argument_group(f"({name}) Training options(step, batch_size, path) Arguments")
        g.add_argument("--train_dir", required=True, type=str)
        for flag, default in (("step_save_summaries", 10), ("step_save_verbose_summaries", 2000),
                              ("step_save_first_n_summaries", 30), ("step_save_checkpoint", 500), ("step_min_summaries", 0),
                              ("class_sampling_factor", 20), ("maximum_num_labels_for_metric", 10)):
            g.add_argument(f"--{flag}", default=default, type=int)
        g.add_argument("--step_evaluation", default=500, type=utils.positive_int)
        g.add_argument("--write_pbtxt", dest="write_pbtxt", action="store_true")
        g.add_argument("--no-write_pbtxt", dest="write_pbtxt", action="store_false")
        g.set_defaults(write_pbtxt=True)
        g.add_argument("--max_to_keep", default=5, type=utils.positive_int)
        g.add_argument("--max_outputs", default=5, type=utils.positive_int)
        g.add_argument("--max_epoch_from_restore", default=50000, type=float)
        g.add_argument("--max_step_from_restore", default=sys.maxsize, type=int)
        g = parser.add_argument_group("Learning Rate Scheduling Arguments")
        g.add_argument("--learning_rate", default=1e-4, type=float)
        g.add_argument("--boundaries", default=[100000, 200000], type=int, nargs="*")
        g.add_argument("--boundaries_epoch", dest="boundaries_epoch", action="store_true")
        g.add_argument("--no-boundaries_epoch", dest="boundaries_epoch", action="store_false")
        g.add_argument("--lr_list", default=[1e-3, 1e-4, 1e-5], type=float, nargs="*")
        g.add_argument("--relative_schedule", dest="relative", action="store_true")
        g.add_argument("--absolute_schedule", dest="relative", action="store_false")
        g.set_defaults(relative=True, boundaries_epoch=True)
        g.add_argument("--checkpoint_format", default="tf", choices=["tf", "npz"],
                       help="tf: tensor-bundle files like tf.train.Saver (<Model>-<step>.index/.data-*); npz: one NumPy archive")
        g = parser.add_argument_group("B200 data-parallel (no reference counterpart)")
        g.add_argument("--data_parallel", action="store_true",
                       help="one process per GPU under torchrun; gradients are averaged with one NCCL all-reduce per step")


class SingleLabelAudioTrainer(TrainerBase, AudioBase):
    def __init__(self, model, session, args, dataset, dataset_name, name="AudioTrainer"):
        super().__init__(model, session, args, dataset, dataset_name, name)
        self.label_names = self.dataset.label_names
        assert len(self.label_names) == self.args.num_classes
        self.use_class_metrics = len(self.label_names) < self.args.maximum_num_labels_for_metric
        self.setup_trainer()
        self.metric_manager = AudioMetricManager(is_training=True, use_class_metrics=self.use_class_metrics,
                                                 exclude_metric_names=self.args.exclude_metric_names)
        self.metric_tf_op = self.metric_manager.build_metric_ops({
            "dataset_split_name": self.dataset_name, "label_names": self.dataset.label_names,
            "losses": self.build_basic_loss_ops(), "learning_rate": self.learning_rate_placeholder,
            "wavs": self.model.audio_original})
        self.log.info(f"--checkpoint_path {self.train_dir_name}")

    def build_evaluate_iterations(self, iters):
        if iters is not None:
            return iters
        if self.args.evaluation_iterations is not None:
            return self.args.evaluation_iterations
        return max((self.args.class_sampling_factor * self.args.num_classes) // self.args.batch_size, 1)

    @staticmethod
    def add_arguments(parser):
        pass
