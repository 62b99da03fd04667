"""Evaluation driver with the reference's class names and flow (helper/evaluator.py:20-212): restore a checkpoint
by TF variable names, rewind the dataset, run `num_samples // batch_size` forward batches in eval mode (BN moving
statistics, dropout identity), aggregate metrics, keep the best checkpoint per metric in
`<train_dir>/<split>/<metric>/` (the path the test recipe reads, scripts/commands/*.sh line 7)."""
from __future__ import annotations

import shutil
import sys
from pathlib import Path

from ..common import checkpoint as ckpt
from ..common.utils import get_logger
from ..metrics.manager import AudioMetricManager
from .base import AudioBase


class Evaluator:
    def __init__(self, model, session, args, dataset, dataset_name, name):
        self.log = get_logger(name)
        self.model, self.session, self.args = model, session, args
        self.dataset, self.dataset_name = dataset, dataset_name
        if Path(self.args.checkpoint_path).is_dir():
            latest = ckpt.latest_checkpoint(self.args.checkpoint_path)
            if latest is not None:
                self.args.checkpoint_path = latest
            self.log.info(f"Get latest checkpoint and update to it: {self.args.checkpoint_path}")
        p = Path(self.args.checkpoint_path)
        self.watch_path = p if p.is_dir() else p.parent
        self.best = {}

    def build_evaluation_step(self, checkpoint_path):
        return ckpt.checkpoint_step(checkpoint_path)

    def evaluate_once(self, checkpoint_path):
        self.log.info("Evaluation started")
        self.setup_dataset_iterator()
        values = ckpt.load(checkpoint_path)
        if getattr(self.args, "use_ema", False):       # trainables from their EMA shadows (common/model_loader.py:62-67)
            self.model.set_variables_from_ema(values, strict=not self.args.ignore_missing_vars)
        else:
            self.model.set_variables(values, strict=not self.args.ignore_missing_vars)
        step = self.build_evaluation_step(str(checkpoint_path))
        self.model.global_step = step
        metrics = self.run_evaluation(step, is_training=False)
        keep = self.metric_manager.filter_best_keep_metric(metrics)
        if self.args.save_best_keeper:
            self.keep_best(keep, str(checkpoint_path), step)
        self.metric_manager.log_metrics(step, self.log.info)
        self.log.info("Evaluation finished")
        if step >= self.args.max_step_from_restore:
            self.log.info("Evaluation stopped")
            sys.exit()
        return metrics

    def keep_best(self, keep, checkpoint_path, step):
        modes = self.metric_manager.get_best_keep_metric_with_modes()
        for key, value in keep.items():
            better = key not in self.best or (value > self.best[key] if modes[key] == "max" else value < self.best[key])
            if better:
                self.best[key] = value
                target = self.watch_path / self.dataset_name / key
                target.mkdir(parents=True, exist_ok=True)
                for old in list(target.glob("*.npz")) + list(target.glob("*.index")) + list(target.glob("*.data-*")):
                    old.unlink()
                ckpt.copy_checkpoint(checkpoint_path, target)
                (target / "scores.txt").write_text(f"step\t{step}\n{key}\t{value}\nmodel_size\t{self.model.total_params}\n")

    @staticmethod
    def add_arguments(parser):
        g = parser.add_argument_group("(Evaluator) arguments")
        g.add_argument("--valid_type", default="loop", type=str, choices=["loop", "once"])
        g.add_argument("--max_outputs", default=5, type=int)
        g.add_argument("--maximum_num_labels_for_metric", default=10, type=int)
        g.add_argument("--save_best_keeper", dest="save_best_keeper", action="store_true")
        g.add_argument("--no-save_best_keeper", dest="save_best_keeper", action="store_false")
        g.set_defaults(save_best_keeper=True)
        g.add_argument("--flatten_output", dest="flatten_output", action="store_true")
        g.add_argument("--no-flatten_output", dest="flatten_output", action="store_false")
        g.set_defaults(flatten_output=False)
        g.add_argument("--max_step_from_restore", default=int(1e20), type=int)


class SingleLabelAudioEvaluator(Evaluator, AudioBase):
    def __init__(self, model, session, args, dataset, dataset_name):
        super().__init__(model, session, args, dataset, dataset_name, "SingleLabelAudioEvaluator")
        assert len(self.dataset.label_names) == self.args.num_classes
        self.use_class_metrics = len(self.dataset.label_names) < self.args.maximum_num_labels_for_metric
        self.metric_manager = AudioMetricManager(is_training=False, use_class_metrics=self.use_class_metrics,
                                                 exclude_metric_names=self.args.exclude_metric_names)
        self.metric_tf_op = self.metric_manager.build_metric_ops({
            "dataset_split_name": self.dataset_name, "label_names": self.dataset.label_names,
            "losses": self.build_basic_loss_ops(), "learning_rate": None, "wavs": self.model.audio_original})

    def setup_dataset_iterator(self):
        self.dataset.setup_iterator(self.session, self.dataset.placeholders, self.dataset.data)
