"""Trainer of the EMA variant.  Interface of reference ``index_improve/trainer.py`` (Trainer :16-280): the base loop with
``model(data, use_ema=True)`` in the training step (:119) and the codebook utilisation of every level in the evaluation
log (:162-171, :221-253).  The NPU cache housekeeping of :131-132 has no counterpart here."""
from __future__ import annotations

import numpy as np

from ..dp_trainer import DataParallelTrainer as _DataParallelTrainer
from ..trainer import Trainer as _BaseTrainer
from ..utils import set_color


class Trainer(_BaseTrainer):
    def _model_forward(self, data):
        return self.model(data, use_ema=True)

    def _get_codebook_utilization(self):
        try:
            usage_stats = self.model.get_codebook_usage()
            return np.mean([stat["utilization"] for stat in usage_stats]), usage_stats
        except AttributeError:                    # a model without usage statistics (trainer.py:169-171)
            return None, None

    def _generate_valid_output(self, epoch_idx, seconds, collision_rate):
        avg_utilization, usage_stats = self._get_codebook_utilization()
        out = (set_color("epoch %d evaluating", "green") + " [" + set_color("time", "blue") + ": %.2fs, " +
               set_color("collision_rate", "blue") + ": %.4f") % (epoch_idx, seconds, collision_rate)
        if avg_utilization is not None:
            out += ", " + set_color("codebook_utilization", "blue") + ": %.4f" % avg_utilization
            for stat in usage_stats:
                out += (f"\n  Quantizer {stat['quantizer_id']}: {stat['utilization']:.4f} "
                        f"({stat['used_codes']}/{stat['total_codes']})")
        return out + "]"


class DataParallelTrainer(_DataParallelTrainer, Trainer):
    """Data-parallel training of the EMA variant over the GPUs of one box: the step of ``lcrec_b200.dp_trainer`` (one EMA
    step per level over the global batch, see ``DistributedEma``) with this variant's ``use_ema=True`` forward and its
    codebook-utilisation log."""
