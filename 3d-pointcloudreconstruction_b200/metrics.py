"""Evaluation-metric glue of the hot path (mirrors utils/metrics.py): EMD (eps=0.005, iters=50) and Chamfer
distance, both x100, plus the registry / best-value comparison the eval drivers use.  certified_emd_distance is an
extra: the EMD of a true matching with a bound on its distance from the optimum."""
import logging

import torch

try:
    from .dist_chamfer_3D import chamfer_3DDist
    from . import emd_module as emd_func
except ImportError:
    from dist_chamfer_3D import chamfer_3DDist
    import emd_module as emd_func


def certified_emd_distance(pred, gt, eps_end=1e-4):
    """EMD of pred against gt with a certificate, x100 like Metrics._get_emd_distance: returns (value, gap).

    value = sqrt(dist).mean(1).mean() * 100 over the epsilon-scaled auction's matching (emd_module.emd_certified);
    gap = mean over the clouds of (upper - lower) * 100, a bound on how far value can be from the batch mean of the
    optimal EMDs.  gap is NaN when a cloud did not end with a matching."""
    with torch.no_grad():
        dist, _, bounds, _ = emd_func.emd_certified(pred, gt, eps_end=eps_end)
        value = torch.sqrt(dist).mean(1).mean().item() * 100
        gap = (bounds[:, 1] - bounds[:, 0]).mean().item() * 100
    return value, gap


class Metrics(object):
    ITEMS = [
        {"name": "EMD_distance", "enabled": True, "eval_func": "_get_emd_distance", "eval_object": emd_func.emdModule(),
         "is_greater_better": False, "init_value": 32767},
        {"name": "ChamferDistance", "enabled": True, "eval_func": "_get_chamfer_distance", "eval_object": chamfer_3DDist(),
         "is_greater_better": False, "init_value": 32767},
    ]

    @classmethod
    def get(cls, pred, gt):
        return [getattr(cls, item["eval_func"])(pred, gt) for item in cls.items()]

    @classmethod
    def items(cls):
        return [i for i in cls.ITEMS if i["enabled"]]

    @classmethod
    def names(cls):
        return [i["name"] for i in cls.items()]

    @classmethod
    def _get_emd_distance(cls, pred, gt):
        emd_1, _ = cls.ITEMS[0]["eval_object"](pred, gt, eps=0.005, iters=50)
        return torch.sqrt(emd_1).mean(1).mean().item() * 100

    @classmethod
    def _get_chamfer_distance(cls, pred, gt):
        dist1, dist2, _, _ = cls.ITEMS[1]["eval_object"](pred, gt)
        return (torch.mean(dist1) + torch.mean(dist2)).item() * 100

    def __init__(self, metric_name, values):
        self._items = Metrics.items()
        self._values = [item["init_value"] for item in self._items]
        self.metric_name = metric_name
        if isinstance(values, list):
            self._values = values
        elif isinstance(values, dict):
            index = {item["name"]: i for i, item in enumerate(self._items)}
            for k, v in values.items():
                if k not in index:
                    logging.warning("Ignore Metric[Name=%s] due to disability." % k)
                    continue
                self._values[index[k]] = v
        else:
            raise Exception("Unsupported value type: %s" % type(values))

    def state_dict(self):
        return {item["name"]: self._values[i] for i, item in enumerate(self._items)}

    def __repr__(self):
        return str(self.state_dict())

    def better_than(self, other):
        if other is None:
            return True
        idx = next((i for i, it in enumerate(self._items) if it["name"] == self.metric_name), -1)
        if idx == -1:
            raise Exception("Invalid metric name to compare.")
        mine, theirs = self._values[idx], other._values[idx]
        return mine > theirs if self._items[idx]["is_greater_better"] else mine < theirs
