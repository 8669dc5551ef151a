"""Validation metrics of the reference script on the device (SURVEY.md 8f-4): one kernel per batch instead of the ~40 eager ops,
two `get_pflow` calls, `nonzero()` filtering and torchmetrics objects of dss2_run.py:183-209.  The metric formulas live in that kernel's
finaliser (csrc/wls.cu, `dss2_eval_metrics_acc`), which both this module and the captured evaluator (dss2.evaluator) read."""
import torch

from . import _lib
from .ops import require_cuda, stage_rows

_WS = {}

# the ten metrics of one batch, in the order of the finaliser's accumulator (acc11[0..9]; acc11[10] counts the batches)
KEYS = ("rmse_v", "mae_v", "rmse_th", "mae_th", "rmse_loading", "mae_loading", "rmse_loading_trafos", "mae_loading_trafos",
        "prop_std_v", "prop_std_th")


def epoch_means(acc):
    """Host dict of an fp64 accumulator [11]: acc[k] / acc[10] per metric (the script's mean over batches) and "batches".
    One device-to-host copy."""
    a = acc.cpu().tolist()
    nb = a[10]
    res = {k: (a[i] / nb if nb else float("nan")) for i, k in enumerate(KEYS)}
    res["batches"] = int(nb)
    return res


def evaluate_batch(out, y, x, edge_index, edge_attr, x_mean, x_std):
    """Metrics of ONE validation batch, i.e. the terms dss2_run.py:186-205 adds up per batch (the script then averages them over
    the loader).  out [Nt,2] = model output (normalised V, raw theta; NOT modified), y [Nt,2] labels, x [Nt,11] and edge_attr [Et,13]
    the full feature tensors of the batch, x_mean / x_std the dataset statistics.  Returns a dict of python floats:
    rmse_v, mae_v, rmse_th, mae_th, rmse_loading, mae_loading, rmse_loading_trafos, mae_loading_trafos, prop_std_v, prop_std_th."""
    require_cuda()
    lib = _lib.load()
    og, os_ = stage_rows(out.detach())
    yg, ys = stage_rows(y)
    xg, xs = stage_rows(x)
    eg, es = stage_rows(edge_attr)
    if xg.size(1) < 11 or eg.size(1) < 13:
        raise _lib.Dss2Error("evaluate_batch needs the full x [Nt,11] and edge_attr [Et,13] tensors of the batch")
    ei = (edge_index if edge_index.device.type == "cuda" else edge_index.cuda(non_blocking=True)).long().contiguous()
    dev = xg.device
    with torch.cuda.device(dev):
        ws = _WS.get(dev.index)
        if ws is None:
            ws = _WS[dev.index] = torch.zeros(lib.dss2_eval_workspace_bytes(), dtype=torch.uint8, device=dev)
        vmm = torch.empty(2, dtype=torch.float32, device=dev)
        _lib.check(lib.dss2_col_minmax(_lib.ptr(xg), xs, 8, xg.size(0), _lib.ptr(vmm), _lib.stream()), "dss2_col_minmax")
        acc = torch.zeros(11, dtype=torch.float64, device=dev)     # one batch: its values / 1
        _lib.check(lib.dss2_eval_metrics_acc(_lib.ptr(ei), xg.size(0), ei.size(1), _lib.ptr(xg), xs, _lib.ptr(eg), es, _lib.ptr(og), os_,
                                             _lib.ptr(yg), ys, float(x_mean[0]), float(x_std[0]), _lib.ptr(vmm), _lib.ptr(acc),
                                             _lib.ptr(ws), ws.numel(), _lib.stream()), "dss2_eval_metrics_acc")
        res = epoch_means(acc)
    del res["batches"]
    return res
