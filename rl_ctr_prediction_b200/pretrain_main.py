"""CTR pre-training loop API -- drop-in for the reference's ``src/main/pretrain_main.py``.

Same function names, argument meaning and return values (``setup_seed``, ``get_model``,
``get_dataset``, ``train``, ``test``, ``submission``, ``eva_stopping``, ``main``), so a script written
against the reference works after changing its import.  What changes:

* ``get_model`` builds the :mod:`.p_model` classes (fused-row tables + sm_100a kernels);
* ``main`` builds :class:`rl_ctr_prediction_b200.optim.Adam` where the reference builds
  ``torch.optim.Adam`` (:181) -- same arguments, fresh state every epoch like the reference;
* batches are sliced from one pinned int64 tensor (as ``src/all_main/pretrain_main_2.py:61,71-72``
  does) instead of 8 DataLoader worker processes;
* ``fused_train_step`` is the same step with the loss head inside the library (no per-op ATen
  launches); ``train(..., fused=True)`` uses it.

The reference's own ``train`` / ``test`` (which take the optimizer as an argument) also drive these
models unchanged; ``tests/test_gpu_loop.py`` checks exactly that.
"""
from __future__ import annotations

import ctypes as C
import datetime
import os
import random

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from . import optim as _optim
from . import p_model as Model
from .tables import table_struct


def setup_seed(seed):
    """pretrain_main.py:17-22."""
    torch.manual_seed(seed)
    if torch.cuda.is_available():
        torch.cuda.manual_seed_all(seed)
    np.random.seed(seed)
    random.seed(seed)
    torch.backends.cudnn.deterministic = True


_MODELS = {
    "LR": lambda n, f, d: Model.LR(n),
    "FM": lambda n, f, d: Model.FM(n, d),
    "FFM": lambda n, f, d: Model.FFM(n, f, d),
    "DeepFM": lambda n, f, d: Model.DeepFM(n, f, d),
    "W&D": lambda n, f, d: Model.WideAndDeep(n, f, d),
    "FNN": lambda n, f, d: Model.FNN(n, f, d),
    "IPNN": lambda n, f, d: Model.InnerPNN(n, f, d),
    "OPNN": lambda n, f, d: Model.OuterPNN(n, f, d),
    "DCN": lambda n, f, d: Model.DCN(n, f, d),
    "AFM": lambda n, f, d: Model.AFM(n, f, d),
}


def get_model(model_name, feature_nums, field_nums, latent_dims):
    """pretrain_main.py:25-45 (name -> class).  Names outside the hot-path scope raise instead of
    returning None as the reference silently does."""
    try:
        return _MODELS[model_name](int(feature_nums), int(field_nums), int(latent_dims))
    except KeyError:
        raise NotImplementedError(f"model {model_name!r} is outside this build's scope "
                                  f"(available: {sorted(_MODELS)})") from None


def load_encoded(path):
    """``train.txt`` (rows ``click,id_0..id_{F-1}``, the on-disk contract of src/encode/data_.py:85) as int64 [n, 1+F].
    The text is parsed once; a binary image ``<path>.int64.npy`` is kept beside it and memory-mapped on later runs
    (the reference re-parses the CSV with pandas on every start, src/main/pretrain_main.py:52; SURVEY 8f.2).  The image
    is rebuilt whenever the text file is newer."""
    cache = path + ".int64.npy"
    try:
        if os.path.exists(cache) and os.path.getmtime(cache) >= os.path.getmtime(path):
            return np.load(cache, mmap_mode="r")
    except (OSError, ValueError):
        pass
    data = np.loadtxt(path, delimiter=",", dtype=np.int64, ndmin=2)
    try:
        tmp = cache + ".tmp"
        with open(tmp, "wb") as fh:
            np.save(fh, data)
        os.replace(tmp, cache)
    except OSError:
        pass                                   # read-only data directory: keep parsing the text
    return data


def get_dataset(datapath, dataset_name, campaign_id, valid_day, test_day):
    """pretrain_main.py:47-88: ``train.txt`` rows ``click,id_0..id_{F-1}`` (src/encode/data_.py:85) and
    ``day_index.csv`` rows ``day,first_row,last_row``; train = every day but valid/test."""
    data_path = datapath + dataset_name + campaign_id
    train_fm = load_encoded(data_path + "train.txt")
    field_nums = train_fm.shape[1] - 1
    feature_nums = int(train_fm[:, 1:].max()) + 1
    day_indexs = np.loadtxt(data_path + "day_index.csv", delimiter=",", dtype=np.int64, ndmin=2)

    def rows_of(day):
        rec = day_indexs[day_indexs[:, 0] == day][0]
        return train_fm[rec[1]: rec[2] + 1]

    train_days = [d for d in day_indexs[:, 0].tolist() if d not in (valid_day, test_day)]
    train_data = np.concatenate([rows_of(d) for d in train_days], axis=0) if train_days else train_fm[:0]
    return train_fm, day_indexs, train_data, rows_of(valid_day), rows_of(test_day), field_nums, feature_nums


class BatchSlices:
    """Iterable of ``(features int64[b,F], labels int64[b])`` batches cut from one pinned tensor
    (the last batch is partial, like a DataLoader without ``drop_last``)."""

    def __init__(self, data: np.ndarray, batch_size: int):
        t = torch.from_numpy(np.ascontiguousarray(data.astype(np.int64)))
        self.data = t.pin_memory() if torch.cuda.is_available() else t
        self.batch_size = int(batch_size)

    def __len__(self):
        return (len(self.data) + self.batch_size - 1) // self.batch_size

    def __iter__(self):
        for s in range(0, len(self.data), self.batch_size):
            chunk = self.data[s: s + self.batch_size]
            yield chunk[:, 1:], chunk[:, 0]


def fused_train_step(model, optimizer, features, labels):
    """One training step of pretrain_main.py:96-102 with the loss head inside the library:
    sort -> catch-up -> gather+interaction -> sigmoid+BCE (+ their autograd) -> segment-reduce+Adam.
    Numerically the same step as ``loss(model(x), y); zero_grad(); backward(); optimizer.step()`` with
    ``nn.BCELoss``.  LR / FM / FFM run entirely in the library; models with a dense tail keep autograd for the tail
    (graphs.fused_logit_step).  Returns the loss (device scalar)."""
    if hasattr(model, "logit"):                 # DeepFM / W&D / FNN / IPNN / OPNN / DCN / AFM: autograd for the dense tail, fused head
        from . import graphs
        return graphs.fused_logit_step(model, optimizer, features, labels)
    lib = _lib.load()
    x = Model._check_ids(features)
    B, F = x.shape
    dev = x.device
    g = model._geom
    st = _lib.stream()
    y = labels.reshape(-1).contiguous()
    sid, sslot = Model.sort_ids(x, g.n_rows)
    opt = model._opt
    t = table_struct(model.table.data, g)
    ids_ptr, stage = _lib.ptr(x), None
    if opt is not None and opt.lookup_on:
        stage, gathered = Model.lookup_rows(model, (sid, sslot), x.numel(), F)
        t, ids_ptr = Model.gathered_struct(gathered, x.numel(), g), None
    elif opt is not None:
        opt.catchup(t, sid, x.numel(), type(model).__name__, model._meta(B, F))
    logit = torch.empty(B, dtype=torch.float32, device=dev)
    sums = partners = None
    if model._kind == "ffm":
        partners = torch.empty(B * F, g.row_stride, dtype=torch.float32, device=dev)
        _lib.call("rlctr_ffm_fwd", lib.rlctr_ffm_fwd, _lib.ptr(x), C.byref(t), _lib.ptr(model.bias.data), _lib.ptr(logit),
                  None, 1, _lib.ptr(partners), B, F, model.latent_dims, st, key="rlctr_ffm_fwd[train]",
                  meta=model._meta(B, F))
    else:
        if model._kind == "fm":
            sums = torch.empty(B, g.row_stride, dtype=torch.float32, device=dev)
        _lib.call("rlctr_embed_fwd", lib.rlctr_embed_fwd, ids_ptr, C.byref(t), _lib.ptr(model.bias.data),
                  _lib.ptr(logit), None, 1, _lib.ptr(sums), None, 0, B, F, _lib.RLCTR_FM_TERM if model._fm_term else 0, st,
                  key=f"rlctr_embed_fwd[{type(model).__name__}]",
                  meta=dict(model._meta(B, F), sums=sums is not None, rows=False, streamed=stage is not None))
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    dlogit = torch.empty(B, dtype=torch.float32, device=dev)
    dbias = torch.empty(1, dtype=torch.float32, device=dev)
    yi = y if y.dtype == torch.int64 else None
    yf = None if yi is not None else y.float()
    _lib.check(lib.rlctr_bce_fwd_bwd(_lib.ptr(logit), _lib.ptr(yi), _lib.ptr(yf), None, _lib.ptr(loss), _lib.ptr(dlogit),
                                     _lib.ptr(dbias), _lib.ptr(model._reduce_ws(dev)), B, st), "rlctr_bce_fwd_bwd")
    model._stash = Model.RowsStash(sorted_ids=sid, sorted_slots=sslot, n=B * F, dlogit=dlogit, sums=sums, extra=None,
                                   staged=partners, fields=F,
                                   flags=_lib.RLCTR_STAGED_PARTNER if partners is not None else 0, stage=stage)
    model.bias.grad = dbias
    optimizer.step()
    return loss.reshape(())


def train_graphed(model, optimizer, data_loader, loss, device):
    """The same epoch as ``train`` with the step replayed as a CUDA graph (:mod:`.graphs`): the host->device copy of batch
    i+1 overlaps step i, and every step's loss is read from pinned memory one step later instead of stalling the GPU with
    ``.item()``.  Same numbers as ``train`` (a batch of another size -- the last one -- takes the eager step)."""
    from . import graphs
    model.train()
    step = graphs.GraphedTrainStep([(model, optimizer)], loss)
    it = iter(data_loader)
    try:
        cur = next(it)
    except StopIteration:
        return float("nan")
    handle = step.prefetch(cur[0].long(), cur[1])
    total_loss, intervals, pending = 0.0, 0, None
    while handle is not None:
        nxt = next(it, None)
        nxt_handle = step.prefetch(nxt[0].long(), nxt[1]) if nxt is not None else None
        fetch = step.losses_to_host(step(handle))
        if pending is not None:
            total_loss += pending()[0]
        pending, handle = fetch, nxt_handle
        intervals += 1
    total_loss += pending()[0]
    return total_loss / intervals


def train(model, optimizer, data_loader, loss, device, fused=False, graphed=False):
    """pretrain_main.py:91-107: returns the mean of the per-batch losses."""
    if graphed:
        return train_graphed(model, optimizer, data_loader, loss, device)
    model.train()
    total_loss, intervals = 0.0, 0
    for features, labels in data_loader:
        features = features.long().to(device, non_blocking=True)
        labels = torch.unsqueeze(labels, 1).to(device, non_blocking=True)
        if fused and getattr(model, "mlp", None) is None:
            train_loss = fused_train_step(model, optimizer, features, labels)
        else:
            y = model(features)
            train_loss = loss(y, labels.float())
            model.zero_grad()
            train_loss.backward()
            optimizer.step()
        total_loss += train_loss.item()
        intervals += 1
    return total_loss / intervals


def _predict_all(model, data_loader, loss, device):
    """Predictions and labels of the whole loader, kept on the device (no per-batch .tolist())."""
    model.eval()
    targets, predicts, losses = [], [], []
    with torch.no_grad():
        for features, labels in data_loader:
            features = features.long().to(device, non_blocking=True)
            labels = torch.unsqueeze(labels, 1).to(device, non_blocking=True)
            y = model(features)
            if loss is not None:
                losses.append(loss(y, labels.float()))
            targets.append(labels)
            predicts.append(y)
    return torch.cat(targets), torch.cat(predicts), losses


def test(model, data_loader, loss, device):
    """pretrain_main.py:110-126: (AUC, mean per-batch loss).  The AUC is computed on the device (metrics.roc_auc_score:
    rlctr_auc_logloss, sklearn's tie handling) instead of .tolist() + sklearn.metrics.roc_auc_score."""
    from . import metrics
    targets, predicts, losses = _predict_all(model, data_loader, loss, device)
    mean_loss = torch.stack(losses).double().mean().item() if losses else float("nan")   # mean of the per-batch losses (:126)
    return metrics.roc_auc_score(targets, predicts), mean_loss


def submission(model, data_loader, device):
    """pretrain_main.py:128-139: (list of [pctr], AUC)."""
    from . import metrics
    targets, predicts, _ = _predict_all(model, data_loader, None, device)
    return predicts.cpu().numpy().tolist(), metrics.roc_auc_score(targets, predicts)


def eva_stopping(valid_aucs, valid_losses, type):
    """pretrain_main.py:239-251: stop after five strictly worsening epochs."""
    series, worse = (valid_aucs, lambda a, b: a < b) if type == "auc" else (valid_losses, lambda a, b: a > b)
    if len(series) < 5:
        return False
    return all(worse(series[-k], series[-k - 1]) for k in range(1, 5))


def main(data_path, dataset_name, campaign_id, valid_day, test_day, latent_dims, model_name, epoch, learning_rate,
         weight_decay, early_stop_type, batch_size, device, save_param_dir, optimizer_mode="lazy", fused=False, graphed=False):
    """pretrain_main.py:142-236.  Rolling window of 5 checkpoints, early stop, best -> ``<name>best.pth``,
    prediction CSVs -- with the reference's state_dict keys, so checkpoints are interchangeable."""
    os.makedirs(save_param_dir + campaign_id, exist_ok=True)
    device = torch.device(device)
    latent_dims = int(latent_dims)             # the reference's argparse leaves it a string (SURVEY section 5)
    _, _, train_data, valid_data, test_data, field_nums, feature_nums = get_dataset(
        data_path, dataset_name, campaign_id, valid_day, test_day)
    loaders = [BatchSlices(d, batch_size) for d in (train_data, valid_data, test_data)]
    model = get_model(model_name, feature_nums, field_nums, latent_dims).to(device)
    if model_name in ("IPNN", "OPNN", "FNN"):                              # :164-166: start from the FM checkpoint's embedding
        # the reference reads 'models/model_params/<campaign>FMbest.pth' relative to its working directory; here the
        # checkpoint directory this run writes to (the same place the FM run of `main` left FMbest.pth)
        fm_ckpt = save_param_dir + campaign_id + "FMbest.pth"
        if not os.path.exists(fm_ckpt):
            raise FileNotFoundError(f"{model_name} starts from the FM embedding (reference pretrain_main.py:164-166): "
                                    f"train FM first so that {fm_ckpt} exists")
        model.load_embedding(torch.load(fm_ckpt, map_location=device))
    loss = nn.BCELoss()
    valid_aucs, valid_losses, early_stop_index, is_early_stop = [], [], 0, False
    ckpt = lambda tag: save_param_dir + campaign_id + model_name + str(tag) + ".pth"
    start = datetime.datetime.now()
    for epoch_i in range(epoch):
        t0 = datetime.datetime.now()
        learning_rate += 1e-4                                               # :180
        optimizer = _optim.Adam(params=model.parameters(), lr=learning_rate, weight_decay=weight_decay,
                                mode=optimizer_mode)                       # :181, fresh state per epoch
        train_average_loss = train(model, optimizer, loaders[0], loss, device, fused=fused, graphed=graphed)
        torch.save(model.state_dict(), ckpt(epoch_i % 5))
        auc, valid_loss = test(model, loaders[1], loss, device)
        valid_aucs.append(auc)
        valid_losses.append(valid_loss)
        print("epoch:", epoch_i, "training average loss:", train_average_loss, "validation auc:", auc,
              "validation loss:", valid_loss, "[{}s]".format((datetime.datetime.now() - t0).seconds))
        if eva_stopping(valid_aucs, valid_losses, early_stop_type):
            early_stop_index, is_early_stop = (epoch_i - 4) % 5, True
            break
    if is_early_stop:
        test_model = get_model(model_name, feature_nums, field_nums, latent_dims).to(device)
        test_model.load_state_dict(torch.load(ckpt(early_stop_index), map_location=device))
    else:
        test_model = model
    auc, test_loss = test(test_model, loaders[2], loss, device)
    torch.save(test_model.state_dict(), ckpt("best"))
    print("\ntest auc:", auc, datetime.datetime.now(), "[{}s]".format((datetime.datetime.now() - start).seconds))
    submission_path = data_path + dataset_name + campaign_id + model_name + "/"
    os.makedirs(submission_path, exist_ok=True)
    day_aucs = []
    for day, loader in ((valid_day, loaders[1]), (test_day, loaders[2])):
        predicts, day_auc = submission(test_model, loader, device)
        np.savetxt(submission_path + str(day) + "_test_submission.csv",
                   np.column_stack([np.arange(len(predicts)), np.asarray(predicts).reshape(-1)]),
                   delimiter=",", fmt=["%d", "%.9g"])
        day_aucs.append([day, day_auc])
    np.savetxt(submission_path + "day_aucs.csv", np.column_stack([np.arange(2), np.asarray(day_aucs)]), delimiter=",",
               fmt=["%d", "%d", "%.17g"])
    for i in range(5):
        if os.path.exists(ckpt(i)):
            os.remove(ckpt(i))
    return auc, test_loss


if __name__ == "__main__":
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--data_path", default="../../data/")
    ap.add_argument("--dataset_name", default="ipinyou/", help="ipinyou, cretio, yoyi")
    ap.add_argument("--valid_day", default=11, type=int)
    ap.add_argument("--test_day", default=12, type=int)
    ap.add_argument("--campaign_id", default="1458/", help="1458, 3386")
    ap.add_argument("--model_name", default="FM", help="LR, FM, FFM, DeepFM")
    ap.add_argument("--latent_dims", default=8, type=int)
    ap.add_argument("--epoch", type=int, default=100)
    ap.add_argument("--learning_rate", type=float, default=1e-3)
    ap.add_argument("--weight_decay", type=float, default=1e-5)
    ap.add_argument("--early_stop_type", default="loss", help="auc, loss")
    ap.add_argument("--batch_size", type=int, default=4096)
    ap.add_argument("--device", default="cuda:0")
    ap.add_argument("--save_param_dir", default="../models/model_params/")
    ap.add_argument("--optimizer_mode", default="lazy", choices=["lazy", "dense", "sparse"])
    ap.add_argument("--fused", action="store_true")
    ap.add_argument("--graphed", action="store_true", help="replay the training step as a CUDA graph (graphs.GraphedTrainStep)")
    a = ap.parse_args()
    setup_seed(1)
    main(a.data_path, a.dataset_name, a.campaign_id, a.valid_day, a.test_day, a.latent_dims, a.model_name, a.epoch,
         a.learning_rate, a.weight_decay, a.early_stop_type, a.batch_size, a.device, a.save_param_dir,
         a.optimizer_mode, a.fused, a.graphed)
