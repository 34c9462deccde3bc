"""Host-side mirror of the reference's model classes for the PAMRec path.

``PAMRECModel(hparams, iterator_creator, graph=None, seed=None)`` keeps the public surface that
``example/00_quick_start/sequential.py`` drives (reference files: PAM = models/sequential/pamrec.py,
SBM = models/sequential/sequential_base_model.py, BM = models/base_model.py):

    fit_step, fit, run_weighted_eval, run_eval, predict, load_model,
    train(sess, feed), eval(sess, feed), eval_with_user(sess, feed), infer(sess, feed)

``sess`` arguments are accepted and ignored: the "session" is a ``pamrec_b200.engine.Engine`` that runs the
whole step as hand-written CUDA kernels behind the C ABI.  There is no CPU path.
"""
import math
import os
import random

import numpy as np
import torch

from . import checkpoint as CK
from . import dist as D
from . import summary as SUM
from .deeprec_utils import attention_topk, cal_metric, cal_weighted_metric, filter_single_class_users, full_ranking_metrics, load_dict
from .engine import Engine, PamrecError
from .prefetch import Prefetcher
from .sequential_iterator import LocalFeed

__all__ = ["PAMRECModel", "MMoEModel_original", "PLEModel", "ShareBottomModel", "SASRecModel", "SequentialBaseModel", "BaseModel", "latest_checkpoint",
           "initial_variables"]


# ----------------------------------------------------------------------------- initial values
def initial_variables(shapes, hparams, seed):
    """Initial value of every variable by TF name (SURVEY.md Appendix B).

    Same initializer families as the reference: ``hparams.init_method`` for variables created under a scope
    that carries ``self.initializer`` (BM:165-193), TF's default glorot_uniform for the time-aware tables and
    conv1d kernels, zeros for biases / LN beta / BN beta, ones for LN gamma / BN gamma / moving variance.
    TF's Philox streams are not reproducible, so the draws come from a seeded torch generator.
    """
    g = torch.Generator().manual_seed(0 if seed is None else int(seed))
    sigma = float(hparams.init_value)
    method = hparams.init_method
    out = {}
    for name, shape in shapes.items():
        leaf = name.rsplit("/", 1)[-1]
        shape = tuple(int(s) for s in shape)
        if leaf in ("moving_mean", "beta", "bias") or leaf.startswith("b_nn_") or name.endswith("ln/Variable") \
                or name.endswith("ln_1/Variable"):
            t = torch.zeros(shape)
        elif leaf in ("moving_variance", "gamma", "Variable_1"):
            t = torch.ones(shape)
        elif leaf.endswith("timeaware_embedding") or leaf == "kernel":
            fan_in, fan_out = (shape[0] * shape[1], shape[0] * shape[2]) if len(shape) == 3 else shape
            lim = math.sqrt(6.0 / (fan_in + fan_out))
            t = (torch.rand(shape, generator=g) * 2 - 1) * lim
        elif method == "uniform":
            t = (torch.rand(shape, generator=g) * 2 - 1) * sigma
        elif method == "normal":
            t = torch.randn(shape, generator=g) * sigma
        elif method in ("tnormal",) or method not in ("xavier_normal", "xavier_uniform", "he_normal", "he_uniform"):
            t = torch.empty(shape)
            torch.nn.init.trunc_normal_(t, mean=0.0, std=sigma, a=-2 * sigma, b=2 * sigma, generator=g)
        else:
            fan_in, fan_out = (shape[0], shape[-1]) if len(shape) > 1 else (shape[0], shape[0])
            if method.startswith("xavier"):
                std = math.sqrt(2.0 / (fan_in + fan_out))
            else:
                std = math.sqrt(2.0 / fan_in)
            if method.endswith("uniform"):
                t = (torch.rand(shape, generator=g) * 2 - 1) * (std * math.sqrt(3.0))
            else:
                t = torch.randn(shape, generator=g) * std
        out[name] = t.numpy().astype(np.float32)
    return out


# ----------------------------------------------------------------------------- candidate ranking
def candidate_ids(table, candidates, n_items, source="the file"):
    """Candidate item ids for ranking: every item with a category in ``table`` (item -> category, -1 = unknown; item 0 never)
    when ``candidates`` is None, else ``candidates`` checked: non-empty integer ids in [1, n_items), no duplicates, each with a
    known category.  Raises ValueError otherwise."""
    table = np.asarray(table)
    if candidates is None:
        ids = np.flatnonzero(table >= 0)
        ids = ids[ids >= 1]
        if ids.size == 0:
            raise ValueError("no candidates: {} names no item with a category".format(source))
        return ids
    ids = np.asarray(candidates).reshape(-1)
    if ids.size == 0 or not np.issubdtype(ids.dtype, np.integer):
        raise ValueError("candidates must be a non-empty list of integer vocabulary ids")
    ids = ids.astype(np.int64)
    bad = (ids < 1) | (ids >= n_items)
    if bad.any():
        raise ValueError("candidate ids must be in [1, {}): {}".format(n_items, ids[bad][:5].tolist()))
    if np.unique(ids).size != ids.size:
        raise ValueError("candidates hold duplicate ids")
    if (table[ids] < 0).any():
        raise ValueError("candidates without a category in {}: {}".format(source, ids[table[ids] < 0][:5].tolist()))
    return ids


def attention_line(user, pred, items, weights, item_key):
    """One line of explain(): user key, tab, the prediction, then per pooling slot a tab and the comma-separated ``item_key:weight``
    entries of items [P, K] / weights [P, K] (entries with item -1 are left out).  Floats are written as str() of their float32."""
    cols = [",".join("{}:{}".format(item_key.get(int(i), str(int(i))), np.float32(w)) for i, w in zip(items[s], weights[s]) if i >= 0)
            for s in range(len(items))]
    return "\t".join([str(user), str(np.float32(pred))] + cols)


# ----------------------------------------------------------------------------- checkpoints
def latest_checkpoint(model_dir):
    """tf.train.latest_checkpoint: reads ``<dir>/checkpoint`` written by Saver.save."""
    idx = os.path.join(model_dir, "checkpoint")
    if not os.path.exists(idx):
        return None
    with open(idx) as f:
        for line in f:
            if line.startswith("model_checkpoint_path:"):
                name = line.split(":", 1)[1].strip().strip('"')
                return name if os.path.isabs(name) else os.path.join(model_dir, name)
    return None


class Saver:
    """Counterpart of ``tf.train.Saver(max_to_keep=epochs)`` (BM:62).  One checkpoint per ``save_path`` keyed by TF variable
    name: model variables + BN moving statistics — exactly the Saver's var-list in the reference, which is built before the
    optimizer exists, so Adam slots are NOT part of a checkpoint (SURVEY.md section 5).  File formats: pamrec_b200/checkpoint.py
    (``hparams.checkpoint_format``: "safetensors" by default, "tf" for a TensorFlow tensor-bundle, "npz" legacy;
    ``hparams.save_optimizer`` adds the Adam state under the ``optimizer/`` key-space so that training can resume exactly -
    an extension, off by default like in the reference).  ``restore`` reads any of the formats."""

    def __init__(self, model, max_to_keep=5):
        self.model = model
        self.max_to_keep = max(int(max_to_keep), 1)
        self.kept = []
        self.fmt = getattr(model.hparams, "checkpoint_format", "safetensors")
        self.with_optimizer = bool(getattr(model.hparams, "save_optimizer", False))
        if self.fmt not in CK.FORMATS:
            raise ValueError("checkpoint_format must be one of {}".format(CK.FORMATS))

    def save(self, sess=None, save_path=None):
        d = os.path.dirname(save_path)
        if d:
            os.makedirs(d, exist_ok=True)
        eng = self.model.engine
        variables = eng.get_variables()                          # collective when the tables are sharded over ranks
        optimizer = eng.get_optimizer_state() if self.with_optimizer else None
        if save_path in self.kept:
            self.kept.remove(save_path)
        self.kept.append(save_path)
        dropped = []
        while len(self.kept) > self.max_to_keep:                 # every rank trims its list; rank 0 deletes the files
            dropped.append(self.kept.pop(0))
        if eng.rank != 0:
            torch.distributed.barrier()                          # rank 0 finishes writing before anyone may restore
            return save_path
        CK.save(save_path, variables, fmt=self.fmt, optimizer=optimizer)   # tmp + os.replace: the old files stay valid until now
        CK.remove(save_path, keep_fmt=self.fmt)                  # then a copy of this path written earlier in another format
        for p in dropped:
            CK.remove(p)
        with open(os.path.join(d, "checkpoint"), "w") as f:      # the CheckpointState text proto tf.train.latest_checkpoint reads
            f.write('model_checkpoint_path: "{}"\n'.format(os.path.basename(save_path)))
            for p in self.kept:
                f.write('all_model_checkpoint_paths: "{}"\n'.format(os.path.basename(p)))
        if eng.world > 1:
            torch.distributed.barrier()
        return save_path

    def restore(self, sess, path):
        variables, optimizer = CK.load(path)
        known = self.model.engine.variable_shapes()
        # a checkpoint written by the reference's Saver holds every global variable of ITS graph; names this graph does not
        # have (none for PAMRec as shipped) are reported, not silently dropped
        extra = sorted(set(variables) - set(known))
        if extra:
            raise KeyError("checkpoint {} holds variables this model does not have: {}".format(path, extra[:5]))
        for name, val in variables.items():
            if tuple(val.shape) != tuple(known[name]):
                raise ValueError("checkpoint {}: {} has shape {}, the model expects {}".format(path, name, val.shape, known[name]))
        self.model.engine.set_variables(variables)
        if optimizer is not None:
            self.model.engine.set_optimizer_state(optimizer)


class _Session:
    """Placeholder for ``tf.Session``: kept so that ``model.sess`` exists."""
    graph = None


# ----------------------------------------------------------------------------- models
class BaseModel:
    def __init__(self, hparams, iterator_creator, graph=None, seed=None):
        """BM:20-75: seed python/numpy RNGs, build iterator, variables and the device session."""
        self.seed = seed
        np.random.seed(seed)
        random.seed(seed)
        self.graph = graph
        self.iterator = iterator_creator(hparams, self.graph)
        self.train_num_ngs = hparams.train_num_ngs
        self.hparams = hparams
        self.keep_prob_train = 1 - np.array(hparams.dropout)
        self.keep_prob_test = np.ones_like(hparams.dropout)
        self._check_supported(hparams)
        self._build_graph()
        self.saver = Saver(self, max_to_keep=hparams.epochs)
        self.sess = _Session()

    def _check_supported(self, hp):
        """The kernels implement the graph that config/mmoe.yaml + the quick-start flags build; anything that would
        change the arithmetic is refused rather than silently approximated."""
        def need(cond, what):
            if not cond:
                raise ValueError("pamrec_b200: unsupported configuration: " + what)
        need(hp.method == "classification", "method must be classification (BM:93-113)")
        need(hp.loss in ("cross_entropy_loss", "softmax"), "loss must be cross_entropy_loss or softmax (BM:195-242; square_loss and "
                                                            "log_loss have no auxiliary branch that PAMRec defines consistently)")
        need(hp.optimizer == "adam", "optimizer must be adam (BM:270-271)")
        self._check_emb_dims(hp, need)
        need(list(hp.layer_sizes) == [100, 64], "tower sizes of config/mmoe.yaml")
        self._check_mixing(hp, need)
        need(list(hp.activation)[:2] == ["relu", "relu"], "activation must be [relu, relu]")
        need(bool(hp.enable_BN), "enable_BN must be True")
        need(all(float(d) == 0.0 for d in hp.dropout) and float(hp.embedding_dropout) == 0.0 and not hp.user_dropout,
             "dropout must be 0 (SURVEY.md Appendix A)")
        need(not getattr(hp, "add_feature", False), "add_feature must be False")
        need(not getattr(hp, "fine_tune", False), "fine_tune must be False")
        need(float(hp.embed_l1) == 0.0 and float(hp.layer_l1) == 0.0 and float(hp.cross_l1) == 0.0 and
             float(hp.cross_l2) == 0.0, "L1 / cross regularisation must be 0")
        need(1 <= hp.max_seq_length <= 256, "max_seq_length must be in [1, 256]")
        need(hp.batch_size % 5 == 0, "batch_size must be a multiple of 5 (IT:684-685, PAM:73-75)")
        need(isinstance(getattr(hp, "summary_step", 1), int) and getattr(hp, "summary_step", 1) >= 1,
             "summary_step must be an integer >= 1")

    def _check_mixing(self, hp, need):
        need(list(hp.expert_layer_sizes) == [100, 64] and list(hp.gate_layer_sizes) == [64, 5] and hp.expert_num == 5,
             "expert / gate sizes of config/mmoe.yaml")

    def _check_emb_dims(self, hp, need):
        need(hp.item_embedding_dim == 16 and hp.cate_embedding_dim == 4 and hp.user_embedding_dim == 20,
             "embedding dims must be 16 / 4 / 20 (config/mmoe.yaml:22-24)")

    @staticmethod
    def _emb_dims(hp):
        """(item, cate, user) embedding widths of the engine, as _check_supported admitted them."""
        return int(hp.item_embedding_dim), int(hp.cate_embedding_dim), int(hp.user_embedding_dim)

    def _build_graph(self):
        raise NotImplementedError

    # ---- BM:350-399
    def train(self, sess, feed_dict):
        raise NotImplementedError

    def load_model(self, model_path=None):
        """BM:401-417."""
        act_path = self.hparams.load_saved_model
        if model_path is not None:
            act_path = model_path
        try:
            self.saver.restore(self.sess, act_path)
        except Exception:
            raise IOError("Failed to find any matching files for {0}".format(act_path))


class SequentialBaseModel(BaseModel):
    def __init__(self, hparams, iterator_creator, graph=None, seed=None):
        """SBM:22-54."""
        self.hparams = hparams
        self.need_sample = hparams.need_sample
        self.train_num_ngs = hparams.train_num_ngs
        if self.train_num_ngs is None:
            raise ValueError("Please confirm the number of negative samples for each positive instance.")
        self.min_seq_length = hparams.min_seq_length
        self.hidden_size = hparams.hidden_size
        self.embedding_keep_prob_train = 1.0 - hparams.embedding_dropout
        self.embedding_keep_prob_test = 1.0
        super().__init__(hparams, iterator_creator, graph=graph, seed=seed)

    # ------------------------------------------------------------------ device steps
    def _score_async(self, feed_dict):
        """Queue the scoring of one batch: staged H2D copy, forward pass (BN inference mode), D2H copy of the predictions into a
        pinned ring slot.  Returns a handle whose ``result()`` waits for that copy and gives pred [B,1]: the eval loops queue
        batch i + 1 before they read batch i, the way train_async pipelines sess.run (SBM:437-447 blocks per batch)."""
        eng = self.engine
        n = None
        if isinstance(feed_dict, LocalFeed):
            # the iterator already dealt this rank its rows (r, r + W, ...) of a batch of global_rows rows
            n = feed_dict.global_rows
            db = eng.upload(feed_dict, training=False, staged=True, global_batch=n)
        elif eng.world > 1 and self.feed_is_global:
            # data-parallel scoring: rank r scores rows r, r + W, ... of the batch; the scores are summed back into place
            local, n = D.split_feed(feed_dict, eng.world, eng.rank, grouped=False)
            db = eng.upload(local, training=False, staged=True, global_batch=n)
        else:
            db = eng.upload(feed_dict, training=False, staged=True)
        pred = eng.forward(db, training=False)
        if n is not None:
            full = torch.zeros(n, dtype=torch.float32, device=eng.device)
            full[eng.rank::eng.world] = pred
            pred = eng.all_reduce_(full)
        return eng.to_host_async(pred)

    def _score(self, feed_dict):
        return self._score_async(feed_dict).result().reshape(-1, 1)

    def _scored(self, filename, **kw):
        """(feed, pred [B,1]) over a file with the device one batch ahead of the host."""
        pending = None
        for feed in Prefetcher(self.iterator.load_data_from_file(filename, batch_num_ngs=0, **kw)):
            if not feed:
                continue
            queued = (feed, self._score_async(feed))
            if pending is not None:
                yield pending[0], pending[1].result().reshape(-1, 1)
            pending = queued
        if pending is not None:
            yield pending[0], pending[1].result().reshape(-1, 1)

    @staticmethod
    def _labels_users(feed_dict):
        if isinstance(feed_dict, LocalFeed):                     # every row of the global batch, not just this rank's
            return feed_dict.global_labels_satisfied, feed_dict.global_users
        return feed_dict["labels_satisfied"], feed_dict["users"]

    def eval(self, sess, feed_dict):
        """SBM:415-418 / BM:373-386 -> (pred [B,1], labels [B,1])."""
        return self._score(feed_dict), np.asarray(self._labels_users(feed_dict)[0], np.float32).reshape(-1, 1)

    def eval_with_user(self, sess, feed_dict):
        """SBM:502-516 -> (users [B], pred [B,1], labels [B,1])."""
        labels, users = self._labels_users(feed_dict)
        return np.asarray(users).astype(np.int32), self._score(feed_dict), np.asarray(labels, np.float32).reshape(-1, 1)

    def infer(self, sess, feed_dict):
        """SBM:557-560 / BM:388-399 -> [pred]."""
        return [self._score(feed_dict)]

    # ------------------------------------------------------------------ summaries (SBM:268-274)
    _writer = None

    def _pending_step(self, losses):
        """Wrap a queued step's PendingLosses.  With ``write_tfevents`` every ``summary_step``-th optimiser step (an extension:
        the reference summarises every step, summary_step = 1, the default) also queues the histograms of every checkpoint
        variable on the device behind it; the handle's result() then carries the serialized Summary and hands it to the open
        event file."""
        eng = self.engine
        hist = None
        if self.hparams.write_tfevents and eng.step % getattr(self.hparams, "summary_step", 1) == 0:
            hist = eng.histograms(eng.variable_shapes())
        return _PendingStep(losses, self.SCALARS, hist, eng.step, self)

    def _open_summaries(self):
        """fit / fit_step: a new event file in SUMMARIES_DIR when write_tfevents is set (rank 0 writes; every rank bins)."""
        if self.hparams.write_tfevents and self.hparams.SUMMARIES_DIR and self.engine.rank == 0:
            self._writer = SUM.EventFileWriter(self.hparams.SUMMARIES_DIR)

    def _flush_summaries(self):
        if self._writer is not None:
            self._writer.flush()

    def _close_summaries(self):
        if self._writer is not None:
            w, self._writer = self._writer, None
            w.close()

    # ------------------------------------------------------------------ loops
    def _maybe_save(self, progress, tag):
        if self.hparams.save_model and self.hparams.MODEL_DIR:
            if not os.path.exists(self.hparams.MODEL_DIR):
                os.makedirs(self.hparams.MODEL_DIR)
            if progress:
                self.saver.save(sess=self.sess, save_path=self.hparams.MODEL_DIR + tag)

    def fit(self, train_file, valid_file, valid_num_ngs, eval_metric="group_auc"):
        """SBM:133-224: epoch loop, evaluation after every epoch, early stop on epochs."""
        if not self.need_sample and self.train_num_ngs < 1:
            raise ValueError("Please specify a positive integer of negative numbers for training without sampling needed.")
        if valid_num_ngs < 1:
            raise ValueError("Please specify a positive integer of negative numbers for validation.")
        if self.need_sample and self.train_num_ngs < 1:
            self.train_num_ngs = 1
        self._open_summaries()
        try:
            self._fit_epochs(train_file, valid_file, valid_num_ngs, eval_metric)
        finally:
            self._close_summaries()
        return self

    def _fit_epochs(self, train_file, valid_file, valid_num_ngs, eval_metric):
        eval_info = []
        best_metric, self.best_epoch = 0, 0
        for epoch in range(1, self.hparams.epochs + 1):
            self.hparams.current_epoch = epoch
            file_iterator = Prefetcher(self.iterator.load_data_from_file(train_file, min_seq_length=self.min_seq_length,
                                                                         batch_num_ngs=self.train_num_ngs))
            self.batch_train(file_iterator, self.sess)
            self._flush_summaries()
            valid_res = self.run_weighted_eval(valid_file, valid_num_ngs)
            print("eval valid at epoch {0}: {1}".format(epoch, ",".join(str(k) + ":" + str(v) for k, v in valid_res.items())))
            eval_info.append((epoch, valid_res))
            progress = False
            early_stop = self.hparams.EARLY_STOP
            if valid_res[eval_metric] > best_metric:
                best_metric = valid_res[eval_metric]
                self.best_epoch = epoch
                progress = True
            elif early_stop > 0 and epoch - self.best_epoch >= early_stop:
                print("early stop at epoch {0}!".format(epoch))
                break
            self._maybe_save(progress, "epoch_" + str(epoch))
        print(eval_info)
        print("best step: {0}".format(self.best_epoch))

    def fit_step(self, train_file, valid_file, valid_num_ngs, eval_metric="group_auc"):
        """SBM:239-377: step loop, evaluation every ``eval_step`` steps, early stop on steps, checkpoint on improvement."""
        if self.need_sample and self.train_num_ngs < 1:
            self.train_num_ngs = 1
        self._open_summaries()
        try:
            self._fit_steps(train_file, valid_file, valid_num_ngs, eval_metric)
        finally:
            self._close_summaries()
        return self

    def _fit_steps(self, train_file, valid_file, valid_num_ngs, eval_metric):
        eval_info = []
        best_metric, self.best_step = 0, 0
        step = 0
        break_flag = False
        for epoch in range(1, self.hparams.epochs + 1):
            print("epoch:{}".format(epoch))
            if break_flag:
                break
            self.hparams.current_epoch = epoch
            file_iterator = Prefetcher(self.iterator.load_data_from_file(train_file, min_seq_length=self.min_seq_length,
                                                                         batch_num_ngs=self.train_num_ngs))
            pending = None                                   # the step in flight: its losses are read after the next is queued
            for batch_data_input in file_iterator:
                if not batch_data_input:
                    continue
                queued = self.train_async(self.sess, batch_data_input)
                if pending is not None:
                    self.step_train(step - 1, pending.result())
                pending = queued
                step += 1
                if step % self.hparams.eval_step == 0:
                    self.step_train(step - 1, pending.result())
                    pending = None
                    self._flush_summaries()
                    valid_res = self.run_weighted_eval(valid_file, valid_num_ngs)
                    print("eval valid at epoch {0} step {1}: {2}".format(
                        epoch, step, ",".join(str(k) + ":" + str(v) for k, v in valid_res.items())))
                    eval_info.append((step, valid_res))
                    progress = False
                    early_stop = self.hparams.EARLY_STOP
                    if valid_res[eval_metric] > best_metric:
                        best_metric = valid_res[eval_metric]
                        self.best_step = step
                        progress = True
                    elif early_stop > 0 and step - self.best_step >= early_stop * self.hparams.eval_step:
                        print("early stop at epoch {0}, step {1}!".format(epoch, step))
                        break_flag = True
                        file_iterator.close()
                        break
                    self._maybe_save(progress, "step_" + str(step))
            if pending is not None:
                self.step_train(step - 1, pending.result())
        print(eval_info)
        print("best step: {0}".format(self.best_step))

    def run_eval(self, filename, num_ngs):
        """SBM:380-413."""
        preds, labels, group_preds, group_labels = [], [], [], []
        group = num_ngs + 1
        for feed, step_pred in self._scored(filename, min_seq_length=self.min_seq_length):
            step_labels = np.asarray(self._labels_users(feed)[0], np.float32).reshape(-1, 1)
            preds.extend(np.reshape(step_pred, -1))
            labels.extend(np.reshape(step_labels, -1))
            group_preds.extend(np.reshape(step_pred, (-1, group)))
            group_labels.extend(np.reshape(step_labels, (-1, group)))
        res = cal_metric(labels, preds, self.hparams.metrics)
        res.update(cal_metric(group_labels, group_preds, self.hparams.pairwise_metrics))
        return res

    def run_weighted_eval(self, filename, num_ngs, calc_mean_alpha=False, manual_alpha=False):
        """SBM:420-500: score every impression, drop groups without a positive (pairwise metrics) and users whose labels
        are all 0 or all 1 (point + user-weighted metrics)."""
        if calc_mean_alpha:
            raise NotImplementedError("alpha outputs belong to the CLSR models, not to PAMRec (SBM:518-532)")
        users, preds, labels, group_preds, group_labels = [], [], [], [], []
        group = num_ngs + 1
        for feed, step_pred in self._scored(filename, min_seq_length=self.min_seq_length):
            step_labels, step_user = self._labels_users(feed)
            step_labels = np.asarray(step_labels, np.float32).reshape(-1, 1)
            users.append(np.reshape(np.asarray(step_user).astype(np.int32), -1))    # the reference extends Python lists row by row
            preds.append(np.reshape(step_pred, -1))                                   # (SBM:449-455); arrays per batch, joined once
            labels.append(np.reshape(step_labels, -1))
            gp = np.reshape(step_pred, (-1, group))
            gl = np.reshape(step_labels, (-1, group))
            keep = gl.sum(axis=1) != 0                           # SBM:456-460: groups without a positive are dropped
            group_preds.append(gp[keep])
            group_labels.append(gl[keep])
        cat = lambda parts, dt: np.concatenate(parts) if parts else np.zeros(0, dt)
        users, preds, labels = cat(users, np.int32), cat(preds, np.float32), cat(labels, np.float32)
        group_preds = np.concatenate(group_preds) if group_preds else []
        group_labels = np.concatenate(group_labels) if group_labels else []
        users, preds, labels = filter_single_class_users(users, preds, labels, as_arrays=True)
        res = cal_metric(labels, preds, self.hparams.metrics)
        res.update(cal_metric(group_labels, group_preds, self.hparams.pairwise_metrics))
        res.update(cal_weighted_metric(users, preds, labels, self.hparams.weighted_metrics))
        return res

    def predict(self, infile_name, outfile_name):
        """SBM:534-555: one score per line (data parallel: every rank scores, rank 0 writes)."""
        writer = self.engine.rank == 0
        wt = open(outfile_name, "w") if writer else None
        try:
            for _, step_pred in self._scored(infile_name):
                step_pred = np.reshape(step_pred, -1)
                if writer:
                    wt.write("\n".join(map(str, step_pred)))
                    wt.write("\n")
        finally:
            if wt:
                wt.close()
        return self

    # ------------------------------------------------------------------ candidate ranking (no reference counterpart)
    def _ranked(self, filename, top_k, exclude_history, candidates, want_rank, **kw):
        """(feed, topk_items [B,K], topk_scores [B,K], own_rank [B] or None) per scoring batch of ``filename``, every line ranked
        against the candidates on the device (Engine.rank_candidates)."""
        eng = self.engine
        if eng.world > 1 or (torch.distributed.is_available() and torch.distributed.is_initialized()
                             and torch.distributed.get_world_size() > 1):
            raise ValueError("candidate ranking runs on one GPU, not under torch.distributed with several ranks")
        if not 1 <= int(top_k) <= 1024:
            raise ValueError("top_k must be between 1 and 1024, not {}".format(top_k))
        table = self.iterator.item_categories([filename])
        ids = candidate_ids(table, candidates, eng.dims[1], filename)
        items = torch.as_tensor(ids.astype(np.int32)).to(eng.device)
        cates = torch.as_tensor(table[ids].astype(np.int32)).to(eng.device)

        def batches():
            for feed in self.iterator.load_data_from_file(filename, batch_num_ngs=0, **kw):
                if feed:
                    db = eng.upload(feed, training=False, staged=True)
                    yield (feed,) + eng.rank_candidates(db, items, cates, top_k, exclude_history, want_rank).result()
        return batches()

    def recommend(self, infile_name, outfile_name, top_k=10, exclude_history=True, candidates=None):
        """The ``top_k`` items this model ranks first for every line of ``infile_name`` (an evaluation file), scored on the device
        against the candidates: ``candidates=None`` is every item with a known category in the file, else a list of vocabulary
        ids.  exclude_history skips the items of the line's history (not its own item).  Writes one line per input line:
        user key, tab, comma-separated item keys, tab, comma-separated float32 scores (best first; fewer when fewer candidates
        remain).  Returns dict(users [N] user ids, items [N, K] item ids (-1 past the last), scores [N, K] float32)."""
        user_key = {v: k for k, v in reversed(list(self.iterator.userdict.items()))}
        item_key = {v: k for k, v in reversed(list(self.iterator.itemdict.items()))}
        users, items, scores = [], [], []
        ranked = self._ranked(infile_name, top_k, exclude_history, candidates, False)
        with open(outfile_name, "w") as wt:
            for feed, top_items, top_scores, _ in ranked:
                u = np.asarray(feed["users"]).reshape(-1).astype(np.int64)
                for r in range(top_items.shape[0]):
                    n = int((top_items[r] >= 0).sum())
                    wt.write("{}\t{}\t{}\n".format(user_key.get(int(u[r]), str(int(u[r]))),
                                                   ",".join(item_key.get(int(i), str(int(i))) for i in top_items[r, :n]),
                                                   ",".join(str(x) for x in top_scores[r, :n])))
                users.append(u)
                items.append(top_items)
                scores.append(top_scores)
        cat = lambda parts, shape, dt: np.concatenate(parts) if parts else np.zeros(shape, dt)
        return dict(users=cat(users, (0,), np.int64), items=cat(items, (0, top_k), np.int32), scores=cat(scores, (0, top_k), np.float32))

    def run_full_ranking_eval(self, filename, ks=(10,), exclude_history=False, candidates=None):
        """Full-ranking evaluation: every line with label 1 of ``filename`` ranks its own item against all candidates
        (``candidates`` as in recommend) on the device; hit@k, ndcg@k and mrr averaged over those lines (deeprec_utils
        full_ranking_metrics; a positive that is not a candidate counts as a miss)."""
        ks = tuple(int(k) for k in ks)
        ranks, labels = [], []
        for feed, _, _, rank in self._ranked(filename, 1, exclude_history, candidates, True, min_seq_length=self.min_seq_length):
            ranks.append(rank)
            labels.append(np.asarray(self._labels_users(feed)[0]).reshape(-1))
        cat = lambda parts: np.concatenate(parts) if parts else np.zeros(0)
        return full_ranking_metrics(cat(ranks), cat(labels), ks)

    # ------------------------------------------------------------------ attention weights (no reference counterpart)
    # per pooling slot: the history columns its weights index (PAMRec: the full history; the DIN siblings: satisfied-only, then
    # full; SASRec: its satisfied-only input)
    ATTENTION_SLOTS = (("item_history", "mask"),)

    def explain(self, infile_name, outfile_name, top_k=5, maps=False):
        """The attention weights behind every score of ``infile_name`` (a scoring file, read as predict reads it), computed on the
        device by the forward pass that scores the line (Engine.attention).  Writes one line per input line: user key, tab, the
        prediction, then per pooling slot a tab and up to ``top_k`` comma-separated ``item_key:weight`` entries over the line's real
        history positions (mask > 0), by weight descending, then position ascending.  maps=True (PAMRec, SASRec) also returns the
        encoder's attention maps.  Returns dict(users [N], pred [N] float32, pool [N, P, T] float32, positions [N, P, top_k] (indices
        into the slot's history, -1 past the last), items [N, P, top_k] (-1 there), weights [N, P, top_k] float32 (0 there),
        maps [N, 2, T, T] float32 or None).  maps=True holds the maps of every line of the file in host memory: N x 2 x T x T x 4
        bytes (32 GB for 100 000 lines at T = 200, twice that while the batches are joined at the end); for a large file call
        Engine.attention per batch instead."""
        eng = self.engine
        T = eng.dims[3]
        if eng.world > 1 or (torch.distributed.is_available() and torch.distributed.is_initialized()
                             and torch.distributed.get_world_size() > 1):
            raise ValueError("explain runs on one GPU, not under torch.distributed with several ranks")
        if not isinstance(top_k, (int, np.integer)) or not 1 <= int(top_k) <= T:
            raise ValueError("top_k must be between 1 and max_seq_length ({}), not {}".format(T, top_k))
        if maps and eng.model not in ("pamrec", "sasrec"):
            raise ValueError("attention maps need a self-attention encoder (PAMRec, SASRec), not {}".format(eng.model))
        top_k = int(top_k)
        user_key = {v: k for k, v in reversed(list(self.iterator.userdict.items()))}
        item_key = {v: k for k, v in reversed(list(self.iterator.itemdict.items()))}
        parts = {k: [] for k in ("users", "pred", "pool", "positions", "items", "weights", "maps")}
        with open(outfile_name, "w") as wt:
            for feed in self.iterator.load_data_from_file(infile_name, batch_num_ngs=0):
                if not feed:
                    continue
                got = eng.attention(eng.upload(feed, training=False, staged=True), maps=maps).result()
                B = got["pred"].shape[0]
                u = np.asarray(feed["users"]).reshape(-1).astype(np.int64)
                pos, wts, its = [], [], []
                for slot, (hist, mask) in enumerate(self.ATTENTION_SLOTS):
                    h = np.asarray(feed[hist]).reshape(B, T)
                    p, w = attention_topk(got["pool"][:, slot], np.asarray(feed[mask]).reshape(B, T) > 0, top_k)
                    pos.append(p)
                    wts.append(w)
                    its.append(np.where(p >= 0, np.take_along_axis(h, np.maximum(p, 0), -1), -1))
                pos, wts, its = np.stack(pos, 1), np.stack(wts, 1), np.stack(its, 1)
                for r in range(B):
                    wt.write(attention_line(user_key.get(int(u[r]), str(int(u[r]))), got["pred"][r], its[r], wts[r], item_key) + "\n")
                for k, v in (("users", u), ("pred", got["pred"]), ("pool", got["pool"]), ("positions", pos), ("items", its),
                             ("weights", wts), ("maps", got["maps"])):
                    parts[k].append(v)
        P = len(self.ATTENTION_SLOTS)
        empty = dict(users=((0,), np.int64), pred=((0,), np.float32), pool=((0, P, T), np.float32), positions=((0, P, top_k), np.int64),
                     items=((0, P, top_k), np.int64), weights=((0, P, top_k), np.float32), maps=((0, 2, T, T), np.float32))
        out = {k: np.concatenate(v) if v else np.zeros(*empty[k]) for k, v in parts.items() if k != "maps"}
        out["maps"] = (np.concatenate(parts["maps"]) if parts["maps"] else np.zeros(*empty["maps"])) if maps else None
        return out


class _PendingStep:
    """A queued train step: ``result()`` gives train()'s tuple (update, extra_update_ops, <one float per loss name>, summary).
    summary is None unless histograms were queued behind the step; then it is the serialized Summary of the loss scalars and
    the histograms, also handed to the model's open event file at the optimiser step ``step``."""

    def __init__(self, pending, scalars, hist=None, step=0, model=None):
        self._pending, self._scalars, self._hist, self._step, self._model = pending, scalars, hist, step, model
        self._value = None

    def result(self):
        if self._value is None:
            l = self._pending.result()
            values = [float(v) for v in l[:len(self._scalars)]]
            summary = None
            if self._hist is not None:
                hist = self._hist.result()
                for name, h in hist.items():
                    if h["nonfinite"]:
                        raise PamrecError("Nan in summary histogram for: {} (step {})".format(name, self._step))
                summary = SUM.summary_proto(zip(self._scalars, values), hist.items())
                if self._model._writer is not None:
                    self._model._writer.add_summary(summary, self._step)
            self._value = [None, None] + values + [summary]
        return self._value


class PAMRECModel(SequentialBaseModel):
    """PAM:25: the playback-duration-augmented model.  The graph (embeddings, time-aware 2-block encoder, attention
    pooling, MMoE, three towers, four-term loss, per-tensor clip + Adam) is libpamrec_b200.so."""
    ENGINE_MODEL = "pamrec"
    SCALARS = ("loss", "data_loss", "regular_loss", "auxiliary_data_loss", "order_loss")     # train()'s tuple, PAM:444-448

    def _build_graph(self):
        hp = self.hparams
        n_users = len(load_dict(hp.user_vocab))        # SBM:565-567
        n_items = len(load_dict(hp.item_vocab))
        n_cates = len(load_dict(hp.cate_vocab))
        engine_hp = dict(
            learning_rate=float(hp.learning_rate), embed_l2=float(hp.embed_l2), layer_l2=float(hp.layer_l2),
            max_grad_norm=float(hp.max_grad_norm), is_clip_norm=int(bool(hp.is_clip_norm)),
            fuzhu_weight=float(getattr(hp, "fuzhu_weight", 0.5)), discrepancy_loss_weight=float(hp.discrepancy_loss_weight),
            loss=hp.loss, softmax_group=int(hp.train_num_ngs or 0) + 1)
        mode = getattr(hp, "sparse_adam", "dense_exact")
        # data parallel (no reference counterpart): one process per GPU under torchrun.  hparams.batch_size stays the GLOBAL
        # batch when feeds come from the iterator (every rank reads the same file and trains on its groups of each batch);
        # dp_feed="local" means the caller hands each rank its own share (bench.py's weak-scaling arrays).
        world, rank = 1, 0
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            world, rank = torch.distributed.get_world_size(), torch.distributed.get_rank()
        self.feed_is_global = getattr(hp, "dp_feed", "global") != "local"
        ngs = max(int(hp.train_num_ngs or 0), 0)                             # in-batch negatives multiply the rows of a batch;
        if ngs < 1 and hp.need_sample:                                       # fit / fit_step force one negative when sampling
            ngs = 1                                                          # is "needed" (SBM:153-154, SBM:257-258)
        cap = hp.batch_size * (1 + ngs)
        if world > 1 and self.feed_is_global:
            cap = max(-(-(cap // 5) // world) * 5, -(-cap // world))
        tables = getattr(hp, "tables", None)
        self.engine = Engine(n_users, n_items, n_cates, hp.max_seq_length, cap, hp=engine_hp, sparse_adam=mode,
                             world_size=world, rank=rank, tables=tables, model=self.ENGINE_MODEL, emb_dims=self._emb_dims(hp))
        default_dev = "cuda:{}".format(int(os.environ.get("LOCAL_RANK", 0))) if world > 1 else "cuda:0"
        self.engine.allocate(getattr(hp, "device", default_dev))
        self.engine.init_comm()
        self.engine.set_variables(initial_variables(self.engine.variable_shapes(), hp, self.seed))
        if world > 1 and self.feed_is_global and hasattr(self.iterator, "shard"):
            self.iterator.shard = (world, rank)      # the native batcher materialises this rank's rows only (LocalFeed)

    def train(self, sess, feed_dict):
        """PAM:426-453: one optimisation step.  Returns the reference's 8-tuple
        (update, extra_update_ops, loss, data_loss, regular_loss, auxiliary_data_loss, order_loss, summary)."""
        return self.train_async(sess, feed_dict).result()

    def train_async(self, sess, feed_dict):
        """train() split in two: the feed is staged, copied to the device and the step queued; ``.result()`` of the returned
        handle waits for the losses and gives train()'s 8-tuple.  Queuing step i + 1 before reading step i keeps the device busy
        while the host packs the next feed (fit_step / batch_train below and bench.py's e2e loop run one step ahead)."""
        eng = self.engine
        if isinstance(feed_dict, LocalFeed):
            db = eng.upload(feed_dict, training=True, staged=True, global_batch=feed_dict.global_rows)
        elif eng.world > 1 and self.feed_is_global:
            local, n = D.split_feed(feed_dict, eng.world, eng.rank, grouped=True)
            db = eng.upload(local, training=True, staged=True, global_batch=n)
        else:
            db = eng.upload(feed_dict, training=True, staged=True)
        return self._pending_step(eng.train_step_async(db))

    def step_train(self, step, step_result):
        """PAM:455-465."""
        (_, _, step_loss, step_data_loss, _, step_aux, order_loss, _) = step_result
        if step % self.hparams.show_step == 0:
            print("step {0:d} , total_loss: {1:.4f}, data_loss: {2:.4f}, auxiliary_data_loss: {3:.4f}, order_loss: {4:.4f}".format(
                step, step_loss, step_data_loss, step_aux, order_loss))

    def batch_train(self, file_iterator, train_sess):
        """PAM:467-503 (the reference unpacks a 7-tuple from an 8-tuple there and would raise; this version works)."""
        step, epoch_loss = 0, 0.0

        def account(step, r):
            if step % self.hparams.show_step == 0:
                print("step {0:d} , total_loss: {1:.4f}, data_loss: {2:.4f}, auxiliary_data_loss: {3:.4f}".format(
                    step, r[2], r[3], r[5]))
            return r[2]
        pending = None
        for feed in file_iterator:
            if feed:
                queued = self.train_async(train_sess, feed)
                if pending is not None:
                    epoch_loss += account(step, pending.result())
                pending = queued
                step += 1
        if pending is not None:
            epoch_loss += account(step, pending.result())
        return epoch_loss


# ----------------------------------------------------------------------------- sibling multi-task baselines (SURVEY.md section 8(f) N3)
class _DinMultiTask(PAMRECModel):
    """What MMoEModel_original, PLEModel and ShareBottomModel share (models/sequential/mmoe.py, ple.py, sharebottom.py): the
    input pipeline, DIN attention pooling of the satisfied-only and of the full history against the target (`_attention_fcn`),
    two towers, loss = data + regular + 0.5 * auxiliary, and the host loops - which differ from PAMRec's only in the 7-tuple
    that train() returns (no order loss, MM:341-373).  One GPU.  Embedding widths (item / cate / user): 16 / 4 (config/mmoe.yaml)
    or 32 / 8 (the reference's ple.yaml and sharebottom.yaml, and 32 / 8 / 16 in its sasrec.yaml), each with a user width of 16,
    20 or 40; the kernels are compiled for both item / cate pairs."""

    SCALARS = ("loss", "data_loss", "regular_loss", "auxiliary_data_loss")                  # MM:341-373
    ATTENTION_SLOTS = (("satisfied_item_history", "satisfied_mask"), ("item_history", "mask"))

    def _check_supported(self, hp):
        super()._check_supported(hp)
        if list(getattr(hp, "att_fcn_layer_sizes", [80, 40])) != [80, 40]:
            raise ValueError("pamrec_b200: unsupported configuration: att_fcn_layer_sizes must be [80, 40]")
        if hp.loss != "cross_entropy_loss":
            raise ValueError("pamrec_b200: unsupported configuration: the sibling models train with cross_entropy_loss")

    def _check_emb_dims(self, hp, need):
        need((hp.item_embedding_dim, hp.cate_embedding_dim) in ((16, 4), (32, 8)) and hp.user_embedding_dim in (16, 20, 40),
             "embedding dims (item / cate / user) must be 16 / 4 or 32 / 8, with user 16, 20 or 40 "
             "(config/mmoe.yaml: 16 / 4 / 20; the reference's ple.yaml / sharebottom.yaml: 32 / 8 / 40, sasrec.yaml: 32 / 8 / 16)")
        if torch.distributed.is_available() and torch.distributed.is_initialized() and torch.distributed.get_world_size() > 1:
            raise ValueError("pamrec_b200: the sibling models run on one GPU")

    def train_async(self, sess, feed_dict):
        return self._pending_step(self.engine.train_step_async(self.engine.upload(feed_dict, training=True, staged=True)))

    def step_train(self, step, step_result):
        """MM:375-385."""
        (_, _, step_loss, step_data_loss, _, step_aux, _) = step_result
        if step % self.hparams.show_step == 0:
            print("step {0:d} , total_loss: {1:.4f}, data_loss: {2:.4f}, auxiliary_data_loss: {3:.4f}".format(
                step, step_loss, step_data_loss, step_aux))


class MMoEModel_original(_DinMultiTask):
    """MM:24: five experts, two BN + ReLU gates over all of them (MM:26-50)."""
    ENGINE_MODEL = "mmoe"


class PLEModel(_DinMultiTask):
    """PLE:24: three shared experts, two per task; each task's gate mixes the shared ones and its own (PLE:25-59)."""
    ENGINE_MODEL = "ple"

    def _check_mixing(self, hp, need):
        need(list(hp.expert_layer_sizes) == [100, 64] and list(hp.gate_layer_sizes) == [64, 5] and
             getattr(hp, "share_expert_num", None) == 3 and getattr(hp, "independent_expert_num", None) == 2,
             "expert / gate sizes and expert counts of config/ple.yaml (3 shared + 2 per task, gates 64 -> 5)")


class ShareBottomModel(_DinMultiTask):
    """SB:24: no mixing layer, both towers read concat(long, short, target) (SB:196-203)."""
    ENGINE_MODEL = "sharebottom"

    def _check_mixing(self, hp, need):
        pass


class SASRecModel(_DinMultiTask):
    """models/sequential/sasrec.py:16: the satisfied-only history + a position table through two (item + cate)-wide self-attention blocks with
    dense Q / K / V, read out at the last satisfied position, one tower; loss = data + regular.  train() returns the base class's
    5-tuple (update, extra_update_ops, loss, data_loss, summary) (BM:350-372)."""
    ENGINE_MODEL = "sasrec"
    SCALARS = ("loss", "data_loss")                                                        # BM:350-372
    ATTENTION_SLOTS = (("satisfied_item_history", "satisfied_mask"),)

    def _check_mixing(self, hp, need):
        pass

    def step_train(self, step, step_result):
        """SBM:227-236."""
        (_, _, step_loss, step_data_loss, _) = step_result
        if step % self.hparams.show_step == 0:
            print("step {0:d} , total_loss: {1:.4f}, data_loss: {2:.4f}".format(step, step_loss, step_data_loss))

    def batch_train(self, file_iterator, train_sess):
        """SBM:87-125."""
        step, epoch_loss, pending = 0, 0.0, None
        for feed in file_iterator:
            if feed:
                queued = self.train_async(train_sess, feed)
                if pending is not None:
                    epoch_loss += pending.result()[2]
                pending = queued
                step += 1
        if pending is not None:
            epoch_loss += pending.result()[2]
        return epoch_loss
