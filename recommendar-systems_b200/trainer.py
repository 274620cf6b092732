"""Trainer / TopKEvaluator with the reference's contract.

Mirror of /root/reference/src/common/trainer.py:47-548 (`fit`, `_train_epoch` including the
mirror-gradient schedule of models with `mg_enable`, `evaluate`) and
/root/reference/src/utils/topk_evaluator.py:19-149 + utils/metrics.py:12-109.

Differences, all on the host side of the hot path:
* `evaluate` propagates once per pass (`model.restore_embeddings`) and runs the fused
  score + mask + top-K kernel per user batch instead of materialising [Bu, n_items] scores; it
  still hands `batch_matrix_list` (int64 [Bu, max(topk)]) to the evaluator. Ties are broken by
  lower item id (the reference's torch.topk order is arbitrary).
* the hit matrix is built with vectorised numpy (sorted ground truth + searchsorted) instead of a
  Python membership loop; the metric formulas are the reference's, in float64.
* with `sync_free` (default) the loss is accumulated on the device and the NaN abort
  (trainer.py:201-203) is evaluated once per epoch instead of forcing a host sync per batch.
"""
from __future__ import annotations

import itertools
from logging import getLogger
from time import time

import numpy as np
import torch
import torch.optim as optim
from torch.nn.utils.clip_grad import clip_grad_norm_

from . import ops


# ------------------------------------------------------------------------------------- metrics
def recall_(hits, pos_len):
    return (np.cumsum(hits, axis=1) / pos_len.reshape(-1, 1)).mean(axis=0)


def recall2_(hits, pos_len):
    return np.cumsum(hits, axis=1).sum(axis=0) / pos_len.sum()


def precision_(hits, pos_len):
    return (hits.cumsum(axis=1) / np.arange(1, hits.shape[1] + 1)).mean(axis=0)


def ndcg_(hits, pos_len):
    """metrics.py:35-64: per-user IDCG truncated at min(pos_len, K)."""
    k = hits.shape[1]
    disc = 1.0 / np.log2(np.arange(1, k + 1, dtype=np.float64) + 1)
    idcg_all = np.cumsum(disc)
    idcg_len = np.minimum(pos_len, k)
    idcg = idcg_all[np.minimum(np.arange(k)[None, :], idcg_len[:, None] - 1)]
    dcg = np.cumsum(np.where(hits, disc[None, :], 0.0), axis=1)
    return (dcg / idcg).mean(axis=0)


def map_(hits, pos_len):
    """metrics.py:67-92."""
    k = hits.shape[1]
    pre = hits.cumsum(axis=1) / np.arange(1, k + 1)
    sum_pre = np.cumsum(pre * hits.astype(np.float64), axis=1)
    ranges = np.minimum(np.arange(1, k + 1)[None, :], np.minimum(pos_len, k)[:, None])
    return (sum_pre / ranges).mean(axis=0)


metrics_dict = {"ndcg": ndcg_, "recall": recall_, "recall2": recall2_, "precision": precision_,
                "map": map_}


class TopKEvaluator:
    """utils/topk_evaluator.py:19-149."""

    def __init__(self, config):
        self.config = config
        self.metrics = config["metrics"]
        self.topk = config["topk"]
        if isinstance(self.metrics, str):
            self.metrics = [self.metrics]
        for m in self.metrics:
            if m.lower() not in metrics_dict:
                raise ValueError("There is no user grouped topk metric named {}!".format(m))
        self.metrics = [m.lower() for m in self.metrics]
        if isinstance(self.topk, int):
            self.topk = [self.topk]
        for k in self.topk:
            if k <= 0:
                raise ValueError("topk must be a positive integer or a list of positive integers, "
                                 "but get `{}`".format(k))

    @staticmethod
    def hit_matrix(pos_items, topk_index):
        """topk_evaluator.py:88-93 vectorised: hits[u, r] = topk_index[u, r] in pos_items[u]."""
        n, k = topk_index.shape
        lens = np.fromiter((len(p) for p in pos_items), dtype=np.int64, count=n)
        stride = int(topk_index.max()) + 2 if topk_index.size else 1
        flat = np.concatenate(pos_items) if n else np.zeros(0, np.int64)
        keys = np.sort(np.repeat(np.arange(n, dtype=np.int64), lens) * stride + flat)
        q = np.arange(n, dtype=np.int64)[:, None] * stride + topk_index
        pos = np.searchsorted(keys, q.ravel())
        pos = np.minimum(pos, len(keys) - 1)
        return (keys[pos] == q.ravel()).reshape(n, k)

    def evaluate(self, batch_matrix_list, eval_data, is_test=False, idx=0):
        pos_len_list = eval_data.get_eval_len_list()
        topk = torch.cat(batch_matrix_list, dim=0)
        assert len(pos_len_list) == len(topk)
        if topk.is_cuda and hasattr(eval_data, "gt_csr"):
            result = self._device_metrics(topk, eval_data)
        else:
            hits = self.hit_matrix(eval_data.get_eval_items(), topk.numpy())
            result = self._calculate_metrics(pos_len_list, hits)
        out = {}
        for metric, value in zip(self.metrics, result):
            for k in self.topk:
                out["{}@{}".format(metric, k)] = round(value[k - 1], 4)
        return out

    def _device_metrics(self, topk, eval_data):
        """Hit matrix + every metric @1..K on the GPU (mmrec_topk_metrics_f64); only the [5, K]
        float64 sums come back to the host."""
        rowptr, items = eval_data.gt_csr()
        return self._metrics_from_sums(ops.topk_metric_sums(topk, rowptr, items), topk.shape[0], eval_data)

    def result_from_sums(self, sums, n, eval_data):
        """The reference's result dict from the device sums of a (graph-replayed) evaluation."""
        result = self._metrics_from_sums(sums, n, eval_data)
        out = {}
        for metric, value in zip(self.metrics, result):
            for k in self.topk:
                out["{}@{}".format(metric, k)] = round(value[k - 1], 4)
        return out

    def evaluate_sums(self, sums, eval_data):
        """The result dict of a user-sharded evaluation (parallel.ShardedEvalData): `sums` are this
        rank's [5, K] metric sums; they are summed over the evaluation data's process group and
        divided by its global counts, so every rank returns the same dict."""
        sums = eval_data.reduce_metric_sums(sums)
        return self.result_from_sums(sums, eval_data.n_users_global, eval_data)

    def _metrics_from_sums(self, sums, n, eval_data):
        sums = sums.cpu().numpy()
        total_pos = getattr(eval_data, "total_pos", None)        # global count of sharded evaluation data
        if total_pos is None:
            if getattr(eval_data, "_total_pos", None) is None:
                eval_data._total_pos = float(np.asarray(eval_data.get_eval_len_list(), dtype=np.int64).sum())
            total_pos = eval_data._total_pos
        rows = {"recall": sums[0] / n, "recall2": sums[1] / total_pos, "precision": sums[2] / n,
                "ndcg": sums[3] / n, "map": sums[4] / n}
        return np.stack([rows[m] for m in self.metrics], axis=0)

    def _calculate_metrics(self, pos_len_list, hits):
        return np.stack([metrics_dict[m](hits, np.asarray(pos_len_list)) for m in self.metrics],
                        axis=0)


def early_stopping(value, best, cur_step, max_step, bigger=True):
    """utils/utils.py:57-98."""
    stop_flag = update_flag = False
    better = value > best if bigger else value < best
    if better:
        cur_step, best, update_flag = 0, value, True
    else:
        cur_step += 1
        if cur_step > max_step:
            stop_flag = True
    return best, cur_step, stop_flag, update_flag


def dict2str(d):
    return "".join(str(k) + ": " + "%.04f" % v + "    " for k, v in d.items())


# ------------------------------------------------------------------------------------- trainer
class Trainer:
    def __init__(self, config, model, mg=False):
        self.config, self.model = config, model
        self.logger = getLogger()
        self.learner = config["learner"]
        self.learning_rate = config["learning_rate"]
        self.epochs = config["epochs"]
        self.eval_step = min(config["eval_step"], self.epochs)
        self.stopping_step = config["stopping_step"]
        self.clip_grad_norm = config["clip_grad_norm"]
        self.valid_metric = config["valid_metric"].lower()
        self.valid_metric_bigger = config["valid_metric_bigger"]
        self.test_batch_size = config["eval_batch_size"]
        self.device = config["device"]
        wd = config["weight_decay"]
        self.weight_decay = 0.0 if wd is None else (eval(wd) if isinstance(wd, str) else wd)
        self.req_training = config["req_training"]
        self.start_epoch = self.cur_step = 0
        tmp = {f"{j.lower()}@{k}": 0.0 for j, k in itertools.product(config["metrics"], config["topk"])}
        self.best_valid_score = -1
        self.best_valid_result, self.best_test_upon_valid = tmp, tmp
        self.train_loss_dict = {}
        self.optimizer = self._build_optimizer()
        sch = config["learning_rate_scheduler"]
        self.lr_scheduler = optim.lr_scheduler.LambdaLR(self.optimizer,
                                                        lr_lambda=lambda e: sch[0] ** (e / sch[1]))
        self.evaluator = TopKEvaluator(config)
        if hasattr(model, "dropout_counter") and hasattr(self.optimizer, "_hyper") and self.optimizer.param_groups:
            # in-kernel dropout streams follow the optimizer's device-side update count
            g0 = self.optimizer.param_groups[0]
            model.dropout_counter = self.optimizer._hyper(g0, g0["params"][0].device)[1:2]
        self.mg = mg
        self.alpha1, self.alpha2, self.beta = config["alpha1"], config["alpha2"], config["beta"]
        self.mg_target_rel_step = float(config.get("mg_target_rel_step", 1e-3))
        self.mg_alpha_max_scale = float(config.get("mg_alpha_max_scale", 20.0))
        self.sync_free = bool(config.get("sync_free", True))
        # steady-state steps are replayed from a CUDA graph (needs the device-side Adam counters)
        self.use_cuda_graph = bool(config.get("cuda_graph", True)) and \
            hasattr(self.optimizer, "lr_tensor") and not self.clip_grad_norm and not self.mg
        self.graph_warmup = int(config.get("graph_warmup", 2))
        self.use_eval_graph = bool(config.get("cuda_graph", True)) and bool(config.get("eval_cuda_graph", True))
        self._graphs = {}
        self._eval_graphs = {}
        self.replayed_launches = 0
        # the [I, F] gradients of the trainable feature tables stay low-rank (ops.LowRankGrad) when the
        # optimizer is the fused Adam, which consumes them tile by tile; anything that needs `p.grad`
        # itself (gradient clipping, the non-model mirror schedule, torch optimizers) keeps them dense
        model.lowrank_table_grad = bool(config.get("lowrank_table_grad", True)) and \
            hasattr(self.optimizer, "lowrank_params") and not self.clip_grad_norm and not self.mg

    def _build_optimizer(self):
        """trainer.py:126-143."""
        name = self.learner.lower()
        kw = dict(lr=self.learning_rate, weight_decay=self.weight_decay)
        if name == "adam" and self.config.get("fused_adam", True) and \
                all(p.is_cuda for p in self.model.parameters()):
            from .optim import FusedAdam
            return FusedAdam(self.model.parameters(), **kw)
        cls = {"adam": optim.Adam, "sgd": optim.SGD, "adagrad": optim.Adagrad,
               "rmsprop": optim.RMSprop}.get(name)
        if cls is None:
            self.logger.warning("Received unrecognized optimizer, set default Adam optimizer")
            return optim.Adam(self.model.parameters(), lr=self.learning_rate)
        return cls(self.model.parameters(), **kw)

    # ---- one step of the mirror-gradient schedule (trainer.py:268-335) ----------------------
    def _mirror_gradient_step(self, loss_func, mirror_input):
        """trainer.py:268-335. Same arithmetic, but alpha_eff stays a device scalar (no host
        round trip, CUDA-graph capturable) and the gradients of pass 1 are kept by reference
        instead of being cloned (zero_grad(set_to_none) detaches them from the parameters)."""
        opt, model = self.optimizer, self.model
        opt.zero_grad(set_to_none=True)
        loss_curr = loss_func(mirror_input)
        (sum(loss_curr) if isinstance(loss_curr, tuple) else loss_curr).backward()
        params, grads = [], []
        for p in model.parameters():
            if p.requires_grad and p.grad is not None:
                params.append(p)
                grads.append(p.grad.detach())
        # feature tables whose gradient is the never-materialised product dY W (ops.LowRankGrad)
        tables = opt.lowrank_params() if hasattr(opt, "lowrank_params") else []
        alpha_base = float(getattr(model, "mg_alpha", 0.5))
        sharded = [getattr(p, "_mmrec_sharded", False) for p in params]
        fused = hasattr(opt, "lr_tensor") and not any(sharded) and len(opt.param_groups) == 1
        if tables and not fused:
            raise RuntimeError("low-rank table gradients need the fused single-group optimizer path")
        with torch.no_grad():
            from .optim import axpy_multi, lowrank_sumsq, mirror_coef
            if fused:
                # one pass over (theta, g) for both RMS values + the scalar arithmetic on the device;
                # a table brings sum theta^2 from the Adam pass that just updated it and sum g^2 from
                # a tensor-core pass over the factors of its gradient
                numel = float(sum(g.numel() for g in grads) + sum(p.numel() for p in tables))
                extra = None
                if tables:
                    T = len(tables)
                    extra = torch.empty(2 * T, dtype=torch.float64, device=params[0].device)
                    for t, p in enumerate(tables):
                        extra[t:t + 1].copy_(opt.state[p]["sumsq"])
                        lowrank_sumsq(p, extra[T + t:])
                both = mirror_coef(params, grads, opt._hyper(opt.param_groups[0], params[0].device), numel,
                                   alpha_base, self.mg_alpha_max_scale, self.mg_target_rel_step,
                                   extra, len(tables), len(tables))
                coef, model._alpha_eff = both[0:1], both[1]
                for p in tables:
                    # the mirror point theta - coef * dY W of a table is never written: the next
                    # forward / backward evaluate the projection there from the factors (the W factor
                    # is snapshotted because the live W is about to be displaced itself)
                    lr = p._mmrec_lowrank
                    p._mmrec_delta = (coef, lr.dY, lr.W.clone())
            else:
                dev = params[0].device
                if hasattr(opt, "lr_tensor"):
                    lr = opt.lr_tensor().to(torch.float32)
                else:
                    lr = torch.tensor([opt.param_groups[0].get("lr", 1.0)], dtype=torch.float32, device=dev)
                if any(sharded):
                    # item-range sharded feature tables: their rows' squares are summed over the group
                    from . import parallel
                    grp = getattr(model, "_table_group", None)
                    numel = float(sum(getattr(p, "_mmrec_global_numel", p.numel()) for p in params))
                    g2 = parallel.sharded_sumsq([g for g, s in zip(grads, sharded) if not s],
                                                [g for g, s in zip(grads, sharded) if s], grp)
                    p2 = parallel.sharded_sumsq([p.detach() for p, s in zip(params, sharded) if not s],
                                                [p.detach() for p, s in zip(params, sharded) if s], grp)
                else:
                    numel = float(sum(g.numel() for g in grads))
                    g2 = torch.stack(torch._foreach_norm(grads)).pow(2).sum()
                    p2 = torch.stack(torch._foreach_norm([p.detach() for p in params])).pow(2).sum()
                grad_rms = (g2 / numel).sqrt()
                param_rms = (p2 / numel).sqrt() + 1e-12
                alpha_eff = torch.clamp(self.mg_target_rel_step * param_rms / (lr * grad_rms + 1e-12),
                                        min=alpha_base, max=alpha_base * self.mg_alpha_max_scale)
                model._alpha_eff = alpha_eff                      # device scalar (logging only)
                coef = (alpha_eff * lr).reshape(1).contiguous()
            axpy_multi(params, grads, coef, sign=-1.0)        # theta' = theta - alpha_eff*lr*g
        opt.zero_grad(set_to_none=True)
        loss_mirror = loss_func(mirror_input)
        (sum(loss_mirror) if isinstance(loss_mirror, tuple) else loss_mirror).backward()
        beta = -float(getattr(model, "mg_beta", 0.2))
        every = all(p.grad is not None for p in params)
        for p in tables:
            p._mmrec_delta = None
        if tables and not every:
            raise RuntimeError("mirror-gradient step: a dense parameter lost its gradient in the mirror pass")
        if fused and every:
            # back to theta inside the Adam pass (same fmaf as the axpy), gradients scaled as they are read
            opt.step(grad_scale=beta, undo=({p: g for p, g in zip(params, grads)}, coef))
        else:
            with torch.no_grad():
                axpy_multi(params, grads, coef, sign=1.0)         # back to theta
                if not hasattr(opt, "lr_tensor"):                 # plain torch optimizer
                    mg = [p.grad for p in model.parameters() if p.requires_grad and p.grad is not None]
                    torch._foreach_mul_(mg, beta)
            if hasattr(opt, "lr_tensor"):
                opt.step(grad_scale=beta)                         # FusedAdam scales the gradients as it reads them
            else:
                opt.step()
        opt.zero_grad(set_to_none=True)

    def _train_batch(self, interaction, batch_idx=0, loss_func=None):
        """Body of the batch loop of trainer.py:186-335 for one [3, B] interaction; returns the
        detached loss of the first forward (what the reference accumulates)."""
        loss_func = loss_func or self.model.calculate_loss
        self.optimizer.zero_grad(set_to_none=True)
        second_inter = interaction
        losses = loss_func(interaction)
        loss = sum(losses) if isinstance(losses, tuple) else losses
        first = loss.detach()
        model_has_mirror = bool(getattr(self.model, "mg_enable", False))
        if not model_has_mirror:
            if self.mg and batch_idx % self.beta == 0:
                (self.alpha1 * loss).backward()
                self.optimizer.step()
                self.optimizer.zero_grad()
                losses = loss_func(second_inter)
                loss = sum(losses) if isinstance(losses, tuple) else losses
                (-1 * self.alpha2 * loss).backward()
            else:
                loss.backward()
            if self.clip_grad_norm:
                clip_grad_norm_(self.model.parameters(), **self.clip_grad_norm)
            self.optimizer.step()
            return first
        loss.backward()
        if self.clip_grad_norm:
            clip_grad_norm_(self.model.parameters(), **self.clip_grad_norm)
        self.optimizer.step()
        mg_interval = int(getattr(self.model, "mg_interval", 0))
        if mg_interval > 0 and int(getattr(self.model, "global_step", 0)) % mg_interval == 0:
            self._mirror_gradient_step(loss_func, second_inter)
        return first

    # ---- CUDA-graph replay of the steady-state step ------------------------------------------
    def _graph_key(self, interaction):
        m = self.model
        interval = int(getattr(m, "mg_interval", 0)) if getattr(m, "mg_enable", False) else 0
        is_mg = bool(interval > 0 and (int(getattr(m, "global_step", 0)) + 1) % interval == 0)
        return (tuple(interaction.shape), is_mg, int(getattr(m, "graph_version", 0)))

    def _train_batch_graphed(self, interaction, batch_idx=0):
        """Run `_train_batch` through a captured CUDA graph once the same control-flow variant
        (batch shape, mirror-gradient or plain step, adjacency version) has been seen
        `graph_warmup` times; the first executions and ragged batches run eagerly."""
        key = self._graph_key(interaction)
        ent = self._graphs.get(key)
        if ent is None:
            stale = [k for k in self._graphs if k[2] != key[2]]
            for k in stale:
                del self._graphs[k]
            ent = self._graphs[key] = {"seen": 0, "graph": None}
        if ent["graph"] is None:
            if ent["seen"] < self.graph_warmup:
                ent["seen"] += 1
                return self._train_batch(interaction, batch_idx)
            if hasattr(self.optimizer, "sync_lr"):
                self.optimizer.sync_lr()
            static_in = interaction.clone()
            gs0 = int(getattr(self.model, "global_step", 0))
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            from . import lib
            l0 = lib.launch_count()
            with torch.cuda.graph(g):
                static_out = self._train_batch(static_in, batch_idx)
            ent.update(graph=g, static_in=static_in, static_out=static_out,
                       launches=lib.launch_count() - l0,
                       step_delta=int(getattr(self.model, "global_step", 0)) - gs0)
            if ent["step_delta"]:
                self.model.global_step = gs0       # capture ran no kernels; the replay below does
        return self._replay(ent, interaction)

    def _replay(self, ent, interaction):
        if hasattr(self.optimizer, "sync_lr"):
            self.optimizer.sync_lr()
        ent["static_in"].copy_(interaction, non_blocking=True)
        ent["graph"].replay()
        self.replayed_launches += ent["launches"]     # library kernels inside the replayed graph
        if ent["step_delta"]:
            self.model.global_step += ent["step_delta"]
        return ent["static_out"].clone()

    def _post_loss_read(self, loss, idx):
        """Start the device -> host copy of one step's loss (4 bytes) into a pinned slot; returns
        (slot, event). Slots rotate: at most two reads are pending at any time."""
        if not (torch.is_tensor(loss) and loss.is_cuda):
            return None, None
        ring = self.__dict__.get("_loss_slots")
        if ring is None or ring[0].dtype != loss.dtype:
            ring = self._loss_slots = [torch.empty(1, dtype=loss.dtype).pin_memory() for _ in range(4)]
            self._loss_events = [torch.cuda.Event() for _ in range(4)]
        slot, ev = ring[idx % 4], self._loss_events[idx % 4]
        slot.copy_(loss.detach().reshape(1), non_blocking=True)
        ev.record()
        return slot, ev

    def _train_epoch(self, train_data, epoch_idx, loss_func=None, max_batches=None):
        """trainer.py:145-356. The batch loop is software-pipelined: the step is enqueued (a CUDA
        graph replay returns at once), THEN the loader draws the next batch -- host-side negative
        sampling overlaps the device step -- and only then the loss is read back. Batches, RNG
        call order and the per-step loss / NaN semantics are the reference's. `max_batches` stops
        early (bench.py times K steps through this entry point)."""
        if not self.req_training:
            return 0.0, []
        self.model.train()
        loss_func = loss_func or self.model.calculate_loss
        total_loss = None
        first_nan = None
        loss_batches = []
        graphed = self.use_cuda_graph and loss_func == self.model.calculate_loss
        it = iter(train_data)
        interaction = next(it, None)
        batch_idx = 0
        unread = []                      # (loss, batch index) enqueued but not yet read back
        while interaction is not None:
            loss = self._train_batch_graphed(interaction, batch_idx) if graphed \
                else self._train_batch(interaction, batch_idx, loss_func)
            batch_idx += 1
            if max_batches is not None and batch_idx >= max_batches:
                interaction = None
                if hasattr(train_data, "pr"):
                    train_data.pr = 0                  # abandoned epoch: the next one starts clean
            else:
                interaction = next(it, None)
                if interaction is None and epoch_idx + 1 < self.epochs and hasattr(train_data, "prefetch_shuffle") \
                        and bool(self.config.get("prefetch_epoch_shuffle", True)):
                    # the device still has the last step(s) queued: shuffle for the next epoch under them
                    train_data.prefetch_shuffle()
            loss_batches.append(loss)
            if self.sync_free:
                total_loss = loss.clone() if total_loss is None else total_loss + loss
                # index of the first NaN batch, kept on the device (read once, at the end of the epoch)
                bad = torch.isnan(loss).reshape(())
                here = torch.full((), batch_idx - 1, dtype=torch.int64, device=loss.device)
                first_nan = torch.where(bad, here, torch.full_like(here, -1)) if first_nan is None else \
                    torch.where((first_nan < 0) & bad, here, first_nan)
                continue
            # per-batch read-back (trainer.py:196-203), one step behind: the loss of batch i is
            # read after batch i + 1 has been enqueued, so the device never waits for the host.
            # A NaN therefore aborts one batch later than in the reference.
            # `loss.item()` would not do that: its copy is enqueued BEHIND the step that was just
            # launched, so it returns when batch i + 1 is done and the device then idles while the
            # host enqueues the next replay (measured: 50 us per 2.33 ms step). The loss goes to a
            # pinned slot by an asynchronous copy followed by an event instead; waiting for the
            # event of batch i leaves batch i + 1 running.
            unread.append((loss, batch_idx - 1) + self._post_loss_read(loss, batch_idx - 1))
            while len(unread) > (1 if interaction is not None else 0):
                lt, bi, slot, ev = unread.pop(0)
                if ev is None:
                    v = lt.item()
                else:
                    ev.synchronize()
                    v = slot.item()
                total_loss = v if total_loss is None else total_loss + v
                if v != v:
                    self.logger.info("Loss is nan at epoch: {}, batch index: {}. Exiting.".format(epoch_idx, bi))
                    return lt, torch.tensor(0.0)
        if self.sync_free and total_loss is not None:
            if torch.isnan(total_loss):
                # trainer.py:201-203 reports the batch and returns before its backward; here the batch
                # index is exact but the remaining batches of the epoch have already been applied
                self.logger.info("Loss is nan at epoch: {}, batch index: {}. Exiting.".format(
                    epoch_idx, int(first_nan.item()) if first_nan is not None else -1))
                return total_loss, torch.tensor(0.0)
            total_loss = total_loss.item()
        return total_loss, loss_batches

    def _valid_epoch(self, valid_data):
        valid_result = self.evaluate(valid_data)
        valid_score = valid_result[self.valid_metric] if self.valid_metric else valid_result["NDCG@20"]
        return valid_score, valid_result

    def fit(self, train_data, valid_data=None, test_data=None, saved=False, verbose=True):
        """trainer.py:385-506."""
        for epoch_idx in range(self.start_epoch, self.epochs):
            t0 = time()
            self.model.cur_epoch = epoch_idx
            self.model.pre_epoch_processing()
            train_loss, _ = self._train_epoch(train_data, epoch_idx)
            if torch.is_tensor(train_loss):
                break
            self.lr_scheduler.step()
            self.train_loss_dict[epoch_idx] = sum(train_loss) if isinstance(train_loss, tuple) else train_loss
            t1 = time()
            post_info = self.model.post_epoch_processing()
            if verbose:
                self.logger.info("epoch %d training [time: %.2fs, train loss: %.4f]" % (epoch_idx, t1 - t0, train_loss))
                if post_info is not None:
                    self.logger.info(post_info)
            if (epoch_idx + 1) % self.eval_step == 0:
                v0 = time()
                valid_score, valid_result = self._valid_epoch(valid_data)
                self.best_valid_score, self.cur_step, stop_flag, update_flag = early_stopping(
                    valid_score, self.best_valid_score, self.cur_step, max_step=self.stopping_step,
                    bigger=self.valid_metric_bigger)
                v1 = time()
                _, test_result = self._valid_epoch(test_data)
                if verbose:
                    self.logger.info("epoch %d evaluating [time: %.2fs, valid_score: %f]" % (epoch_idx, v1 - v0, valid_score))
                    self.logger.info("valid result: \n" + dict2str(valid_result))
                    self.logger.info("test result: \n" + dict2str(test_result))
                if update_flag:
                    if verbose:
                        self.logger.info("██ " + str(self.config["model"]) + "--Best validation results updated!!!")
                    self.best_valid_result = valid_result
                    self.best_test_upon_valid = test_result
                if stop_flag:
                    if verbose:
                        self.logger.info("+++++Finished training, best eval result in epoch %d" %
                                         (epoch_idx - self.cur_step * self.eval_step))
                    break
        return self.best_valid_score, self.best_valid_result, self.best_test_upon_valid

    @torch.no_grad()
    def evaluate_topk(self, eval_data):
        """Fused evaluation: list of int64 [Bu, max(topk)] (trainer.py:509-527)."""
        self.model.eval()
        k = max(self.config["topk"])
        users = eval_data.eval_u
        n, step = users.shape[0], eval_data.step
        # The reference scores `eval_batch_size` users at a time because it materialises the
        # [Bu, n_items] score matrix; the fused kernel keeps scores on chip, so several reference
        # batches go out as one launch (a fuller wave, the top-K fill phase paid once per user) and
        # the result is cut back into the reference's batch list.
        fuse = step * max(1, int(self.config.get("eval_fuse_users", 32768)) // step)
        out = []
        for start in range(0, n, fuse):
            stop = min(n, start + fuse)
            rowptr, cols = eval_data.mask_csr(start, stop)
            ids = self.model.full_sort_topk(users[start:stop], k, rowptr, cols)
            out.extend(ids.split(step, dim=0))
        return out

    @torch.no_grad()
    def evaluate(self, eval_data, is_test=False, idx=0):
        """trainer.py:509-528. On CUDA the whole pass -- evaluation forward, fused score + mask +
        top-K, device metrics -- is captured in a CUDA graph the second time a loader is evaluated
        and replayed afterwards (parameters are read in place, so replays see the current model);
        one [5, K] float64 copy comes back to the host.
        User-sharded evaluation data (parallel.ShardedEvalData, reduce_metric_sums): every rank scores
        its own users (model.eval_metric_sums) and the sums are reduced over the group; eager, the
        pass has NCCL calls."""
        if hasattr(eval_data, "reduce_metric_sums"):
            self.model.eval()
            sums = self.model.eval_metric_sums(eval_data, max(self.config["topk"]))
            return self.evaluator.evaluate_sums(sums, eval_data)
        if not self.use_eval_graph or not hasattr(eval_data, "gt_csr") or not eval_data.eval_u.is_cuda:
            return self.evaluator.evaluate(self.evaluate_topk(eval_data), eval_data, is_test=is_test, idx=idx)
        key = (id(eval_data), id(self.model))
        ent = self._eval_graphs.get(key)
        if ent is None:
            self._eval_graphs[key] = {"graph": None, "eval_data": eval_data}     # first pass: eager warm-up
            return self.evaluator.evaluate(self.evaluate_topk(eval_data), eval_data, is_test=is_test, idx=idx)
        if ent["graph"] is None:
            from . import lib
            rowptr, items = eval_data.gt_csr()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            l0 = lib.launch_count()
            with torch.cuda.graph(g):
                self.model._eval_cache = None
                topk = torch.cat(self.evaluate_topk(eval_data), dim=0)
                sums = ops.topk_metric_sums(topk, rowptr, items)
            self.model._eval_cache = None          # the captured forward wrote into graph-owned memory
            ent.update(graph=g, sums=sums, topk=topk, launches=lib.launch_count() - l0)
        self.model.eval()
        ent["graph"].replay()
        self.replayed_launches += ent["launches"]
        return self.evaluator.result_from_sums(ent["sums"], ent["topk"].shape[0], eval_data)
