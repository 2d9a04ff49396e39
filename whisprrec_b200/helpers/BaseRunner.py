"""Training / evaluation driver with the reference's interface (reference src/helpers/BaseRunner.py).

Same flags, same epoch loop, same early stopping, same log lines.  Differences are all underneath:

* fit():   the epoch's batches are assembled once on the host in the reference's order (the torch-global-generator
           draws of DataLoader + RandomSampler are replayed, BaseRunner.py:188-193), uploaded once, and every
           step is `model.predict` (fused forward+backward kernel) + `optimizer.step` (fused Adam sweep).
           Per-step losses stay on the device and are read back once per epoch (the reference syncs every
           step, :200).
* evaluate(): ranks come from the fused score/mask/rank kernel and HR/NDCG from wr_metrics; the
           [n_eval, n_items] score matrix of interface() (:242-257) is never built.
"""
import gc
import logging
import os
import threading
from time import time

import numpy as np
import torch

from ..utils import utils
from .. import _lib


def dataloader_draws(n, shuffle):
    """What `iter(DataLoader(...))` takes from torch's global CPU generator (torch/utils/data/dataloader.py
    `_base_seed`, torch/utils/data/sampler.py RandomSampler.__iter__).  Returns the epoch permutation for a
    shuffling loader, None for a sequential one.  Keeping these draws keeps every later epoch's order equal
    to the reference's."""
    torch.empty((), dtype=torch.int64).random_()
    if not shuffle:
        return None
    seed = int(torch.empty((), dtype=torch.int64).random_().item())
    g = torch.Generator()
    g.manual_seed(seed)
    return torch.randperm(n, generator=g).numpy()


class BaseRunner(object):
    @staticmethod
    def parse_runner_args(parser):
        parser.add_argument('--epoch', type=int, default=200, help='Number of epochs.')
        parser.add_argument('--check_epoch', type=int, default=1, help='Check some tensors every check_epoch.')
        parser.add_argument('--test_epoch', type=int, default=-1,
                            help='Print test results every test_epoch (-1 means no print).')
        parser.add_argument('--early_stop', type=int, default=10,
                            help='The number of epochs when dev results drop continuously.')
        parser.add_argument('--lr', type=float, default=5e-4, help='Learning rate.')
        parser.add_argument('--l2', type=float, default=0, help='Weight decay in optimizer.')
        parser.add_argument('--batch_size', type=int, default=2048, help='Batch size during training.')
        parser.add_argument('--eval_batch_size', type=int, default=2048, help='Batch size during testing.')
        parser.add_argument('--optimizer', type=str, default='Adam', help='optimizer: SGD, Adam, Adagrad, Adadelta')
        parser.add_argument('--num_workers', type=int, default=5,
                            help='Number of processors when prepare batches in DataLoader')
        parser.add_argument('--pin_memory', type=int, default=0, help='pin_memory in DataLoader')
        parser.add_argument('--topk', type=str, default='10,20', help='The number of items recommended to each user.')
        parser.add_argument('--metric', type=str, default='NDCG, HR', help='metrics: NDCG, RECALL')
        return parser

    @staticmethod
    def metrics_from_ranks(gt_rank, topk, metrics):
        """BaseRunner.py:76-88 given the rank of the ground-truth item (host, float64)."""
        gt_rank = np.asarray(gt_rank)
        out = dict()
        for k in topk:
            hit = gt_rank <= k
            for metric in metrics:
                key = '{}@{}'.format(metric, k)
                name = metric.lower()
                if name in ('hr', 'recall'):
                    out[key] = hit.mean()
                elif name == 'ndcg':
                    out[key] = np.mean(hit / np.log2(gt_rank + 1))
                elif name == 'precision':
                    out[key] = hit.sum() / (hit.shape[0] * k)
                else:
                    raise ValueError('Undefined evaluation metric: {}.'.format(metric))
        return out

    @staticmethod
    def evaluate_method(predictions, topk, metrics):
        """BaseRunner.py:50-92: `predictions` is [n, 1 + n_candidates] with the ground truth in column 0."""
        order = (-predictions).argsort(axis=1)
        gt_rank = np.argwhere(order == 0)[:, 1] + 1
        return BaseRunner.metrics_from_ranks(gt_rank, topk, metrics)

    # runner flags copied onto the instance under the reference's attribute names (BaseRunner.py:94-110)
    _PLAIN_ATTRS = ('epoch', 'check_epoch', 'test_epoch', 'early_stop', 'batch_size', 'eval_batch_size', 'l2',
                    'num_workers', 'pin_memory')

    def __init__(self, args):
        for name in self._PLAIN_ATTRS:
            setattr(self, name, getattr(args, name))
        self.learning_rate, self.optimizer_name = float(args.lr), args.optimizer
        self.topk = [int(k) for k in args.topk.split(',')]
        self.metrics = [name.strip().upper() for name in args.metric.split(',')]
        self.main_metric = '%s@%d' % (self.metrics[0], self.topk[0])      # early stopping watches this one
        self.time = None                                # [start of train(), last lap]
        self.eval_precision = getattr(args, 'eval_precision', 2)     # the ranks of 0, on the tensor cores
        self.last_epoch_stats = {}

    def _check_time(self, start=False):
        """Lap timer of BaseRunner.py:112-118: seconds since the previous call (the start time on a (re)start)."""
        now = time()
        if start or self.time is None:
            self.time = [now, now]
            return now
        lap, self.time[1] = now - self.time[1], now
        return lap

    def _build_optimizer(self, model):
        logging.info('Optimizer: ' + self.optimizer_name)
        return model.build_optimizer(self.optimizer_name, self.learning_rate, self.l2)

    def _run_epoch(self, number, data_dict, history):
        """One pass of the reference's epoch body (BaseRunner.py:133-166): fit, dev (and optionally test) evaluation,
        checkpoint on a new best, one log line in the reference's format.  Returns True when training should stop."""
        model = data_dict['train'].model
        self._check_time()
        gc.collect()
        torch.cuda.empty_cache()
        loss = self.fit(data_dict['train'], epoch=number)
        fit_seconds = self._check_time()
        if model.check_list and self.check_epoch > 0 and (number - 1) % self.check_epoch == 0:
            utils.check(model.check_list)
        dev = self.evaluate(data_dict['dev'], self.topk[:1], self.metrics)
        history.append(dev)
        line = 'Epoch {:<5} loss={:<.4f} [{:<3.1f} s]    dev=({})'.format(number, loss, fit_seconds,
                                                                        utils.format_metric(dev))
        if self.test_epoch > 0 and (number - 1) % self.test_epoch == 0:
            test = self.evaluate(data_dict['test'], self.topk[:1], self.metrics)
            line += ' test=({})'.format(utils.format_metric(test))
        line += ' [{:<.1f} s]'.format(self._check_time())
        watched = [h[self.main_metric] for h in history]
        if watched[-1] == max(watched) or getattr(model, 'stage', None) == 1:
            model.save_model()
            line += ' *'
        logging.info(line)
        if self.early_stop > 0 and self.eval_termination(watched):
            logging.info('Early stop at %d based on dev result.' % number)
            return True
        return False

    def train(self, data_dict):
        """BaseRunner.py:126-178: epochs until the budget or the early-stop rule ends them, then reload the best."""
        model = data_dict['train'].model
        history = []                                    # dev results, one dict per finished epoch
        self._check_time(start=True)
        try:
            for number in range(1, self.epoch + 1):
                if self._run_epoch(number, data_dict, history):
                    break
        except KeyboardInterrupt:
            logging.info('Early stop manually')
            answer = input('Exit completely without evaluation? (y/n) (default n):')
            if answer.lower().startswith('y'):
                logging.info(os.linesep + '-' * 45 + ' END: ' + utils.get_time() + ' ' + '-' * 45)
                exit(1)
        watched = [h[self.main_metric] for h in history]
        best = watched.index(max(watched))
        logging.info(os.linesep + 'Best Iter(dev)={:>5}\t dev=({}) [{:<.1f} s] '.format(
            best + 1, utils.format_metric(history[best]), self.time[1] - self.time[0]))
        model.load_model()

    def epoch_batches(self, dataset):
        """The epoch's (user, pos, neg) in the reference's batch order, as int64 device tensors."""
        model = dataset.model
        dev = model.tables.P.device
        # BaseRunner.py:184 then :188-193.  The sampler consumes NumPy's global generator, the loader draws torch's:
        # two independent streams, so the device sampler (a C call that waits for the GPU) runs beside the CPU randperm.
        failure = []

        def sample():
            try:
                torch.cuda.set_device(dev)                   # the CUDA current device is per thread
                dataset.actions_before_epoch()
            except BaseException as e:  # noqa: BLE001 - re-raised on the caller's thread
                failure.append(e)
        if len(dataset) >= 200_000:                          # below that a thread hand-over costs more than it hides
            worker = threading.Thread(target=sample)
            worker.start()
            try:
                perm = dataloader_draws(len(dataset), shuffle=True)
            finally:
                worker.join()
            if failure:
                raise failure[0]
        else:
            dataset.actions_before_epoch()
            perm = dataloader_draws(len(dataset), shuffle=True)
        if getattr(dataset, 'neg_device', None) is not None:
            # negatives were drawn on the device: only the permutation crosses the bus
            user, item = dataset._device_cols(dev)[:2]
            p = torch.from_numpy(perm).to(dev)
            return torch.stack([user[p], item[p], dataset.neg_device[p]])
        cols = [dataset.data['user_id'], dataset.data['item_id'], dataset.data['neg_items']]
        host = torch.from_numpy(np.stack([np.asarray(c, dtype=np.int64)[perm] for c in cols]))
        return host.to(dev, non_blocking=False)

    def fit(self, dataset, epoch=-1):
        """BaseRunner.py:180-201."""
        model = dataset.model
        model.fuse()
        if model.optimizer is None:
            model.optimizer = self._build_optimizer(model)
        if model.num_neg != 1:
            raise NotImplementedError('the fused BPR step takes one negative per interaction (reference default)')
        model.train()
        t0 = time()
        batches = self.epoch_batches(dataset)
        t1 = time()
        n = batches.shape[1]
        starts = list(range(0, n, self.batch_size))
        losses = torch.empty(len(starts), dtype=torch.float32, device=batches.device)
        fused_step = hasattr(model, 'train_step')
        if model.sharded is not None:
            return self._fit_sharded(model, batches, starts, losses, t0, t1)
        if hasattr(model, 'train_epoch'):
            model.train_epoch(batches.contiguous(), self.batch_size, losses)      # the whole step loop in one C call
            starts = []
        for s, lo in enumerate(starts):
            hi = min(n, lo + self.batch_size)
            batch = {'user_id': batches[0, lo:hi], 'pos_item': batches[1, lo:hi], 'neg_items': batches[2, lo:hi],
                     'batch_size': hi - lo, 'phase': 'train'}
            if fused_step:
                model.train_step(batch, loss_out=losses[s:s + 1])      # :196-199 in one launch
                continue
            model.optimizer.zero_grad()
            loss = model.predict(batch, loss_out=losses[s:s + 1])
            loss.backward()
            model.optimizer.step()
        loss_host = losses.cpu().numpy()                    # one sync per epoch
        model.tables.ws.raise_on_status()
        self.last_epoch_stats = {'host_prep_s': t1 - t0, 'device_s': time() - t1, 'steps': len(loss_host), 'rows': n}
        return np.mean(loss_host).item()

    def _fit_sharded(self, model, batches, starts, losses, t0, t1):
        """The same epoch on row-sharded tables: every rank built the same batches (same seeds) and takes its
        slice of each; the global batch -- hence the result -- is the single-GPU one."""
        st = model.sharded
        n = batches.shape[1]
        for s, lo in enumerate(starts):
            hi = min(n, lo + self.batch_size)
            if hi - lo < st.layout.world:        # the same test on every rank: nobody enters the step alone
                raise NotImplementedError('a (last) batch of %d rows is smaller than the %d ranks; choose a batch size '
                                          'that does not leave such a remainder' % (hi - lo, st.layout.world))
            a, b = st.layout.batch_slice(hi - lo)
            loss = model.sharded_train_step(batches[0, lo + a:lo + b], batches[1, lo + a:lo + b],
                                            batches[2, lo + a:lo + b], hi - lo, self.learning_rate, self.l2)
            losses[s:s + 1].copy_(loss[:1])
        if model.optimizer is not None:
            model.optimizer.step_count = st.step_count
        loss_host = losses.cpu().numpy()
        st.ws.raise_on_status()
        self.last_epoch_stats = {'host_prep_s': t1 - t0, 'device_s': time() - t1, 'steps': len(starts), 'rows': n}
        return np.mean(loss_host).item()

    def eval_termination(self, criterion):
        """BaseRunner.py:203-208: stop after `early_stop` epochs that never improved on their predecessor, or once the
        best epoch lies more than `early_stop` epochs back."""
        patience = self.early_stop
        stalled = len(criterion) > patience and utils.non_increasing(criterion[-patience:])
        epochs_since_best = len(criterion) - criterion.index(max(criterion))
        return bool(stalled or epochs_since_best > patience)

    def _eval_inputs(self, dataset):
        """Device copies of the eval rows and the history CSR, cached on the dataset / model."""
        model = dataset.model
        t = model.fuse()
        dev = t.P.device
        if getattr(dataset, '_dev_rows', None) is None or dataset._dev_rows[0].device != dev:
            dataset._dev_rows = (torch.from_numpy(np.asarray(dataset.data['user_id'], dtype=np.int64)).to(dev),
                                 torch.from_numpy(np.asarray(dataset.data['item_id'], dtype=np.int64)).to(dev))
        if getattr(model, '_dev_hist', None) is None or model._dev_hist[0].device != dev:
            ptr, idx = dataset.corpus.history_csr()
            if len(idx) == 0:
                idx = np.zeros(1, dtype=np.int32)
            model._dev_hist = (torch.from_numpy(ptr).to(dev), torch.from_numpy(idx).to(dev))
        return dataset._dev_rows, model._dev_hist

    def rank_topk(self, dataset, k=0):
        """Ranks of the ground-truth items (and optionally the top-k lists) on the device."""
        model = dataset.model
        model.eval()
        dataloader_draws(len(dataset), shuffle=False)        # the `_base_seed` draw of BaseRunner.py:229-234
        if not model.test_all:
            raise KeyError('neg_items')                      # what the reference hits with --test_all 0
        (user, pos), (hptr, hidx) = self._eval_inputs(dataset)
        if model.sharded is not None:
            from .. import sharded as S
            st = model.sharded
            if getattr(model, '_dev_hist_local', None) is None:
                lp, li = st.layout.localise_history(*dataset.corpus.history_csr())
                model._dev_hist_local = (torch.from_numpy(lp).to(user.device), torch.from_numpy(li).to(user.device))
            shards, items_local = model.sharded_eval_tables()
            rank, target, tki, tkv = S.sharded_eval(st, shards, items_local, user, pos, model._dev_hist_local, k=k,
                                                    precision=self.eval_precision)
            return rank, target, tki, tkv, None
        ue, ie = model.eval_tables()
        out = _lib.eval_rank_topk(ue, ie, user, pos, hptr, hidx, model.tables.ws, k=k,
                                  precision=self.eval_precision)
        return out

    def recommend(self, dataset, k=None):
        """Top-k recommendation lists for each row of `dataset`: (items int64 [n, k], scores float32 [n, k]) as host
        NumPy arrays, best first, in the corpus's item codes.  The user's history is masked as in evaluation; rows with
        fewer than k candidates are padded with (-1, -inf).  k defaults to max(self.topk).  At the default precision 2
        the lists equal precision 0's.  On a sharded model every rank returns the same lists.  k is at most 256 (lists
        of more than 32 items at precision 0 or 2)."""
        k = max(self.topk) if k is None else int(k)
        if not 1 <= k <= _lib.TOPK_LONG_KMAX:
            raise ValueError(f'recommend: k must be in 1..{_lib.TOPK_LONG_KMAX}, got {k}')
        _, _, tki, tkv, _ = self.rank_topk(dataset, k=k)
        dataset.model.tables.ws.raise_on_status()
        return tki.to(torch.int64).cpu().numpy(), tkv.cpu().numpy()

    def evaluate(self, dataset, topks, metrics):
        """BaseRunner.py:210-216 -> {metric@k: float64}."""
        rank = self.rank_topk(dataset)[0]
        ws = dataset.model.tables.ws
        for m in metrics:
            if m.lower() not in ('hr', 'ndcg', 'recall', 'precision'):
                raise ValueError('Undefined evaluation metric: {}.'.format(m))
        res = _lib.metrics(rank, topks, ws).cpu().numpy()   # [2, nk] float64: HR, NDCG
        ws.raise_on_status()
        out = dict()
        for i, k in enumerate(topks):
            for metric in metrics:
                name = metric.lower()
                key = '{}@{}'.format(metric, k)
                if name in ('hr', 'recall'):
                    out[key] = res[0, i]
                elif name == 'ndcg':
                    out[key] = res[1, i]
                else:
                    out[key] = res[0, i] / k                # hits / (n * k)
        return out

    def interface(self, dataset):
        """BaseRunner.py:218-258: the dense [n, 1 + n_items] prediction matrix (compatibility API; small data)."""
        model = dataset.model
        model.eval()
        dataloader_draws(len(dataset), shuffle=False)
        (user, pos), (hptr, hidx) = self._eval_inputs(dataset)
        ue, ie = model.eval_tables()
        _, target, _, _, scores = _lib.eval_rank_topk(ue, ie, user, pos, hptr, hidx, model.tables.ws, scores=True)
        scores, target = scores.cpu().numpy(), target.cpu().numpy()
        hp, hi = dataset.corpus.history_csr()
        if model.test_all:
            for row, u in enumerate(dataset.data['user_id']):
                scores[row, hi[hp[u]:hp[u + 1]]] = -np.inf
        return np.concatenate([target[:, np.newaxis], scores], axis=1)

    def print_res(self, dataset):
        result_dict = self.evaluate(dataset, self.topk, self.metrics)
        return '(' + utils.format_metric(result_dict) + ')'
