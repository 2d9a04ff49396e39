"""Model base classes with the reference's protocol (reference src/models/BaseModel.py).

`BaseModel` / `GeneralModel` / nested `Dataset` keep the names, constructor arguments, flags and state_dict
keys of the reference, so `main.py` and `BaseRunner` drive them unchanged.  What differs is underneath:

* parameters live in ONE contiguous fp32 table [n_users + n_items, D] on the device (`FusedTables`), the
  two `nn.Embedding.weight`s are views into it, and Adam's m / v and the dense gradient are tables of the
  same shape, so the optimizer is a single streaming sweep (wr_adam_l2_sweep);
* `predict` runs the fused forward+backward kernel and leaves the gradient in the table; the returned loss
  is a device scalar whose `.backward()` is a no-op, so `loss = model.predict(b); loss.backward();
  model.optimizer.step()` still reads like BaseRunner.py:196-199;
* negative sampling (`Dataset.actions_before_epoch`) consumes NumPy's global MT19937 stream exactly as
  BaseModel.py:167-177 does, but only walks the rows whose first draw was rejected.
"""
import logging

import numpy as np
import torch
import torch.nn as nn

from ..utils import utils
from .. import _lib


class FusedLoss(torch.Tensor):
    """Loss of a fused forward+backward launch: the gradient already sits in the model's grad table."""

    def backward(self, *args, **kwargs):  # noqa: D401 - keeps BaseRunner.py:198 valid
        return None


class FusedAdam(object):
    """torch.optim.Adam(params, lr, weight_decay=l2) for a model whose tables are fused (BaseRunner.py:120-124).

    `zero_grad` is a no-op (the sweep leaves the gradient table zeroed) and `step` is one kernel over all rows.
    """

    def __init__(self, model, lr, weight_decay=0.0, betas=(0.9, 0.999), eps=1e-8):
        self.model, self.lr, self.weight_decay, self.betas, self.eps = model, float(lr), float(weight_decay), betas, eps
        self.step_count = 0

    def zero_grad(self, set_to_none=True):
        return None

    def step(self, dev_scalars=None):
        self.model.quiesce()
        t = self.model.tables
        self.step_count += 1
        _lib.adam_l2_sweep(t.P, t.M, t.V, t.G, self.step_count, self.lr, self.weight_decay, self.betas[0],
                           self.betas[1], self.eps, dev_scalars=dev_scalars)

    def state_dict(self):
        self.model.quiesce()
        t = self.model.tables
        return {'step': self.step_count, 'exp_avg': t.M.clone(), 'exp_avg_sq': t.V.clone()}


class FusedTables(object):
    """P / M / V / G as contiguous [n_users + n_items, D] fp32 device tables plus the kernel workspace."""

    def __init__(self, user_weight, item_weight):
        dev = user_weight.device
        if dev.type != 'cuda':
            raise _lib.WhisprError('whisprrec_b200 runs on a CUDA device only (no CPU fallback); '
                                   'got parameters on %s' % dev)
        self.n_users, self.n_items, self.D = user_weight.shape[0], item_weight.shape[0], user_weight.shape[1]
        n = self.n_users + self.n_items
        self.P = torch.empty((n, self.D), dtype=torch.float32, device=dev)
        self.P[:self.n_users].copy_(user_weight)
        self.P[self.n_users:].copy_(item_weight)
        self.M = torch.zeros_like(self.P)
        self.V = torch.zeros_like(self.P)
        self.G = torch.zeros_like(self.P)
        self.ws = _lib.Workspace(dev)
        self.loss = torch.zeros(1, dtype=torch.float32, device=dev)

    def users(self, t):
        return t[:self.n_users]

    def items(self, t):
        return t[self.n_users:]


class BaseModel(nn.Module):
    reader, runner = None, None
    extra_log_args = []

    @staticmethod
    def parse_model_args(parser):
        parser.add_argument('--model_path', type=str, default='', help='Model save path.')
        parser.add_argument('--buffer', type=int, default=1, help='Whether to buffer feed dicts for dev/test')
        return parser

    def __init__(self, args, corpus):
        super(BaseModel, self).__init__()
        self.device = args.device
        self.model_path = args.model_path
        self.buffer = args.buffer
        self.optimizer = None
        self.check_list = list()

    def forward(self, *args, **kwargs):
        pass

    def loss(self, out_dict):
        pass

    def save_model(self, model_path=None):
        """BaseModel.py:48-53: state_dict only (same keys / shapes / dtype as the reference).  Sharded: the rows
        are collected from their owners first and rank 0 writes the file."""
        model_path = self.model_path if model_path is None else model_path
        self.quiesce()
        st = getattr(self, 'sharded', None)
        if st is not None:
            self.unshard()
            if st.peers.rank != 0:
                return
        utils.check_dir(model_path)
        torch.save(self.state_dict(), model_path)

    def load_model(self, model_path=None):
        model_path = self.model_path if model_path is None else model_path
        st = getattr(self, 'sharded', None)
        if st is not None:
            st.peers.host_sync()                 # rank 0 has finished writing
        self.load_state_dict(torch.load(model_path))
        if st is not None:
            t = self.tables
            st.load_full(t.users(t.P), t.items(t.P))
        logging.info('Load model from ' + model_path)

    def quiesce(self):
        """Nothing of this model runs asynchronously to its stream by default (BPRMF's host-fed kernel overrides)."""

    def count_variables(self):
        return sum(p.numel() for p in self.parameters() if p.requires_grad)

    def actions_after_train(self):
        pass

    class Dataset(torch.utils.data.Dataset):
        def __init__(self, model, corpus, phase):
            self.model = model
            self.corpus = corpus
            self.phase = phase
            self.buffer_dict = dict()
            self.data = utils.df_to_dict(corpus.data_df[phase])

        def __len__(self):
            for key in self.data:
                return len(self.data[key])
            return 0

        def __getitem__(self, index):
            return self._get_feed_dict(index)

        def _get_feed_dict(self, index):
            pass

        def actions_before_epoch(self):
            pass

        def collate_batch(self, feed_dicts):
            """BaseModel.py:96-127 for the fixed-length fields the general models use."""
            out = dict()
            for key in feed_dicts[0]:
                out[key] = torch.from_numpy(np.array([d[key] for d in feed_dicts]))
            out['batch_size'] = len(feed_dicts)
            out['phase'] = self.phase
            return out


class GeneralModel(BaseModel):
    reader, runner = 'BaseReader', 'BaseRunner'

    @staticmethod
    def parse_model_args(parser):
        parser.add_argument('--num_neg', type=int, default=1, help='The number of negative items during training.')
        parser.add_argument('--test_all', type=int, default=1, help='Whether testing on all the items.')
        return BaseModel.parse_model_args(parser)

    def __init__(self, args, corpus):
        super().__init__(args, corpus)
        self.user_num = int(corpus.n_users)
        self.item_num = int(corpus.n_items)
        self.num_neg = args.num_neg
        self.test_all = args.test_all
        self.tables = None
        # The reference takes any embedding size; here training runs any multiple of 4 but the full-ranking evaluation
        # kernels exist for a few sizes only.  Say so now, not at the first dev evaluation after an epoch of training.
        emb = getattr(args, 'embedding_size', None)
        if emb is not None and int(emb) not in _lib.EVAL_DIMS:
            raise ValueError('--embedding_size %s: the evaluation kernels of whisprrec_b200 support %s'
                             % (emb, ', '.join(str(d) for d in _lib.EVAL_DIMS)))

    # ---- fused parameter tables ----------------------------------------------------------------------
    def _embedding_pair(self):
        """(user nn.Embedding, item nn.Embedding) -- named differently by BPRMF and LightGCN."""
        raise NotImplementedError

    def fuse(self):
        """Move the two embedding weights into one device table (idempotent; re-fuses after `.to()`)."""
        ue, ie = self._embedding_pair()
        t = self.tables
        if t is not None and ue.weight.data_ptr() == t.P.data_ptr() and \
                ie.weight.data_ptr() == t.P[t.n_users:].data_ptr():
            return t
        t = FusedTables(ue.weight.data, ie.weight.data)
        ue.weight.data = t.users(t.P)
        ie.weight.data = t.items(t.P)
        ue.weight.grad = t.users(t.G)
        ie.weight.grad = t.items(t.G)
        self.tables = t
        self._on_fused()
        return t

    def _on_fused(self):
        pass

    def _prepare_grads(self):
        """Integration level L1 (SURVEY.md section 8b): when something other than FusedAdam drives the step -- the
        reference's own BaseRunner builds `torch.optim.Adam(model.parameters())` and calls `zero_grad()`, which since
        torch 2.0 sets `.grad = None` -- the gradient table is cleared here (no fused sweep re-zeroes it) and the two
        `.grad` views into it are re-attached, so `loss.backward(); optimizer.step()` sees the kernel's gradient."""
        t = self.tables
        ue, ie = self._embedding_pair()
        if not isinstance(self.optimizer, FusedAdam):
            t.G.zero_()
        if ue.weight.grad is None or ue.weight.grad.data_ptr() != t.G.data_ptr():
            ue.weight.grad = t.users(t.G)
            ie.weight.grad = t.items(t.G)

    # ---- one box, several GPUs: row-sharded tables over NVLink peer memory (whisprrec_b200/sharded.py) ----
    sharded = None

    def shard(self, peers):
        """Distribute the (replicated-at-init) tables over the ranks of `peers`; from here on fit() / evaluate()
        run the sharded kernels.  Every rank must call this with identically initialised parameters."""
        from .. import sharded as S
        self.quiesce()
        t = self.fuse()
        lay = S.ShardLayout(t.n_users, t.n_items, peers.world, peers.rank)
        st = S.ShardedTables(peers, lay, t.D)
        st.load_full(t.users(t.P), t.items(t.P))
        st.M.copy_(lay.shard_of_table(t.M))
        st.V.copy_(lay.shard_of_table(t.V))
        st.step_count = self.optimizer.step_count if self.optimizer is not None else 0
        self.sharded = st
        self._on_sharded()
        return st

    def _on_sharded(self):
        pass

    def sharded_train_step(self, user, pos, neg, B_global, lr, l2, batch=None):
        """This rank's slice of one global batch; returns the batch loss (device view, same on every rank).  batch: the
        whole global batch ([3, B_global] ids, the same on every rank), for models whose step needs more than the
        slice (SGL); the others ignore it."""
        raise NotImplementedError

    def sharded_eval_tables(self):
        """(wr_shards of the table to score, this rank's item rows of it)."""
        st = self.sharded
        return st.T, st.item_rows(st.P)

    def unshard(self):
        """Copy the shards back into the full fused tables (checkpointing, hand-over to single-GPU code)."""
        st, t = self.sharded, self.tables
        u, i = st.gather_full()
        t.users(t.P).copy_(u)
        t.items(t.P).copy_(i)
        st.peers.barrier()

    def build_optimizer(self, name, lr, l2):
        """What BaseRunner._build_optimizer hands back for this model."""
        if name != 'Adam':
            raise NotImplementedError('the fused step implements Adam (the reference default); got ' + name)
        self.fuse()
        return FusedAdam(self, lr, weight_decay=l2)

    def eval_tables(self):
        """(user table, item table) that full-ranking evaluation scores with."""
        self.quiesce()
        t = self.fuse()
        return t.users(t.P), t.items(t.P)

    def _finish_loss(self, t):
        return t.loss[0].detach().as_subclass(FusedLoss)

    def calculate_loss(self, feed_dict):
        pass

    class Dataset(BaseModel.Dataset):
        def _get_feed_dict(self, index):
            """BaseModel.py:152-164."""
            user_id, target_item = self.data['user_id'][index], self.data['item_id'][index]
            if self.phase != 'train' and self.model.test_all:
                neg_items = np.arange(1, self.corpus.n_items)
            else:
                neg_items = self.data['neg_items'][index]
            return {'user_id': user_id, 'pos_item': target_item, 'neg_items': neg_items}

        def _device_cols(self, dev):
            """(user, item) of every row and the train CSR as device tensors, uploaded once."""
            c = getattr(self, '_dev_cols', None)
            if c is None or c[0].device != dev:
                ptr, idx = self.corpus.train_csr()
                if len(idx) == 0:
                    idx = np.zeros(1, dtype=np.int32)
                c = self._dev_cols = (torch.from_numpy(np.asarray(self.data['user_id'], dtype=np.int64)).to(dev),
                                      torch.from_numpy(np.asarray(self.data['item_id'], dtype=np.int64)).to(dev),
                                      torch.from_numpy(np.ascontiguousarray(ptr, dtype=np.int64)).to(dev),
                                      torch.from_numpy(np.ascontiguousarray(idx, dtype=np.int32)).to(dev))
            return c

        def actions_before_epoch(self):
            """BaseModel.py:167-177, bit-exact on NumPy's global stream.

            Training (`BaseRunner.fit`, which fuses the tables first) always takes the device sampler below; the NumPy
            loop after it is what a host-side caller without device tables gets (the CPU tests of the data pipeline).

            The reference draws all N*num_neg candidates in one bulk call and then walks every row in order,
            redrawing (one scalar `randint` each) while the candidate is in the user's train set.  Only rows
            whose candidate was rejected ever touch the stream again, so they are found with one vectorised
            membership test and only those are walked -- in the same order, with the same scalar calls.
            """
            n, num_neg, n_items = len(self), self.model.num_neg, int(self.corpus.n_items)
            self.neg_device = None
            t = getattr(self.model, 'tables', None)
            if t is not None and num_neg == 1 and n_items >= 3 and getattr(self.model, 'device_sampler', True):
                # the same draws on the device (wr_neg_sample_mt19937): NumPy's global state goes in and comes back
                # advanced exactly as the host loop below would leave it
                dev = t.P.device
                cols = self._device_cols(dev)
                self.neg_device = _lib.neg_sample_numpy_stream(cols[0], int(self.corpus.n_users), n_items, cols[2],
                                                               cols[3], t.ws)
                self.data['neg_items'] = self.neg_device.cpu().numpy()
                return
            neg = np.random.randint(1, n_items, size=(n, num_neg))
            ptr, idx = self.corpus.train_csr()
            keys = np.repeat(np.arange(len(ptr) - 1, dtype=np.int64), np.diff(ptr)) * n_items + idx   # sorted
            users = np.asarray(self.data['user_id'], dtype=np.int64)

            def clicked(u, items):
                code = u * n_items + items
                pos = np.searchsorted(keys, code)
                pos[pos >= len(keys)] = len(keys) - 1
                return keys[pos] == code if len(keys) else np.zeros(len(code), dtype=bool)

            bad = clicked(np.repeat(users, num_neg), neg.reshape(-1)).reshape(n, num_neg)
            train_sets = self.corpus.train_clicked_set
            for i in np.nonzero(bad.any(axis=1))[0]:
                seen = train_sets[self.data['user_id'][i]]
                for j in range(num_neg):
                    while neg[i][j] in seen:
                        neg[i][j] = np.random.randint(1, n_items)
            self.data['neg_items'] = neg.reshape(-1)
