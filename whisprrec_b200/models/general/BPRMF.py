"""BPRMF on the fused sm_100a path (reference src/models/general/BPRMF.py).

CMD example (same as the reference):
    python main.py --model_name BPRMF --emb_size 64 --lr 1e-3 --l2 1e-6 --dataset 'ml-100k'
"""
import torch
import torch.nn as nn

from .. import BaseModel as _base
from ..BaseModel import GeneralModel
from ..init import xavier_normal_initialization
from ... import _lib


class BPRMF(GeneralModel):
    reader = 'BaseReader'
    runner = 'BaseRunner'
    extra_log_args = ['embedding_size']

    @staticmethod
    def parse_model_args(parser):
        parser.add_argument('--embedding_size', type=int, default=64, help='Size of embedding vectors.')
        return GeneralModel.parse_model_args(parser)

    def __init__(self, args, corpus):
        super().__init__(args, corpus)
        self.emb_size = args.embedding_size
        # Built on the CPU in this order so the torch generator is consumed exactly as BPRMF.py:35-40 does
        # (normal_ x2 inside nn.Embedding, then xavier_normal_ x2): the initial weights are bit-identical.
        self.user_embeddings = nn.Embedding(self.user_num, self.emb_size)
        self.item_embeddings = nn.Embedding(self.item_num, self.emb_size)
        self.apply(xavier_normal_initialization)

    def _embedding_pair(self):
        return self.user_embeddings, self.item_embeddings

    def get_user_embedding(self, user):
        t = self.fuse()
        return _lib.gather_rows(t.users(t.P), user, t.ws)

    def get_item_embedding(self, item):
        t = self.fuse()
        return _lib.gather_rows(t.items(t.P), item, t.ws)

    def forward(self, user, item):
        return self.get_user_embedding(user), self.get_item_embedding(item)

    def quiesce(self):
        """Host-fed training keeps the Adam moments in the SMs' shared memory while its kernel is resident
        (train_step_host); anything else that touches the tables closes it first."""
        ctx = getattr(self, '_host_ctx', None)
        if ctx is not None:
            ctx.sync()

    def predict(self, feed_dict, loss_out=None):
        """BPRMF.py:69-80 + the backward of BaseRunner.py:198 in one launch; gradient lands in tables.G."""
        self.quiesce()
        t = self.fuse()
        self._prepare_grads()
        out = t.loss if loss_out is None else loss_out
        _lib.bpr_fwd_bwd(t.users(t.P), t.items(t.P), feed_dict['user_id'], feed_dict['pos_item'],
                         feed_dict['neg_items'], t.users(t.G), t.items(t.G), out, t.ws)
        return out[0].detach().as_subclass(_base.FusedLoss)

    def train_step(self, feed_dict, loss_out=None):
        """One whole iteration of BaseRunner.fit (BaseRunner.py:196-199: zero_grad, predict, backward,
        optimizer.step) as a single wr_bprmf_step call; the loss stays on the device."""
        self.quiesce()
        t = self.fuse()
        opt = self.optimizer
        out = t.loss if loss_out is None else loss_out
        opt.step_count += 1
        if t.P.numel() > _lib.FUSED_STEP_MAX_ELEMS and getattr(t, 'touched', None) is None:
            t.touched = _lib.row_map(t.P.shape[0], t.P.device)      # streaming path: skip untouched gradient rows
        _lib.bprmf_step(t.P, t.M, t.V, t.G, feed_dict['user_id'], feed_dict['pos_item'], feed_dict['neg_items'],
                        t.n_users, opt.step_count, opt.lr, opt.weight_decay, out, t.ws, beta1=opt.betas[0],
                        beta2=opt.betas[1], eps=opt.eps, touched=getattr(t, 'touched', None))
        return out[0].detach().as_subclass(_base.FusedLoss)

    def train_epoch(self, ids, batch_size, losses):
        """All steps of an epoch (BaseRunner.py:194-200 for every batch) from one C call; `ids` is the epoch's int64
        [3, N] device tensor in batch order, `losses` a device float per step.  Cache-sized tables: ONE resident
        launch for the whole epoch (csrc/epoch_kernel.cu)."""
        self.quiesce()
        t = self.fuse()
        opt = self.optimizer
        steps = _lib.bprmf_epoch(t.P, t.M, t.V, t.G, ids, batch_size, t.n_users, opt.step_count, opt.lr,
                                 opt.weight_decay, losses, t.ws, beta1=opt.betas[0], beta2=opt.betas[1], eps=opt.eps)
        opt.step_count += steps
        return steps

    def train_step_host(self, host_ids, wait=1):
        """The same iteration fed from the host: `host_ids` is an int64 [3, B] host tensor holding the batch's
        user / positive / negative ids (what collate_batch produces, BaseModel.py:96-127).  Covers
        utils.batch_to_gpu (utils.py:33-37), the step and `loss.detach().cpu()` (BaseRunner.py:200) in one C call
        (wr_bprmf_ctx_step) with no launch, copy-engine hop or stream synchronisation per step: a kernel that stays
        resident between calls pulls the ids out of pinned host memory and drops the loss into mapped host memory.
        Pinned tensors are read in place (leave them alone until the step is complete); pageable ones are collated
        into the context's pinned ring first.  wait=1: returns when the step is complete; wait=2: as soon as the loss
        is out; wait=0: at once (up to 16 steps in flight; `host_step_loss(k)` collects the k-th step's loss).
        Returns the batch loss as a float."""
        ctx = getattr(self, '_host_ctx', None)
        opt = self.optimizer
        if ctx is None or ctx._keep[0] is not self.tables.P:       # first call, or the tables were re-fused
            t = self.fuse()
            ctx = self._host_ctx = _lib.BprmfContext(t.P, t.M, t.V, t.G, t.n_users, opt.lr, opt.weight_decay, t.ws,
                                                     beta1=opt.betas[0], beta2=opt.betas[1], eps=opt.eps)
        if host_ids.dtype != torch.int64 or host_ids.dim() != 2 or host_ids.shape[0] != 3 or \
                not host_ids.is_contiguous() or host_ids.is_cuda:
            raise _lib.WhisprError('host_ids must be a contiguous int64 [3, B] host tensor')
        opt.step_count += 1
        return ctx.step(host_ids.data_ptr(), host_ids.shape[1], opt.step_count, wait)

    def host_step_loss(self, k, wait=1):
        """Loss of the k-th train_step_host call of this model (0-based), for calls made with wait=0."""
        return self._host_ctx.wait(k, wait)

    def sharded_train_step(self, user, pos, neg, B_global, lr, l2, batch=None):
        from ... import sharded as S
        return S.bprmf_step(self.sharded, user, pos, neg, B_global, lr, l2)

    def full_predict(self, feed_dict):
        """BPRMF.py:82-91: the dense [B, n_items] score matrix (compatibility API; the runner's evaluation
        uses the fused rank kernel and never materialises it)."""
        self.quiesce()
        t = self.fuse()
        user = feed_dict['user_id']
        pos = feed_dict.get('pos_item', torch.zeros_like(user))
        corpus_hist = self._empty_history(t)
        return _lib.eval_rank_topk(t.users(t.P), t.items(t.P), user, pos, corpus_hist[0], corpus_hist[1], t.ws,
                                   scores=True)[4]

    def _empty_history(self, t):
        if not hasattr(self, '_no_hist'):
            dev = t.P.device
            self._no_hist = (torch.zeros(self.user_num + 1, dtype=torch.int64, device=dev),
                             torch.zeros(1, dtype=torch.int32, device=dev))
        return self._no_hist
