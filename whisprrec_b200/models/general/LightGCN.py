"""LightGCN on the fused sm_100a path (reference src/models/general/LightGCN.py).

CMD example (same as the reference):
    python main.py --model_name LightGCN --emb_size 64 --gcn_layers 3 --lr 1e-3 --l2 1e-8 --dataset 'ml-100k'

The adjacency is kept SPARSE (CSR) on the device.  The reference means to do the same but its device test
(`self.device == 'cuda'`, LightGCN.py:114) compares a torch.device with a str, so it always densifies; the
operator is identical, only the order of the row sums differs.
"""
import numpy as np
import torch
import torch.nn as nn

from .. import BaseModel as _base
from ..BaseModel import GeneralModel
from ..init import xavier_uniform_initialization
from ... import _lib


def build_norm_adj_csr(n_users, n_items, train_ptr, train_idx):
    """CSR structure of [[0, R], [R^T, 0]] plus d^-1/2 per node (LightGCN.py:54-97).

    Returns (rowptr int64 [N+1], col int32 [2E], dinv fp32 [N]); rows and columns ascending.  The edge
    weights fl32(fl32(dinv[r]*1)*dinv[c]) are filled on the device by wr_csr_norm_weights.
    dinv = np.power(fp32(deg) + 1e-10, -0.5) is the reference's own NumPy call (:89-93), so its bits match
    the reference on the same host.
    """
    U, I = int(n_users), int(n_items)
    deg_u = np.diff(train_ptr)
    users = np.repeat(np.arange(U, dtype=np.int64), deg_u)
    items = train_idx.astype(np.int64)
    order = np.lexsort((users, items))                       # item-major, users ascending inside an item
    deg_i = np.bincount(items, minlength=I)
    deg = np.concatenate([deg_u, deg_i])
    rowptr = np.zeros(U + I + 1, dtype=np.int64)
    np.cumsum(deg, out=rowptr[1:])
    col = np.concatenate([U + items, users[order]]).astype(np.int32)
    return rowptr, col, reference_dinv(deg)


def reference_dinv(deg):
    """d^-1/2 exactly as LightGCN.py:89-93 computes it: NumPy's fp32 `power` on fp32(deg) + 1e-10 (that routine is not
    correctly rounded, so only the same NumPy call on the same values reproduces the reference bit for bit)."""
    rowsum = np.asarray(deg).astype(np.float32) + 1e-10
    dinv = np.power(rowsum, -0.5).astype(np.float32)
    dinv[np.isinf(dinv)] = 0.
    return dinv


def build_norm_adj_device(n_users, n_items, users, items, ws=None):
    """The graph construction of LightGCN.py:54-97 on the device, for edge lists the host builder cannot hold
    (10^8 - 10^9 edges): wr_csr_build (hand-written radix sort / dedup / row pointers, csrc/csr_build.cu) for the
    structure, the reference's own NumPy call for d^-1/2 (degrees cross the bus once: 4 bytes per node each way),
    wr_csr_norm_weights for the fp32 weights.  users / items: int64 device tensors (duplicate pairs count once).

    Returns (rowptr int64 [N+1], col int32 [nnz], val fp32 [nnz], dinv fp32 [N]) -- bit-identical to
    build_norm_adj_csr + wr_csr_norm_weights on the same pairs."""
    dev = users.device
    ws = _lib.Workspace(dev) if ws is None else ws
    rowptr, col = _lib.csr_build(users, items, int(n_users), int(n_items), ws)
    deg = (rowptr[1:] - rowptr[:-1]).to(torch.int32).cpu().numpy()
    dinv = torch.from_numpy(reference_dinv(deg)).to(dev)
    val = torch.empty(col.numel(), dtype=torch.float32, device=dev)
    _lib.csr_norm_weights(rowptr, col, dinv, val)
    ws.raise_on_status()
    return rowptr, col, val, dinv


class PropagationEngine(object):
    """LightGCN on fused tables: adjacency (device CSR), layer / pool buffers, and the step built from wr_csr_spmm,
    wr_bpr_fwd_bwd and wr_embloss_fwd_bwd.  Used by the model class below and by scripts/bench_lightgcn_scale.py."""

    def __init__(self, tables, rowptr, col, val, rowptr_host, n_layers, reg_weight):
        t = self.tables = tables
        self.L, self.reg_weight = int(n_layers), float(reg_weight)
        self.rowptr, self.col, self.val = rowptr, col, val
        self.plan = _lib.SpmmPlan(rowptr_host, t.D, t.P.device)       # slices of the long (popular-item) rows
        self.pool = torch.empty_like(t.P)            # mean_k E^k
        self.layer = [torch.empty_like(t.P), torch.empty_like(t.P)]
        self.pool_grad = torch.zeros_like(t.P)       # dL/d(pool); re-zeroed by the last backward SpMM
        self.x_rows = _lib.row_map(t.P.shape[0], t.P.device)        # rows of pool_grad a batch touches (large graphs)

    def propagate(self):
        """LightGCN.py:134-148: L SpMMs with the running layer sum (and the final /(L+1)) in their epilogue."""
        t, L = self.tables, self.L
        if L == 0:
            self.pool.copy_(t.P)
            return
        x = t.P
        for k in range(1, L + 1):
            y = self.layer[(k - 1) & 1]
            _lib.csr_spmm(self.rowptr, self.col, self.val, x, Y=y if k < L else None,
                          acc_in=t.P if k == 1 else self.pool, acc_out=self.pool,
                          acc_div=float(L + 1) if k == L else 1.0, plan=self.plan)
            x = y

    def fwd_bwd(self, user, pos, neg, out):
        """LightGCN.py:150-175 and its backward: propagate, BPR on pooled rows, adjoint propagation, EmbLoss.
        The gradient lands in tables.G, the loss in out[0]."""
        t, L = self.tables, self.L
        self.propagate()
        if L == 0:
            _lib.bpr_fwd_bwd(t.users(t.P), t.items(t.P), user, pos, neg, t.users(t.G), t.items(t.G), out, t.ws)
        else:
            g = self.pool_grad
            _lib.bpr_fwd_bwd(t.users(self.pool), t.items(self.pool), user, pos, neg, t.users(g), t.items(g), out,
                             t.ws, grad_scale=1.0 / (L + 1))
            # pool = 1/(L+1) sum_k A^k E0 with A symmetric  =>  dE0 = H_0,  H_L = g,  H_{k-1} = g + A H_k
            h = g
            # g is zero outside the batch's <= 3 B rows: when those are a small part of the table the first adjoint
            # propagation fetches only them (wr_spmm_plan.x_rows) -- on a graph far beyond L2 that is most of its traffic
            sparse = 12 * user.numel() <= t.P.shape[0]
            if sparse:
                _lib.mark_rows(user, pos, neg, t.n_users, t.P.shape[0] - t.n_users, self.x_rows)
            for k in range(1, L + 1):
                last = k == L
                y = t.G if last else self.layer[(k - 1) & 1]
                # the fused re-zeroing of g is only safe when g is not also the SpMM input (L >= 2)
                _lib.csr_spmm(self.rowptr, self.col, self.val, h, Y=y, add=g, zero_add=last and L > 1,
                              plan=self.plan, x_rows=self.x_rows if sparse and k == 1 else None)
                h = y
            if sparse:
                self.x_rows.zero_()
            if L == 1:
                g.zero_()
        _lib.embloss_fwd_bwd(t.users(t.P), t.items(t.P), user, pos, neg, t.users(t.G), t.items(t.G), out, t.ws,
                             self.reg_weight)


class LightGCN(GeneralModel):
    reader = 'BaseReader'
    runner = 'BaseRunner'
    extra_log_args = ['embedding_size', 'gcn_layers', 'reg_weight']

    @staticmethod
    def parse_model_args(parser):
        parser.add_argument('--embedding_size', type=int, default=64, help='Size of embedding vectors.')
        parser.add_argument('--gcn_layers', type=int, default=2, help='Number of LightGCN layers.')
        parser.add_argument('--reg_weight', type=float, default=1e-05, help='The L2 regularization weight.')
        return GeneralModel.parse_model_args(parser)

    def __init__(self, args, corpus):
        super().__init__(args, corpus)
        self.emb_size = args.embedding_size
        self.gcn_layers = args.gcn_layers
        self.n_users = corpus.n_users
        self.n_items = corpus.n_items
        self.reg_weight = float(args.reg_weight)
        # same construction order as LightGCN.py:45-52: the adjacency build draws nothing from torch's RNG
        self.user_embedding = nn.Embedding(self.n_users, self.emb_size)
        self.item_embedding = nn.Embedding(self.n_items, self.emb_size)
        self._adj_host = build_norm_adj_csr(self.n_users, self.n_items, *corpus.train_csr())
        self.apply(xavier_uniform_initialization)
        self._fresh = False          # pooled tables valid for the current parameters?

    def _embedding_pair(self):
        return self.user_embedding, self.item_embedding

    def _on_fused(self):
        t = self.tables
        dev = t.P.device
        rowptr, col, dinv = self._adj_host
        self.adj_rowptr = torch.from_numpy(rowptr).to(dev)
        self.adj_col = torch.from_numpy(col).to(dev)
        self.adj_val = torch.empty(len(col), dtype=torch.float32, device=dev)
        _lib.csr_norm_weights(self.adj_rowptr, self.adj_col, torch.from_numpy(dinv).to(dev), self.adj_val)
        self.engine = PropagationEngine(t, self.adj_rowptr, self.adj_col, self.adj_val, rowptr, self.gcn_layers,
                                        self.reg_weight)
        self._fresh = False

    # buffers of the engine under the names the tests / bench use
    adj_plan = property(lambda self: self.engine.plan)
    pool = property(lambda self: self.engine.pool)
    layer = property(lambda self: self.engine.layer)
    pool_grad = property(lambda self: self.engine.pool_grad)

    @property
    def norm_adj(self):
        """The normalised adjacency as a torch sparse CSR tensor (reference attribute name)."""
        self.fuse()
        n = self.adj_rowptr.numel() - 1
        return torch.sparse_csr_tensor(self.adj_rowptr, self.adj_col.long(), self.adj_val, size=(n, n))

    def get_ego_embeddings(self):
        return self.fuse().P

    def _propagate(self):
        self.fuse()
        self.engine.propagate()

    def forward(self):
        self._propagate()
        t = self.tables
        return t.users(self.pool), t.items(self.pool)

    def predict(self, feed_dict, loss_out=None):
        """LightGCN.py:150-175 and its backward (PropagationEngine.fwd_bwd)."""
        t = self.fuse()
        self._prepare_grads()
        out = t.loss if loss_out is None else loss_out
        self.engine.fwd_bwd(feed_dict['user_id'], feed_dict['pos_item'], feed_dict['neg_items'], out)
        return out[0].detach().as_subclass(_base.FusedLoss)

    def eval_tables(self):
        return self.forward()

    def _on_sharded(self):
        from ... import sharded as S
        rowptr, col, dinv = self._adj_host
        self.sharded_gcn = S.ShardedLightGCN(self.sharded, rowptr, col, dinv, self.gcn_layers, self.reg_weight)

    def sharded_train_step(self, user, pos, neg, B_global, lr, l2, batch=None):
        return self.sharded_gcn.step(user, pos, neg, B_global, lr, l2)

    def sharded_eval_tables(self):
        g, st = self.sharded_gcn, self.sharded
        g.propagate()
        return g.pool_T, st.item_rows(g.pool)

    def full_predict(self, feed_dict):
        """LightGCN.py:177-187 (compatibility API, dense output; the runner uses the fused rank kernel)."""
        ue, ie = self.forward()
        user = feed_dict['user_id']
        pos = feed_dict.get('pos_item', torch.zeros_like(user))
        dev = ue.device
        if not hasattr(self, '_no_hist'):
            self._no_hist = (torch.zeros(self.user_num + 1, dtype=torch.int64, device=dev),
                             torch.zeros(1, dtype=torch.int32, device=dev))
        return _lib.eval_rank_topk(ue, ie, user, pos, self._no_hist[0], self._no_hist[1], self.tables.ws,
                                   scores=True)[4]
