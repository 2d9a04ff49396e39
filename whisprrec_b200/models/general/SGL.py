"""SGL on the fused sm_100a path (reference src/models/general/SGL.py, SIGIR '21) -- SURVEY.md section 8 f-3.

CMD example (same as the reference):
    python main.py --model_name SGL --emb_size 64 --gcn_layers 2 --lr 1e-3 --l2 0 --dataset 'ml-100k'

One training step (SGL.py:233-246 and its backward) is, on the device:
  three LightGCN propagations of the same ego table -- the full graph and the two edge-dropout views of the epoch
  (wr_csr_spmm with the layer mean in the epilogue), the sum-form BPR term on the main graph's pooled rows
  (wr_bpr_logsig_sum_fwd_bwd), InfoNCE between the views for the batch's users and positive items
  (wr_infonce_fwd_bwd: normalisation, the [B, N] contraction and its backward), the three adjoint propagations (the views
  are not symmetric: their transposed CSRs are built with them), EmbLoss on the ego rows (wr_embloss_fwd_bwd); the
  gradient lands in tables.G and the optimiser is the fused Adam sweep, as for LightGCN.
The views are redrawn every epoch from Python's global `random` stream exactly as utils/augmentor.py:77-111 does
(wr_pyrandom_sample) and assembled on the device (wr_subgraph_csr: radix sort of the kept edges into CSR order, and
into the transposed order), so they are bit-identical to the reference's.
"""
import torch
import torch.nn as nn

from .. import BaseModel as _base
from ..BaseModel import GeneralModel
from ..init import xavier_uniform_initialization
from .LightGCN import build_norm_adj_csr
from ... import _lib
from ...utils import graph_views


class _Graph(object):
    """A normalised adjacency on the device: CSR, its long-row plan, and (views only) the CSR of its transpose."""

    def __init__(self, rowptr, col, val, D, transpose=None):
        self.rowptr, self.col, self.val = rowptr, col, val
        self.plan = _lib.SpmmPlan(rowptr.cpu().numpy(), D, rowptr.device)
        self.T = self if transpose is None else _Graph(*transpose, D=D)      # symmetric: its own transpose


class SGL(GeneralModel):
    reader = 'BaseReader'
    runner = 'BaseRunner'
    extra_log_args = ['embedding_size', 'gcn_layers', 'reg_weight', 'type', 'ssl_tau', 'ssl_weight', 'drop_ratio']

    @staticmethod
    def parse_model_args(parser):
        parser.add_argument('--embedding_size', type=int, default=64, help='Size of embedding vectors.')
        parser.add_argument('--gcn_layers', type=int, default=2, help='Number of SGL layers.')
        parser.add_argument('--type', type=str, default='ED',
                            help="The type to generate views. Range in ['ED', 'ND', 'RW'].")
        parser.add_argument('--reg_weight', type=float, default=1e-4, help='The L2 regularization weight.')
        parser.add_argument('--ssl_tau', type=float, default=0.1, help='The temperature in softmax.')
        parser.add_argument('--ssl_weight', type=float, default=0.05,
                            help='The hyperparameter to control the strengths of SSL.')
        parser.add_argument('--drop_ratio', type=float, default=0.1, help='The dropout ratio.')
        return GeneralModel.parse_model_args(parser)

    def __init__(self, args, corpus):
        super().__init__(args, corpus)
        self.n_users, self.n_items = corpus.n_users, corpus.n_items
        self.emb_size, self.gcn_layers = args.embedding_size, int(args.gcn_layers)
        self.reg_weight, self.type = float(args.reg_weight), str(args.type)
        self.ssl_weight, self.ssl_tau, self.drop_ratio = float(args.ssl_weight), float(args.ssl_tau), float(args.drop_ratio)
        if self.type != 'ED':
            raise NotImplementedError("SGL views: only edge dropout ('ED', the reference default) is implemented")
        if self.gcn_layers < 1:
            raise NotImplementedError('SGL needs at least one propagation layer')
        # same construction order as SGL.py:57-65 (the adjacency build draws nothing from torch's generator)
        self.user_embedding = nn.Embedding(self.n_users, self.emb_size)
        self.item_embedding = nn.Embedding(self.n_items, self.emb_size)
        self._adj_host = build_norm_adj_csr(self.n_users, self.n_items, *corpus.train_csr())
        self.apply(xavier_uniform_initialization)
        self.sub_graphs = None

    def _embedding_pair(self):
        return self.user_embedding, self.item_embedding

    def _on_fused(self):
        t = self.tables
        dev = t.P.device
        rowptr, col, dinv = self._adj_host
        d_rowptr, d_col = torch.from_numpy(rowptr).to(dev), torch.from_numpy(col).to(dev)
        val = torch.empty(len(col), dtype=torch.float32, device=dev)
        _lib.csr_norm_weights(d_rowptr, d_col, torch.from_numpy(dinv).to(dev), val)
        self.train_graph = _Graph(d_rowptr, d_col, val, t.D)
        self.pool = [torch.empty_like(t.P) for _ in range(3)]           # pooled tables: main graph, view 1, view 2
        self.pool_grad = [torch.zeros_like(t.P) for _ in range(3)]
        self.layer = [torch.empty_like(t.P), torch.empty_like(t.P)]
        self._scratch = None
        self.sub_graphs = None

    def graph_construction(self):
        """SGL.py:67-79: the two augmented views of this epoch (edge dropout on Python's global random stream).  Sharded,
        every rank draws the same two views (its Python stream is seeded as every other rank's) and keeps its rows."""
        t = self.fuse()
        g = self.train_graph
        views = []
        for _ in range(2):
            fwd, tr = graph_views.edge_dropout_view_device(g.rowptr, g.col, self.drop_ratio, t.ws)
            views.append((fwd, tr) if self.sharded is not None else _Graph(*fwd, D=t.D, transpose=tr))
        if self.sharded is not None:
            self.sharded_sgl.set_views(views)
            return
        self.sub_graphs = views

    # ---- propagation -----------------------------------------------------------------------------------------------
    def _propagate(self, g, pool):
        """SGL.py:148-163: pool = mean(E0, A E0, ..., A^L E0)."""
        t, L = self.tables, self.gcn_layers
        x = t.P
        for k in range(1, L + 1):
            y = self.layer[(k - 1) & 1]
            _lib.csr_spmm(g.rowptr, g.col, g.val, x, Y=y if k < L else None, acc_in=t.P if k == 1 else pool,
                          acc_out=pool, acc_div=float(L + 1) if k == L else 1.0, plan=g.plan)
            x = y

    def _adjoint(self, g, grad, first):
        """dE0 += H_0 with H_L = grad, H_{k-1} = grad + A^T H_k (grad already carries the 1 / (L + 1) of the mean)."""
        t, L = self.tables, self.gcn_layers
        gt = g.T
        h = grad
        for k in range(1, L + 1):
            last = k == L
            kw = dict(add=grad, zero_add=last and L > 1, plan=gt.plan)
            if not last:
                y = self.layer[(k - 1) & 1]
                _lib.csr_spmm(gt.rowptr, gt.col, gt.val, h, Y=y, **kw)
                h = y
            elif first:
                _lib.csr_spmm(gt.rowptr, gt.col, gt.val, h, Y=t.G, **kw)            # tables.G is zero: overwrite
            else:
                _lib.csr_spmm(gt.rowptr, gt.col, gt.val, h, acc_in=t.G, acc_out=t.G, acc_div=1.0, **kw)
        if L == 1:
            grad.zero_()

    def forward(self, graph=None):
        t = self.fuse()
        self._propagate(self.train_graph if graph is None else graph, self.pool[0])
        return t.users(self.pool[0]), t.items(self.pool[0])

    def predict(self, feed_dict, loss_out=None):
        """SGL.py:233-246 and its backward; the gradient lands in tables.G, the loss in out[0]."""
        t = self.fuse()
        if self.sub_graphs is None:
            self.graph_construction()
        self._prepare_grads()
        out = t.loss if loss_out is None else loss_out
        user, pos, neg = feed_dict['user_id'], feed_dict['pos_item'], feed_dict['neg_items']
        L = self.gcn_layers
        graphs = [self.train_graph] + self.sub_graphs
        for g, pool in zip(graphs, self.pool):
            self._propagate(g, pool)
        scale = 1.0 / (L + 1)
        pm, gm = self.pool[0], self.pool_grad[0]
        _lib.bpr_logsig_sum_fwd_bwd(t.users(pm), t.items(pm), user, pos, neg, t.users(gm), t.items(gm), out, t.ws,
                                    grad_scale=scale)
        p1, p2, g1, g2 = self.pool[1], self.pool[2], self.pool_grad[1], self.pool_grad[2]
        self._scratch = _lib.infonce_fwd_bwd(t.users(p1), t.users(p2), user, self.ssl_tau, self.ssl_weight, scale,
                                             t.users(g1), t.users(g2), out, t.ws, self._scratch)
        self._scratch = _lib.infonce_fwd_bwd(t.items(p1), t.items(p2), pos, self.ssl_tau, self.ssl_weight, scale,
                                             t.items(g1), t.items(g2), out, t.ws, self._scratch)
        for n, (g, grad) in enumerate(zip(graphs, self.pool_grad)):
            self._adjoint(g, grad, first=n == 0)
        _lib.embloss_fwd_bwd(t.users(t.P), t.items(t.P), user, pos, neg, t.users(t.G), t.items(t.G), out, t.ws,
                             self.reg_weight)
        return out[0].detach().as_subclass(_base.FusedLoss)

    def eval_tables(self):
        return self.forward()

    def full_predict(self, feed_dict):
        """SGL.py:248-254 (compatibility API, dense output; the runner uses the fused rank kernel)."""
        ue, ie = self.forward()
        user = feed_dict['user_id']
        pos = feed_dict.get('pos_item', torch.zeros_like(user))
        dev = ue.device
        if not hasattr(self, '_no_hist'):
            self._no_hist = (torch.zeros(self.user_num + 1, dtype=torch.int64, device=dev),
                             torch.zeros(1, dtype=torch.int32, device=dev))
        return _lib.eval_rank_topk(ue, ie, user, pos, self._no_hist[0], self._no_hist[1], self.tables.ws, scores=True)[4]

    def _on_sharded(self):
        from ... import sharded as S
        rowptr, col, dinv = self._adj_host
        self.sharded_sgl = S.ShardedSGL(self.sharded, rowptr, col, dinv, self.gcn_layers, self.reg_weight, self.ssl_tau,
                                        self.ssl_weight)

    def sharded_train_step(self, user, pos, neg, B_global, lr, l2, batch=None):
        """batch: the global batch ([3, B_global] user / positive / negative ids, the same on every rank) -- the sharded
        InfoNCE runs every rank's table rows against all of it."""
        if batch is None:
            raise ValueError('the sharded SGL step needs the global batch (batch=[3, B_global] ids)')
        g = self.sharded_sgl
        if g.views is None:
            self.graph_construction()
        return g.step(user, pos, neg, B_global, lr, l2, batch[0], batch[1])

    def sharded_eval_tables(self):
        g, st = self.sharded_sgl, self.sharded
        g.propagate()
        return g.pool_T, st.item_rows(g.pool)

    class Dataset(GeneralModel.Dataset):
        def actions_before_epoch(self):
            """SGL.py:260-262: negatives first (NumPy's stream), then the epoch's views (Python's random stream)."""
            super().actions_before_epoch()
            self.model.graph_construction()
