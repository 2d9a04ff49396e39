"""Row-sharded BPRMF / LightGCN over the GPUs of one box (SURVEY.md section 8e; include/whisprrec_b200.h,
"one 8 x B200 box").

One process per GPU (torchrun).  `torch.distributed` is only the rendezvous (exchange of the cudaIpc handles) and
the small evaluation collectives; the training step has NO collective call: every rank maps every other rank's
tables (NVLink 5 / NVSwitch peer memory) and the kernels read remote embedding rows and reduce remote gradient rows
themselves, meeting at wr_peer_barrier.

`ShardLayout` is pure host arithmetic (tested on the CPU, also under gloo with world_size 2); `PeerGroup`,
`ShardedTables` and the step / evaluation drivers need one GPU per rank.
"""
import ctypes
import os

import numpy as np
import torch

from . import _lib


class ShardLayout(object):
    """user u -> rank u % world, local row u // world;  item i -> rank i % world, local row rows_u_local + i // world.

    A rank's shard is one [n_local, D] table: its user rows first (padded to rows_u_local = ceil(n_users / world)),
    then its item rows (padded to rows_i_local).  LightGCN node n is user n (n < n_users) or item n - n_users.
    """

    def __init__(self, n_users, n_items, world, rank):
        if not (1 <= world <= _lib.MAX_WORLD and 0 <= rank < world):
            raise ValueError('world must be in [1, %d] and rank in [0, world)' % _lib.MAX_WORLD)
        self.n_users, self.n_items, self.world, self.rank = int(n_users), int(n_items), int(world), int(rank)
        self.rows_u_local = (self.n_users + world - 1) // world
        self.rows_i_local = (self.n_items + world - 1) // world
        self.n_local = self.rows_u_local + self.rows_i_local

    # ---- ownership ----
    def local_users(self, rank=None):
        return np.arange(self.rank if rank is None else rank, self.n_users, self.world, dtype=np.int64)

    def local_items(self, rank=None):
        return np.arange(self.rank if rank is None else rank, self.n_items, self.world, dtype=np.int64)

    def local_nodes(self, rank=None):
        """Global node id of every local row (-1 for the padding rows)."""
        out = np.full(self.n_local, -1, dtype=np.int64)
        u, i = self.local_users(rank), self.local_items(rank)
        out[:len(u)] = u
        out[self.rows_u_local:self.rows_u_local + len(i)] = self.n_users + i
        return out

    def shard_of_table(self, full, rank=None):
        """The [n_local, D] shard of a full [n_users + n_items, D] host / device table (padding rows zero)."""
        nodes = self.local_nodes(rank)
        out = full.new_zeros((self.n_local, full.shape[1])) if torch.is_tensor(full) else \
            np.zeros((self.n_local, full.shape[1]), dtype=full.dtype)
        ok = nodes >= 0
        if torch.is_tensor(full):
            out[torch.from_numpy(np.nonzero(ok)[0]).to(full.device)] = full[torch.from_numpy(nodes[ok]).to(full.device)]
        else:
            out[ok] = full[nodes[ok]]
        return out

    # ---- the batch ----
    def batch_slice(self, n, rank=None):
        """Contiguous slice [lo, hi) of a global batch of n rows that a rank processes (sizes differ by <= 1)."""
        r = self.rank if rank is None else rank
        base, rem = divmod(int(n), self.world)
        lo = r * base + min(r, rem)
        return lo, lo + base + (1 if r < rem else 0)

    # ---- evaluation ----
    def localise_history(self, hist_ptr, hist_idx, rank=None):
        """Per-user history CSR restricted to one item shard, as ascending LOCAL item indices."""
        r = self.rank if rank is None else rank
        hist_ptr, hist_idx = np.asarray(hist_ptr, dtype=np.int64), np.asarray(hist_idx, dtype=np.int64)
        nnz = int(hist_ptr[-1])
        idx = hist_idx[:nnz]
        mine = (idx % self.world) == r
        users = np.repeat(np.arange(len(hist_ptr) - 1, dtype=np.int64), np.diff(hist_ptr))
        counts = np.bincount(users[mine], minlength=len(hist_ptr) - 1)
        ptr = np.zeros(len(hist_ptr), dtype=np.int64)
        np.cumsum(counts, out=ptr[1:])
        local = (idx[mine] // self.world).astype(np.int32)
        if len(local) == 0:
            local = np.zeros(1, dtype=np.int32)
        return ptr, local

    def item_local_index(self, items, rank=None):
        """Local index of each global item id on one shard, -1 where another shard owns it (NumPy or torch)."""
        r = self.rank if rank is None else rank
        mine = (items % self.world) == r
        if torch.is_tensor(items):
            return torch.where(mine, torch.div(items, self.world, rounding_mode='floor'), torch.full_like(items, -1))
        return np.where(mine, items // self.world, -1)

    def item_global_index(self, local, rank=None):
        """Global item id of a shard's local item indices (negative = empty slot, kept)."""
        r = self.rank if rank is None else rank
        if torch.is_tensor(local):
            return torch.where(local >= 0, local * self.world + r, local)
        return np.where(local >= 0, local * self.world + r, local)

    # ---- LightGCN ----
    def local_adjacency(self, rowptr, col, dinv=None, rank=None):
        """This rank's rows of the global node CSR, in local row order; column ids stay GLOBAL node ids.

        Returns (rowptr_local int64 [n_local + 1], col_local int32, src_edge int64) where src_edge maps every local
        edge to its position in the global `col` (so weights computed once globally can be sliced)."""
        nodes = self.local_nodes(rank)
        rowptr = np.asarray(rowptr, dtype=np.int64)
        deg = np.where(nodes >= 0, rowptr[np.maximum(nodes, 0) + 1] - rowptr[np.maximum(nodes, 0)], 0)
        lptr = np.zeros(self.n_local + 1, dtype=np.int64)
        np.cumsum(deg, out=lptr[1:])
        total = int(lptr[-1])
        row_of_edge = np.repeat(np.arange(self.n_local, dtype=np.int64), deg)
        src = rowptr[np.maximum(nodes, 0)][row_of_edge] + (np.arange(total, dtype=np.int64) - lptr[row_of_edge])
        return lptr, np.asarray(col)[src].astype(np.int32), src


def combine_shard_ranks(local_ranks):
    """global rank = 1 + sum over shards of (rank_shard - 1); `local_ranks`: iterable of integer arrays / tensors."""
    total = None
    for r in local_ranks:
        total = (r - 1) if total is None else total + (r - 1)
    return total + 1


class PeerGroup(object):
    """The ranks of one box with every rank's peer blocks mapped into every process."""

    def __init__(self, device, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        if self.world > _lib.MAX_WORLD:
            raise _lib.WhisprError('at most %d ranks (one box)' % _lib.MAX_WORLD)
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise _lib.WhisprError('PeerGroup needs a CUDA device per rank (no CPU fallback)')
        self._blocks = []
        self.epoch = 0
        sig_bytes = 4 * _lib.MAX_WORLD + 4 * 2 * _lib.MAX_WORLD * _lib.PEER_VALUES
        self._sig, self._sig_ptrs = self.alloc_bytes((sig_bytes + 255) // 256 * 256)
        self.flag_ptrs = list(self._sig_ptrs)
        self.slot_ptrs = [p + 4 * _lib.MAX_WORLD for p in self._sig_ptrs]
        self.ws = _lib.Workspace(self.device)      # receives WR_STATUS_PEER_TIMEOUT if a peer never arrives
        self._values = torch.zeros(_lib.PEER_VALUES, dtype=torch.float32, device=self.device)
        self.sums = torch.zeros(_lib.PEER_VALUES, dtype=torch.float32, device=self.device)
        self.host_sync()

    def alloc_bytes(self, nbytes):
        """Symmetric allocation: (this rank's PeerBlock, [base pointer of every rank's block as mapped here])."""
        block = _lib.PeerBlock(nbytes, self.device)
        handles = [None] * self.world
        self.dist.all_gather_object(handles, block.handle(), group=self.group)
        ptrs = [block.ptr if g == self.rank else block.open_peer(handles[g]) for g in range(self.world)]
        self._blocks.append(block)
        return block, ptrs

    def alloc(self, shape, dtype=torch.float32):
        n = 1
        for d in shape:
            n *= int(d)
        nbytes = max(256, (n * torch.empty((), dtype=dtype).element_size() + 255) // 256 * 256)
        block, ptrs = self.alloc_bytes(nbytes)
        return block.tensor(0, shape, dtype), ptrs

    def host_sync(self):
        """Host-side rendezvous (set-up and tear-down only): device work done, then a process-group barrier."""
        torch.cuda.synchronize(self.device)
        self.dist.barrier(group=self.group)

    def barrier(self, values=None):
        """Device-side barrier on the current stream; optionally sums up to 4 floats across the ranks (returns a view
        of the result, valid until the next barrier with values)."""
        self.epoch += 1
        if values is None:
            _lib.peer_barrier(self.flag_ptrs, self.slot_ptrs, self.world, self.rank, self.epoch, ws=self.ws)
            return None
        n = values.numel()
        _lib.peer_barrier(self.flag_ptrs, self.slot_ptrs, self.world, self.rank, self.epoch, values, self.sums[:n],
                          ws=self.ws)
        return self.sums[:n]

    def close(self):
        self.host_sync()
        self.ws.raise_on_status()
        for b in self._blocks:
            b.close()
        self._blocks = []


class ShardedTables(object):
    """P / M / V / G shards of one rank plus the `wr_shards` descriptors of every symmetric table."""

    def __init__(self, peers, layout, D):
        self.peers, self.layout, self.D = peers, layout, int(D)
        self.P, self.T = self.symmetric()
        self.G, self.Gd = self.symmetric()
        dev = peers.device
        self.M = torch.zeros((layout.n_local, self.D), dtype=torch.float32, device=dev)
        self.V = torch.zeros_like(self.M)
        self.ws = _lib.Workspace(dev)
        self.loss_part = torch.zeros(_lib.PEER_VALUES, dtype=torch.float32, device=dev)
        self.loss = torch.zeros(1, dtype=torch.float32, device=dev)
        self.step_count = 0
        # synchronisation words of the single-launch step: [2][8] uint32 flags, then [2][8] float loss slots
        _, sync_ptrs = peers.alloc_bytes(256)
        self.step_flag_ptrs = list(sync_ptrs)
        self.step_slot_ptrs = [p + 4 * 2 * _lib.MAX_WORLD for p in sync_ptrs]
        self.single_launch = _lib.bprmf_step_sharded_supported(layout.n_local, self.D)
        self._sync_epoch = 0           # last epoch the single-launch step has used on this table set

    def inbox(self, B_global):
        """Symmetric gradient inbox for the staged scatter: per sender 3 x (largest per-rank batch) row slots."""
        lay = self.layout
        cap = 3 * ((int(B_global) + lay.world - 1) // lay.world)
        box = getattr(self, '_inbox', None)
        if box is None or box['cap'] < cap:
            rows, row_ptrs = self.peers.alloc((lay.world, cap, self.D))
            idx, idx_ptrs = self.peers.alloc((lay.world, cap), dtype=torch.int32)
            box = self._inbox = {'cap': cap, 'rows': rows, 'idx': idx, 'row_ptrs': row_ptrs, 'idx_ptrs': idx_ptrs}
            self.peers.host_sync()
        return box

    def exchange(self, B_global):
        """Symmetric buffers of the row exchange (wr_xchg_*): request lists and counts at the owners, receive buffers
        at the requesters; sized for 3 x the largest per-rank slice of a batch of B_global rows."""
        lay = self.layout
        cap = 3 * ((int(B_global) + lay.world - 1) // lay.world)
        x = getattr(self, '_xchg', None)
        if x is None or x['cap'] < cap:
            dev = self.peers.device
            req, req_ptrs = self.peers.alloc((lay.world, cap), dtype=torch.int32)
            cnt, cnt_ptrs = self.peers.alloc((64,), dtype=torch.int32)
            recv, recv_ptrs = self.peers.alloc((lay.world, cap, self.D))
            x = self._xchg = {'cap': cap, 'req': req, 'req_ptrs': req_ptrs, 'cnt': cnt, 'cnt_ptrs': cnt_ptrs,
                              'recv': recv, 'recv_ptrs': recv_ptrs,
                              'cnt_local': torch.zeros(64, dtype=torch.int32, device=dev),
                              'where': torch.zeros(cap, dtype=torch.int32, device=dev)}
            self.peers.host_sync()
        return x

    def fetch_rows(self, x, table_local, user, pos, neg):
        """Steps 1 and 2 of the exchange: afterwards x['recv'][x['where'][3 b + role]] is the row of batch entry b."""
        lay = self.layout
        _lib.xchg_request(user, pos, neg, lay.n_users, lay.n_items, lay.world, lay.rank, x['req_ptrs'], x['cnt_ptrs'],
                          x['cap'], x['cnt_local'], x['where'], self.ws)
        self.peers.barrier()
        _lib.xchg_serve(table_local, lay.world, lay.rank, x['req'], x['cnt'], x['cap'], x['recv_ptrs'])
        self.peers.barrier()

    def symmetric(self):
        """A zeroed [n_local, D] fp32 table on every rank -> (local tensor, wr_shards describing all of them)."""
        lay = self.layout
        t, ptrs = self.peers.alloc((lay.n_local, self.D))
        s = _lib.ShardsStruct()
        for g in range(lay.world):
            s.base[g] = ptrs[g]
        s.world, s.rank, s.n_users, s.n_items = lay.world, lay.rank, lay.n_users, lay.n_items
        s.rows_u_local, s.rows_i_local = lay.rows_u_local, lay.rows_i_local
        return t, s

    def load_full(self, full_user, full_item):
        """Take this rank's rows of the full (replicated-at-init) tables."""
        full = torch.cat([full_user, full_item]).to(self.peers.device)
        self.P.copy_(self.layout.shard_of_table(full))
        self.peers.host_sync()

    def gather_full(self, shards=None):
        """Full [n_users, D], [n_items, D] copies of a sharded table (checkpointing / tests)."""
        lay = self.layout
        s = self.T if shards is None else shards
        dev = self.peers.device
        self.peers.barrier()           # every rank's stream has finished writing its rows (single-launch steps
        #                                only tell the NEXT step's kernel, not other readers)
        u = _lib.gather_rows_sharded(s, 0, torch.arange(lay.n_users, device=dev), self.D, self.ws)
        i = _lib.gather_rows_sharded(s, 1, torch.arange(lay.n_items, device=dev), self.D, self.ws)
        return u, i

    def item_rows(self, t):
        lay = self.layout
        return t[lay.rows_u_local:lay.rows_u_local + len(lay.local_items())]

    def adam(self, lr, l2, betas=(0.9, 0.999), eps=1e-8, touched=None):
        self.step_count += 1
        if touched is not None:
            _lib.adam_l2_sweep_marked(self.P, self.M, self.V, self.G, touched, self.step_count, lr, l2, betas[0],
                                      betas[1], eps)
            return
        _lib.adam_l2_sweep(self.P, self.M, self.V, self.G, self.step_count, lr, l2, betas[0], betas[1], eps)

    def settle(self):
        """Meet the other ranks if the last step left without a closing barrier (the exchange protocol does)."""
        if getattr(self, '_unsettled', False):
            self._unsettled = False
            self.peers.barrier()

    def row_map(self):
        """Bitmap over this rank's rows for the row-marked sweep (wr_inbox_scatter_marked sets, the sweep clears)."""
        if getattr(self, '_row_map', None) is None:
            self._row_map = _lib.row_map(self.layout.n_local, self.peers.device)
        return self._row_map


def bprmf_step(tabs, user, pos, neg, B_global, lr, l2):
    """One BPRMF iteration on this rank's slice (user, pos, neg) of a global batch of B_global rows.

    Cache-sized shards: wr_bprmf_step_sharded, one cooperative launch per rank.  Larger ones:
    fwd+bwd with remote gathers / remote REDs -> barrier (all gradient rows have landed; carries the loss) ->
    Adam+L2 over the local shard -> barrier (parameters final before anyone gathers again).
    Returns the batch loss (device scalar view, identical on every rank)."""
    if tabs.single_launch:
        # cache-sized shards: one cooperative launch, both cross-GPU meeting points inside the kernel
        tabs.settle()
        tabs.step_count += 1
        tabs._sync_epoch += 1
        _lib.bprmf_step_sharded(tabs.T, tabs.Gd, tabs.M, tabs.V, user, pos, neg, B_global, tabs.D, tabs.step_count,
                                lr, l2, tabs.step_flag_ptrs, tabs.step_slot_ptrs, tabs.loss, tabs.ws,
                                epoch=tabs._sync_epoch)
        return tabs.loss
    # decided from values every rank shares (slices of one batch differ by a row: a per-rank test could split the ranks
    # between the two protocols, and the staged one allocates collectively)
    per_rank = (int(B_global) + tabs.layout.world - 1) // tabs.layout.world
    staged = tabs.layout.world > 1 and per_rank >= 8192 and tabs.D in (16, 32, 64, 128, 256)
    if staged:
        # large batches: nobody loads from peer memory.  The owners deliver the requested rows (wr_xchg_*), the batch
        # kernel runs on local memory, and the gradient rows are written into the owners' inboxes and reduced there
        # (Running the dense Adam of the rows the batch does not touch on a second stream beside the exchange was tried:
        # 1.54 -> 1.66 ms per step at 8 GPUs, profiles/r02_prof_sharded_n8_v4_adam_overlap_experiment.json -- both sides
        # are HBM-bound, so nothing was hidden and the row-masked sweep is slower than the dense one.)
        inbox = tabs.inbox(B_global)
        x = tabs.exchange(B_global)
        tabs.fetch_rows(x, tabs.P, user, pos, neg)
        # rows reduced in place (entries this rank owns) and rows that arrive through the inbox both mark the row map:
        # those are the only rows of G the sweep has to read and re-zero
        touched = tabs.row_map()
        _lib.bpr_fwd_bwd_exchanged(x['recv'], x['where'], tabs.Gd, inbox['row_ptrs'], inbox['idx_ptrs'], inbox['cap'],
                                   user, pos, neg, B_global, tabs.D, tabs.loss_part, tabs.ws, touched=touched)
        loss = tabs.peers.barrier(tabs.loss_part[:1])
        _lib.inbox_scatter(tabs.G, inbox['rows'], inbox['idx'], tabs.layout.world, inbox['cap'], touched)
        tabs.adam(lr, l2, touched=touched)
        # No meeting point after the sweep: in this protocol a rank's rows are only ever read by the rank itself (it
        # serves them after its own sweep, in stream order), and every buffer a peer writes next -- request lists, receive
        # blocks, inboxes -- is written behind a barrier of the NEXT step that this rank reaches only after the kernels
        # above.  Paths that do read peers' rows meet first (settle()).
        tabs._unsettled = True
        return loss
    tabs.settle()
    _lib.bpr_fwd_bwd_sharded(tabs.T, tabs.Gd, user, pos, neg, B_global, tabs.D, tabs.loss_part, tabs.ws)
    loss = tabs.peers.barrier(tabs.loss_part[:1])
    tabs.adam(lr, l2)
    tabs.peers.barrier()
    return loss


def local_rows(lay, rowptr, col):
    """This rank's rows of a GLOBAL node CSR (int64 rowptr / int32 col tensors, on any device), in local row order:
    (rowptr_local [n_local + 1], col_local (global node ids), src: position of every local edge in `col`,
    rows: local row of every local edge, nodes: global node of every local row, -1 on padding rows)."""
    dev = rowptr.device
    nodes = torch.from_numpy(lay.local_nodes()).to(dev)
    safe = nodes.clamp(min=0)
    deg = torch.where(nodes >= 0, rowptr[safe + 1] - rowptr[safe], torch.zeros_like(safe))
    lptr = torch.zeros(lay.n_local + 1, dtype=torch.int64, device=dev)
    torch.cumsum(deg, 0, out=lptr[1:])
    total = int(lptr[-1].item())
    rows = torch.repeat_interleave(torch.arange(lay.n_local, device=dev), deg)
    src = rowptr[safe][rows] + (torch.arange(total, device=dev) - lptr[:-1][rows])
    return lptr, col[src], src, rows, nodes


class LocalGraph(object):
    """This rank's rows of a GLOBAL node CSR (every rank passes the same; NumPy arrays or device tensors), cut out on the
    device by local_rows; column ids stay global node ids.  Weights: `val` (global, one per edge) sliced, or LightGCN's
    fl32(fl32(dinv[row] * 1) * dinv[col]) from `dinv` (LightGCN.py:89-97)."""

    def __init__(self, tabs, rowptr, col, dinv=None, val=None):
        lay, dev = tabs.layout, tabs.peers.device
        as_dev = lambda a, dt: (a if torch.is_tensor(a) else torch.from_numpy(np.ascontiguousarray(a))).to(dev).to(dt)
        lptr, col_local, src, rows, nodes = local_rows(lay, as_dev(rowptr, torch.int64), as_dev(col, torch.int32))
        safe = nodes.clamp(min=0)
        total = int(lptr[-1].item())
        self.rowptr = lptr
        self.col = col_local.contiguous() if total else torch.zeros(1, dtype=torch.int32, device=dev)
        if not total:
            self.val = torch.zeros(1, dtype=torch.float32, device=dev)
        elif val is not None:
            self.val = as_dev(val, torch.float32)[src].contiguous()
        else:
            dinv_d = as_dev(dinv, torch.float32)
            d_row = torch.where(nodes >= 0, dinv_d[safe], torch.zeros_like(dinv_d[safe]))
            self.val = ((d_row[rows] * 1.0) * dinv_d[self.col[:total].long()]).contiguous()
        del rows, src
        self.plan = _lib.SpmmPlan(lptr.cpu().numpy(), tabs.D, dev)
        self.nnz = total


class ShardedLightGCN(object):
    """LightGCN propagation state of one rank: its rows of the adjacency and the symmetric layer / pool buffers."""

    def __init__(self, tabs, rowptr, col, dinv, n_layers, reg_weight, gather_first=None):
        """rowptr / col / dinv: the GLOBAL node CSR structure and d^-1/2 (NumPy arrays or device tensors; every rank
        passes the same).  The rank's rows are cut out on the device."""
        self.tabs, self.L, self.reg_weight = tabs, int(n_layers), float(reg_weight)
        lay, dev = tabs.layout, tabs.peers.device
        self.graph = LocalGraph(tabs, rowptr, col, dinv=dinv)
        self.rowptr, self.col, self.val = self.graph.rowptr, self.graph.col, self.graph.val
        self.plan, self.nnz = self.graph.plan, self.graph.nnz
        total = self.nnz
        self.pool, self.pool_T = tabs.symmetric()
        self.pool_grad, self.pool_Gd = tabs.symmetric()
        self.layer = [tabs.symmetric(), tabs.symmetric()]
        self.sumsq = torch.zeros(_lib.PEER_VALUES, dtype=torch.float32, device=dev)
        # Neighbour rows: read in place from their owners (small tables: latency matters, the rows are few), or
        # all-gathered into a local copy first (large power-law graphs: every neighbour row is re-read many times and
        # only local memory has those re-reads served by the L2; peer reads always cross NVLink).
        self.gather_first = (lay.world > 1 and total * 4 * tabs.D > (256 << 20)) if gather_first is None \
            else bool(gather_first) and lay.world > 1
        # two symmetric (peer-mapped) copies of the whole table, [world, n_local, D] each: a layer's SpMM reads one while
        # its epilogue -- and the other ranks' -- fill the other with that layer's output (the fused all-gather)
        self.gathered, self.gathered_ptrs = [], []
        if self.gather_first:
            for _ in range(2):
                buf, ptrs = tabs.peers.alloc((lay.world, lay.n_local, tabs.D))
                self.gathered.append(buf)
                self.gathered_ptrs.append(ptrs)
        # all-gathers by the copy engines beside the SpMM (wr_csr_spmm_sharded_dma) where the kernel has the fast row form
        self.dma = self.gather_first and tabs.D in (16, 32, 64, 128, 256)
        # layer outputs: pushed by the SpMM's own epilogue stores.  WR_SPMM_PUSH=dma selects the copy-engine push beside the
        # kernel (wr_csr_spmm_sharded_dma) -- measured slower at 8 GPUs (16.4 vs 14.0 ms per pass, step 99 vs 88 ms,
        # profiles/r02_prof_sharded_n8_v8_*.json), kept as an option
        self.dma_spmm = os.environ.get('WR_SPMM_PUSH', 'store') == 'dma'
        if self.dma:
            self._block_rows = 32
            while self._block_rows * 32 < lay.n_local:
                self._block_rows *= 2
            nblk = (lay.n_local + self._block_rows - 1) // self._block_rows
            self._progress = torch.zeros(2 * nblk, dtype=torch.int32, device=dev)
            self._epoch = 0
            self._side = torch.cuda.Stream(device=dev)
        self.sparse_grad = None       # None: the batch decides (_step_exchanged); True / False force it
        self._cur = 0                 # which copy holds (or receives by all-gather) the next SpMM's input
        self._pushed = None           # base pointer of the shard whose rows the last SpMM pushed into gathered[_cur]
        self._local_views = {}
        tabs.peers.host_sync()

    def _local_view(self, X, which):
        """wr_shards whose peers' bases point into the gathered local copy `which` (own shard read in place)."""
        key = (X.base[X.rank], which)
        v = self._local_views.get(key)
        if v is None:
            v = _lib.ShardsStruct()
            ctypes.memmove(ctypes.addressof(v), ctypes.addressof(X), ctypes.sizeof(v))
            step = self.gathered[which][0].numel() * 4
            for g in range(X.world):
                if g != X.rank:
                    v.base[g] = self.gathered[which].data_ptr() + g * step
            self._local_views[key] = v
        return v

    def _spmm(self, X, push=False, graph=None, **kw):
        """One propagation over `graph` (a LocalGraph; default: this object's adjacency).  push=True: the output Y is the
        next SpMM's input -- its rows go into every peer's other gathered copy while the kernel runs (copy engines;
        store-push epilogue where that is not available), and that SpMM skips its all-gather."""
        t = self.tabs
        g = self.graph if graph is None else graph
        lay = t.layout
        push_ptrs = None
        if self.gather_first:
            cur = self._cur
            step = self.gathered[0][0].numel() * 4
            if self._pushed != X.base[X.rank]:            # input not delivered by the previous SpMM
                if self.dma:                              # push it (copy engines), then meet
                    src = self._shard_tensor(X)
                    _lib.push_shard_dma(src, lay.world, lay.rank,
                                        [None if g == lay.rank else self.gathered_ptrs[cur][g] + lay.rank * step
                                         for g in range(lay.world)])
                    t.peers.barrier()
                else:                                     # pull it
                    _lib.allgather_shards(X, self.gathered[cur], t.D)
            X = self._local_view(X, cur)
            self._pushed = None
            if push:
                push_ptrs = [None if g == lay.rank else self.gathered_ptrs[1 - cur][g] + lay.rank * step
                             for g in range(lay.world)]
                self._pushed = kw['Y'].data_ptr()
                self._cur = 1 - cur
        if push_ptrs is not None and self.dma and self.dma_spmm:
            self._epoch += 1
            _lib.csr_spmm_sharded_dma(g.rowptr, g.col, g.val, lay.n_local, t.D, X, kw.pop('Y'), push_ptrs,
                                      self._progress, self._block_rows, self._epoch, self._side, nnz=g.nnz,
                                      plan=g.plan, **kw)
        else:
            _lib.csr_spmm_sharded(g.rowptr, g.col, g.val, lay.n_local, t.D, X, plan=g.plan,
                                  push_ptrs=push_ptrs, **kw)
        t.peers.barrier()          # every rank's rows of the output exist (everywhere) before anyone reads them

    def _shard_tensor(self, X):
        """The local tensor behind a wr_shards struct of this object (P, the pooled gradient or a layer buffer)."""
        base = X.base[X.rank]
        for cand in self._shard_tensors():
            if cand.data_ptr() == base:
                return cand
        raise _lib.WhisprError('unknown shard')

    def _shard_tensors(self):
        return (self.tabs.P, self.pool_grad, self.pool, self.layer[0][0], self.layer[1][0], self.tabs.G)

    def propagate(self, graph=None, pool=None):
        """LightGCN.py:134-148 on row shards: layer k+1 reads its neighbours' layer-k rows from their owners.
        graph / pool: a LocalGraph and the local pool tensor it fills (default: this object's adjacency and pool)."""
        t, L = self.tabs, self.L
        pool = self.pool if pool is None else pool
        t.settle()
        if L == 0:
            pool.copy_(t.P)
            t.peers.barrier()
            return
        x = t.T
        for k in range(1, L + 1):
            y, ys = self.layer[(k - 1) & 1]
            self._spmm(x, push=k < L, graph=graph, Y=y if k < L else None, acc_in=t.P if k == 1 else pool,
                       acc_out=pool, acc_div=float(L + 1) if k == L else 1.0)
            x = ys

    def step(self, user, pos, neg, B_global, lr, l2):
        """LightGCN.py:150-175 + backward + Adam on this rank's slice of the batch."""
        t, L = self.tabs, self.L
        self.propagate()
        per_rank = (int(B_global) + t.layout.world - 1) // t.layout.world
        if L > 0 and t.layout.world > 1 and per_rank >= 8192 and t.D in (16, 32, 64, 128, 256):
            return self._step_exchanged(user, pos, neg, B_global, lr, l2)
        if L == 0:
            _lib.bpr_fwd_bwd_sharded(t.T, t.Gd, user, pos, neg, B_global, t.D, t.loss_part, t.ws)
        else:
            _lib.bpr_fwd_bwd_sharded(self.pool_T, self.pool_Gd, user, pos, neg, B_global, t.D, t.loss_part, t.ws,
                                     grad_scale=1.0 / (L + 1))
        _lib.embloss_sumsq_sharded(t.T, user, pos, neg, t.D, t.loss_part[1:], t.ws)
        sums = t.peers.barrier(t.loss_part)          # pooled gradients landed; loss and the three norms reduced
        t.loss.copy_(sums[:1])
        self.sumsq[:3].copy_(sums[1:4])
        if L > 0:
            h = self.pool_Gd
            for k in range(1, L + 1):
                last = k == L
                y, ys = (t.G, t.Gd) if last else self.layer[(k - 1) & 1]
                self._spmm(h, push=not last, Y=y, add=self.pool_grad, zero_add=last and L > 1)
                h = ys
            if L == 1:
                self.pool_grad.zero_()
        _lib.embloss_scatter_sharded(t.T, t.Gd, user, pos, neg, B_global, t.D, self.reg_weight, self.sumsq, t.loss,
                                     t.ws)
        t.peers.barrier()                            # every gradient row has landed
        t.adam(lr, l2)
        t.peers.barrier()
        return t.loss


def _step_exchanged(self, user, pos, neg, B_global, lr, l2):
    """The rest of ShardedLightGCN.step for large batches (after propagate): pooled rows delivered by their owners,
    EmbLoss computed by the owners of the ego rows from the request lists -- no loads from peer memory, no remote REDs."""
    t, L = self.tabs, self.L
    lay = t.layout
    world = lay.world
    x, inbox = t.exchange(B_global), t.inbox(B_global)
    # The pooled gradient is zero outside the batch's <= 3 B_global rows.  When those are a small part of the table the
    # first adjoint propagation needs neither the other rows (its SpMM skips them: wr_spmm_plan.x_rows) nor their
    # all-gather: the owners push just the marked rows.  The map is over GLOBAL node ids: every rank marks its slice,
    # the maps are OR-ed (1 bit per node: 1.5 MB for 12 M nodes).
    sparse = self.gather_first and (12 * int(B_global) <= lay.n_users + lay.n_items if self.sparse_grad is None
                                    else bool(self.sparse_grad))
    if sparse:
        gm = self._node_map()
        _lib.mark_rows(user, pos, neg, lay.n_users, lay.n_items, gm)
        t.peers.dist.all_gather_into_tensor(self._node_maps, gm, group=t.peers.group)
        for g in range(world):
            if g != lay.rank:
                gm.bitwise_or_(self._node_maps[g])
    t.fetch_rows(x, self.pool, user, pos, neg)
    _lib.bpr_fwd_bwd_exchanged(x['recv'], x['where'], self.pool_Gd, inbox['row_ptrs'], inbox['idx_ptrs'], inbox['cap'],
                               user, pos, neg, B_global, t.D, t.loss_part, t.ws, grad_scale=1.0 / (L + 1))
    _lib.embloss_owner_sumsq(t.P, world, x['req'], x['cnt'], x['cap'], t.loss_part[1:], t.ws)
    sums = t.peers.barrier(t.loss_part)          # pooled gradient rows are in the inboxes; loss and the three norms reduced
    t.loss.copy_(sums[:1])
    self.sumsq[:3].copy_(sums[1:4])
    _lib.inbox_scatter(self.pool_grad, inbox['rows'], inbox['idx'], world, inbox['cap'])
    if sparse:
        step = self.gathered[0][0].numel() * 4
        cur = self._cur
        _lib.push_marked_rows(self.pool_Gd, t.D, gm, [None if g == lay.rank else self.gathered_ptrs[cur][g] + lay.rank * step
                                                       for g in range(world)])
        self._pushed = self.pool_Gd.base[lay.rank]       # the SpMM below finds its input delivered
    t.peers.barrier()                            # every rank's pooled gradient is complete (and, pushed, has landed)
    h = self.pool_Gd
    for k in range(1, L + 1):
        last = k == L
        y, ys = (t.G, t.Gd) if last else self.layer[(k - 1) & 1]
        self._spmm(h, push=not last, Y=y, add=self.pool_grad, zero_add=last and L > 1,
                   x_rows=gm if sparse and k == 1 else None)
        h = ys
    if sparse:
        gm.zero_()
    if L == 1:
        self.pool_grad.zero_()
    _lib.embloss_owner_scatter(t.P, t.G, world, x['req'], x['cnt'], x['cap'], self.reg_weight, B_global, self.sumsq, t.loss)
    t.adam(lr, l2)
    t.peers.barrier()
    return t.loss


def _node_map(self):
    if getattr(self, '_gm', None) is None:
        lay = self.tabs.layout
        self._gm = _lib.row_map(lay.n_users + lay.n_items, self.tabs.peers.device)
        self._node_maps = torch.zeros((lay.world, self._gm.numel()), dtype=torch.int32, device=self.tabs.peers.device)
    return self._gm


ShardedLightGCN._node_map = _node_map
ShardedLightGCN._step_exchanged = _step_exchanged


class ShardedSGL(ShardedLightGCN):
    """SGL (models/general/SGL.py) on row shards: three pooled tables -- the main graph's and the two edge-dropout
    views' -- propagated from the same ego table, their pooled gradients, and this rank's rows of the views and of their
    transposes (set_views, every epoch).  The main graph, the layer buffers and the SpMM are ShardedLightGCN's.

    InfoNCE is split by table shard (wr_infonce_sharded_*): every rank runs the global batch against its own rows of
    the view tables, so it needs the global batch's user and positive ids.  One protocol at every batch size: the
    peer-load form.  The row exchange that BPRMF / LightGCN switch to at >= 8,192 rows per rank is not implemented for
    SGL."""

    def __init__(self, tabs, rowptr, col, dinv, n_layers, reg_weight, ssl_tau, ssl_weight, gather_first=None):
        super().__init__(tabs, rowptr, col, dinv, n_layers, reg_weight, gather_first=gather_first)
        if self.L < 1:
            raise NotImplementedError('SGL needs at least one propagation layer')
        self.ssl_tau, self.ssl_weight = float(ssl_tau), float(ssl_weight)
        self.view_pool = [tabs.symmetric(), tabs.symmetric()]       # (local tensor, wr_shards) of view 1 / view 2
        self.view_grad = [tabs.symmetric(), tabs.symmetric()]
        self.views = None               # [(LocalGraph of the view, LocalGraph of its transpose)] x 2
        self._slots = None
        self._scratch = [None, None]
        tabs.peers.host_sync()

    def _shard_tensors(self):
        return super()._shard_tensors() + tuple(p for p, _ in self.view_pool + self.view_grad)

    def set_views(self, views):
        """views: the epoch's two views as edge_dropout_view_device returns them (GLOBAL device CSRs, the same on every
        rank); keeps this rank's rows of each view and of its transpose."""
        t = self.tabs
        self.views = [(LocalGraph(t, *fwd[:2], val=fwd[2]), LocalGraph(t, *tr[:2], val=tr[2])) for fwd, tr in views]

    def slots(self, B):
        """Symmetric z / Ga slot arrays of the sharded InfoNCE for a global batch of up to B rows (collective)."""
        lay = self.tabs.layout
        if self._slots is None or self._slots['cap'] < B:
            z, z_ptrs = self.tabs.peers.alloc((lay.world, B))
            ga, ga_ptrs = self.tabs.peers.alloc((lay.world, B, self.tabs.D))
            self._slots = {'cap': B, 'z': z, 'z_ptrs': z_ptrs, 'ga': ga, 'ga_ptrs': ga_ptrs}
            self.tabs.peers.host_sync()
        return self._slots

    def _infonce(self, which, ids, scale):
        """InfoNCE of one block (0: the batch's users, 1: its positive items): three phases, two barriers."""
        t, lay = self.tabs, self.tabs.layout
        B = ids.numel()
        sl = self.slots(B)
        n = lay.n_users if which == 0 else lay.n_items
        n_local = (n - lay.rank + lay.world - 1) // lay.world          # rows u % world == rank of the block
        sc = self._scratch[which] = _lib.infonce_sharded_scratch(B, n_local, t.D, t.peers.device, self._scratch[which])
        (_, p1), (_, p2) = self.view_pool
        (_, g1), (_, g2) = self.view_grad
        _lib.infonce_sharded_partials(p1, p2, which, ids, t.D, self.ssl_tau, sl['z_ptrs'], sc, t.ws)
        t.peers.barrier()               # every rank's partial z has landed
        _lib.infonce_sharded_weights(g2, which, ids, t.D, self.ssl_tau, self.ssl_weight, scale, sl['z_ptrs'],
                                     sl['ga_ptrs'], t.loss, sc)
        t.peers.barrier()               # every rank's partial Ga has landed at the owners
        _lib.infonce_sharded_batch(g1, which, ids, t.D, self.ssl_tau, self.ssl_weight, scale, sl['ga_ptrs'], sc)

    def _adjoint(self, gt, grad, first):
        """SGL._adjoint on shards: dE0 += H_0 with H_L = grad, H_{k-1} = grad + A^T H_k; gt: the transpose's LocalGraph,
        grad: (local tensor, wr_shards) of a pooled gradient."""
        t, L = self.tabs, self.L
        g_local, h = grad
        for k in range(1, L + 1):
            last = k == L
            kw = dict(graph=gt, add=g_local, zero_add=last and L > 1)
            if not last:
                y, ys = self.layer[(k - 1) & 1]
                self._spmm(h, push=True, Y=y, **kw)
                h = ys
            elif first:
                self._spmm(h, Y=t.G, **kw)                                  # tabs.G is zero: overwrite
            else:
                self._spmm(h, acc_in=t.G, acc_out=t.G, acc_div=1.0, **kw)
        if L == 1:
            g_local.zero_()

    def step(self, user, pos, neg, B_global, lr, l2, batch_user, batch_pos, mark=None):
        """SGL.py:233-246 + backward + Adam on this rank's slice (user, pos, neg) of a global batch whose user and
        positive ids are batch_user / batch_pos (the same on every rank).  mark (optional): called with the name of
        each phase as it is issued (scripts/bench_sgl_sharded.py records an event there)."""
        t, L = self.tabs, self.L
        mark = mark or (lambda name: None)
        if self.views is None:
            raise _lib.WhisprError('ShardedSGL.step before set_views')
        pools = [(self.graph, (self.pool, self.pool_T))] + [(v[0], p) for v, p in zip(self.views, self.view_pool)]
        for g, (p, _) in pools:
            self.propagate(g, p)
        mark('propagate_x3')
        scale = 1.0 / (L + 1)
        _lib.bpr_logsig_sum_fwd_bwd_sharded(self.pool_T, self.pool_Gd, user, pos, neg, B_global, t.D, t.loss_part, t.ws,
                                            grad_scale=scale)
        _lib.embloss_sumsq_sharded(t.T, user, pos, neg, t.D, t.loss_part[1:], t.ws)
        sums = t.peers.barrier(t.loss_part)          # BPR sums and the three norms reduced
        t.loss.copy_(sums[:1])
        self.sumsq[:3].copy_(sums[1:4])
        mark('bpr_embloss_norms')
        self._infonce(0, batch_user, scale)          # adds the batch's InfoNCE loss to t.loss once, on every rank
        mark('infonce_users')
        self._infonce(1, batch_pos, scale)
        t.peers.barrier()                            # every pooled gradient row has landed
        mark('infonce_items')
        graphs_t = [self.graph] + [v[1] for v in self.views]
        grads = [(self.pool_grad, self.pool_Gd)] + self.view_grad
        for n, (gt, grad) in enumerate(zip(graphs_t, grads)):
            self._adjoint(gt, grad, first=n == 0)
        mark('adjoint_x3')
        _lib.embloss_scatter_sharded(t.T, t.Gd, user, pos, neg, B_global, t.D, self.reg_weight, self.sumsq, t.loss,
                                     t.ws)
        t.peers.barrier()                            # every gradient row has landed
        mark('embloss_scatter')
        t.adam(lr, l2)
        t.peers.barrier()
        mark('adam')
        return t.loss


def sharded_eval(tabs, shards, item_table_local, user, pos, hist_local, k=0, precision=0):
    """Full-ranking evaluation with the items sharded over the ranks (every rank scores all R rows against its items).

    shards: wr_shards of the table that is scored (P for BPRMF, the pooled table for LightGCN);
    item_table_local: this rank's item rows of it.  Returns (rank int32 [R], target fp32 [R], topk_idx | None,
    topk_val | None), identical on every rank.  The exchange is one all-reduce of the per-shard counts and, for the
    top-k lists, one all-gather of [R, k] candidates followed by the merge kernel."""
    lay, peers, D = tabs.layout, tabs.peers, tabs.D
    dist = peers.dist
    peers.barrier()                    # the table being scored is final on every rank
    urows = _lib.gather_rows_sharded(shards, 0, user, D, tabs.ws)
    prows = _lib.gather_rows_sharded(shards, 1, pos, D, tabs.ws)
    target = _lib.rowdot(urows, prows, round_bf16=(precision == 1))
    pos_local = lay.item_local_index(pos)
    rank_local, tki, tkv = _lib.eval_rank_topk_shard(urows, item_table_local, user, pos_local, lay.n_users,
                                                    hist_local[0], hist_local[1], target, tabs.ws, k=k,
                                                    precision=precision)
    counts = rank_local - 1
    dist.all_reduce(counts, group=peers.group)
    rank = counts + 1
    if k <= 0:
        return rank, target, None, None
    gi = lay.item_global_index(tki).contiguous()
    all_i = torch.empty((lay.world,) + tuple(gi.shape), dtype=gi.dtype, device=gi.device)
    all_v = torch.empty((lay.world,) + tuple(tkv.shape), dtype=tkv.dtype, device=tkv.device)
    dist.all_gather_into_tensor(all_i, gi, group=peers.group)
    dist.all_gather_into_tensor(all_v, tkv.contiguous(), group=peers.group)
    mv, mi = _lib.topk_merge(all_v, all_i, k)
    return rank, target, mi, mv
