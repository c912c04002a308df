"""Stage IV -- complementarity inference (the entry point the reference README names, README.md:14-16,30-32,
whose script is absent from the tree; semantics follow RankingLoss, codae/tool/metering.py:46-79).

context outfit with slot c zeroed -> DAE forward -> predicted embedding p of slot c -> score every catalog
item of category c (squared error against p, or cosine similarity) -> top-k.  The catalog is sharded by rows
across ranks; each rank sweeps its shard (codae_score_topk) and the per-rank lists are all-gathered and merged
deterministically (codae_topk_merge).

Both scorers take an optional filter: `allowed`, a per-shard mask of the rows that may be returned (items in stock, in the
right region), and per call `exclude`, global row indices a query must not get back (the item the outfit already holds).  A
filtered-out row is treated as absent from the catalog, inside the kernels (include/codae_b200.h: filtered top-k).

SwapScorer is the other reading of "scores candidate item swaps by reconstruction error": every candidate is
substituted into the slot, the whole swapped outfit goes through the DAE (tensor-core GEMMs batched over the
candidates) and the swap is scored by the reconstruction error of the swapped outfit.

CompatibilityScorer answers the question asked of a complete outfit: how well do its items go together, and which one fits least?
Each slot is hidden in turn and reconstructed; the per-slot errors, their sum and the slot of largest error come back, and
compatibility_auc scores real outfits against shuffled ones.
"""
import torch

from codae import _C

METRICS = {"sqerr": _C.METRIC_SQERR, "cosine": _C.METRIC_COSINE}


def _allowed_mask(allowed, n_local, device):
    """bool / uint8 [n_local] CUDA tensor on the catalog's device -> contiguous uint8 (None: every row)."""
    if allowed is None:
        return None
    if not isinstance(allowed, torch.Tensor) or allowed.dtype not in (torch.bool, torch.uint8):
        raise RuntimeError("codae: allowed must be a bool or uint8 tensor")
    if allowed.dim() != 1 or allowed.shape[0] != n_local:
        raise RuntimeError("codae: allowed must have shape [%d] (rows of this shard), got %s" % (n_local, tuple(allowed.shape)))
    if not allowed.is_cuda or allowed.device != device:
        raise RuntimeError("codae: allowed must be on the catalog's device %s" % device)
    return allowed.to(torch.uint8).contiguous()


def _exclusions(exclude, shape0, device):
    """int64 CUDA tensor of global row indices, [Q, m] (shape0 = Q) or [m] (shape0 = None), -1 padding; m <= 256."""
    if exclude is None:
        return None
    if not isinstance(exclude, torch.Tensor) or exclude.dtype != torch.int64:
        raise RuntimeError("codae: exclude must be an int64 tensor")
    want = "[m]" if shape0 is None else "[%d, m]" % shape0
    if (exclude.dim() != (1 if shape0 is None else 2) or (shape0 is not None and exclude.shape[0] != shape0)
            or exclude.shape[-1] > _C.TOPK_MAX_EXCLUDE):
        raise RuntimeError("codae: exclude must have shape %s with m <= %d, got %s" % (want, _C.TOPK_MAX_EXCLUDE,
                                                                                   tuple(exclude.shape)))
    if not exclude.is_cuda or exclude.device != device:
        raise RuntimeError("codae: exclude must be on the catalog's device %s" % device)
    return exclude.contiguous()


def _pair_lists(outfits, candidates, io, device):
    """SwapScorer.rerank_local's inputs: outfits fp32 [Q, io] and candidates int64 [Q, m] (Q m <= 2**31 - 1), both on the
    catalog's device; contiguous copies."""
    if not isinstance(outfits, torch.Tensor) or outfits.dtype != torch.float32:
        raise RuntimeError("codae: outfits must be a float32 tensor")
    if outfits.dim() != 2 or outfits.shape[1] != io or outfits.shape[0] < 1:
        raise RuntimeError("codae: outfits must have shape [Q, %d] with Q >= 1, got %s" % (io, tuple(outfits.shape)))
    if not isinstance(candidates, torch.Tensor) or candidates.dtype != torch.int64:
        raise RuntimeError("codae: candidates must be an int64 tensor")
    if candidates.dim() != 2 or candidates.shape[0] != outfits.shape[0] or candidates.shape[1] < 1:
        raise RuntimeError("codae: candidates must have shape [%d, m] with m >= 1, got %s" % (outfits.shape[0],
                                                                                           tuple(candidates.shape)))
    if candidates.numel() > 2 ** 31 - 1:
        raise RuntimeError("codae: candidates has %d entries, more than 2**31 - 1" % candidates.numel())
    for name, t in (("outfits", outfits), ("candidates", candidates)):
        if not t.is_cuda or t.device != device:
            raise RuntimeError("codae: %s must be on the catalog's device %s" % (name, device))
    return outfits.contiguous(), candidates.contiguous()


def _gather_merge(pg, s, i, metric):
    """All-gather of every rank's [Q, k] lists and the deterministic merge (codae_topk_merge); one process: (s, i)."""
    import torch.distributed as dist
    if pg is None and not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
        return s, i
    G = dist.get_world_size(pg)
    gs = torch.empty((G,) + tuple(s.shape), dtype=s.dtype, device=s.device)
    gi = torch.empty((G,) + tuple(i.shape), dtype=i.dtype, device=i.device)
    dist.all_gather_into_tensor(gs, s.contiguous(), group=pg)
    dist.all_gather_into_tensor(gi, i.contiguous(), group=pg)
    out_s, out_i = torch.empty_like(s), torch.empty_like(i)
    _C.topk_merge(gs, gi, metric, out_s, out_i)
    return out_s, out_i


def shard_rows(n_rows, world_size, rank):
    """Contiguous ceil(N/G)-row shards: (row_offset, n_local)."""
    per = (n_rows + world_size - 1) // world_size
    lo = min(rank * per, n_rows)
    return lo, min(per, n_rows - lo)


class ComplementarityScorer:
    # Query batches of at least this many go through the tensor-core path (topk_batched) in the stage-IV script:
    # the measured crossover against the row sweep on a 10 M x 512 catalog (DESIGN.md section 6).
    TC_MIN_Q = 64

    def __init__(self, catalog, embedding_size, metric="sqerr", k=10, inv_scale=1.0, row_offset=0, process_group=None,
                 allowed=None):
        """catalog: [n_local, E] fp32 or bf16 CUDA tensor -- this rank's shard (rows row_offset.. of the global
        catalog).  inv_scale multiplies catalog values before the squared error (1/dataset.scale when the
        catalog is un-scaled like dataset.data_per_category).  allowed: bool / uint8 [n_local] CUDA tensor, the rows of this
        shard that may be returned (None: all)."""
        if metric not in METRICS:
            raise Exception("Unknown metric.")
        if not catalog.is_cuda:
            raise RuntimeError("codae: catalog is not on a CUDA device; the B200 path has no CPU fallback")
        self.catalog = catalog
        self.E = embedding_size
        self.metric = METRICS[metric]
        self.k = k
        self.inv_scale = float(inv_scale)
        self.row_offset = int(row_offset)
        self.pg = process_group
        self.allowed = _allowed_mask(allowed, catalog.shape[0], catalog.device)
        self._ws = {}
        self._ws_batched = {}
        self.last_fallbacks = 0     # queries of the last batched call that were answered by the row sweep

    def _workspace(self, Q):
        ws = self._ws.get(Q)
        if ws is None:
            dev = self.catalog.device
            ws = (_C.score_topk_workspace(dev, Q, self.k), torch.empty((Q, self.k), dtype=torch.float32, device=dev),
                  torch.empty((Q, self.k), dtype=torch.int64, device=dev))
            self._ws[Q] = ws
        return ws

    def topk_local(self, query, exclude=None):
        """(scores [Q,k] f32, global indices [Q,k] i64) of this shard; asynchronous, reuses its buffers.  exclude: int64
        [Q, m] CUDA tensor of global row indices query q must not get back (-1 padding, m <= 256)."""
        q = query.to(torch.float32).contiguous()
        ex = _exclusions(exclude, q.shape[0], self.catalog.device)
        ws, s, i = self._workspace(q.shape[0])
        _C.score_topk(self.catalog, self.E, self.row_offset, q, self.inv_scale, self.metric, self.k, s, i, ws,
                      allow=self.allowed, exclude=ex)
        return s, i

    def _workspace_batched(self, Q):
        ws = self._ws_batched.get(Q)
        if ws is None:
            dev = self.catalog.device
            ws = (_C.score_topk_batched_workspace(self.catalog, self.E, Q, self.k),
                  torch.empty((Q, self.k), dtype=torch.float32, device=dev), torch.empty((Q, self.k), dtype=torch.int64, device=dev),
                  torch.zeros(1, dtype=torch.int32, device=dev), torch.empty(Q, dtype=torch.int32, device=dev))
            self._ws_batched[Q] = ws
        return ws

    def topk_local_batched(self, query, exclude=None):
        """Same inputs and results as topk_local -- the same scores bit for bit and the same indices -- for many queries in
        about one pass over the shard: the tensor cores propose candidates, they are re-scored with the sweep's arithmetic,
        and the queries whose result cannot be certified (last_fallbacks of them) are answered by the sweep.  Synchronises
        once (one 4-byte device-to-host read of that count); reuses its buffers.  k > 64 is the sweep alone."""
        q = query.to(torch.float32).contiguous()
        Q = q.shape[0]
        ex = _exclusions(exclude, Q, self.catalog.device)
        if self.k > _C.TOPK_BATCHED_MAX_K:
            self.last_fallbacks = Q
            return self.topk_local(q, ex)
        ws, s, i, n_unc, unc = self._workspace_batched(Q)
        _C.score_topk_batched(self.catalog, self.E, self.row_offset, q, self.inv_scale, self.metric, self.k, s, i, n_unc, unc, ws,
                              allow=self.allowed, exclude=ex)
        nf = int(n_unc.item())
        self.last_fallbacks = nf
        if nf:
            rows = unc[:nf].long()
            fs, fi = self.topk_local(q.index_select(0, rows), None if ex is None else ex.index_select(0, rows))
            s.index_copy_(0, rows, fs)
            i.index_copy_(0, rows, fi)
        return s, i

    def topk_batched(self, query, exclude=None):
        """Global top-k of a query batch: topk_local_batched on this rank's shard (certification and fallback are per rank),
        then the same all-gather + merge as topk -- every rank reaches it exactly once, whatever its fallback count.
        exclude holds global indices, so every rank is given the same tensor."""
        return _gather_merge(self.pg, *self.topk_local_batched(query, exclude), self.metric)

    def topk(self, query, exclude=None):
        """Global top-k: local sweep, all-gather of k x 12 bytes per query, deterministic merge."""
        return _gather_merge(self.pg, *self.topk_local(query, exclude), self.metric)


def predict_slot(model, outfits, slot, embedding_size):
    """Zero slot `slot` of the (scaled) outfit rows, run the DAE, return the reconstructed slot [Q, E]."""
    E = embedding_size
    mask = torch.ones_like(outfits)
    mask[:, slot * E:(slot + 1) * E] = 0
    with torch.no_grad():
        y = model(model.corrupt(input_data=outfits, mask=mask))
    return y[:, slot * E:(slot + 1) * E].contiguous()


class _DaeChunks:
    """The DAE's Linear layers over chunks of up to `rows` outfit rows, the forward pass of SwapScorer and CompatibilityScorer:
    the caller writes a chunk's input rows into acts[0] (or, on the fp32-parity engine, into the fp32 stage and splits it into
    acts[0]'s three bf16 planes), forward() leaves the reconstructions in acts[-1] (fp32)."""

    def __init__(self, model, rows, io, device):
        self.model, self.rows, self.io, self.device = model, int(rows), io, device
        self._acts = None

    def buffers(self):
        """(engine, activations, fp32 stage or None), allocated once."""
        if self._acts is None:
            m, dev = self.model, self.device
            eng = m.engine_dtype()
            adt = m.act_dtype(eng)
            acts = [m.new_activation(self.rows, self.io, adt, dev)]
            for l, (i, o) in enumerate(m.dims):
                acts.append(m.new_activation(self.rows, o, torch.float32 if l == len(m.dims) - 1 else adt, dev))
            # fp32-parity engine: the rows are built in fp32 and split into the engine's three bf16 planes
            stage = m.new_activation(self.rows, self.io, torch.float32, dev) if eng == _C.F32X3 else None
            self._acts = (eng, acts, stage)
        return self._acts

    def prepare(self):
        """Weights and activation buffers of one scoring call: (engine, activations, fp32 stage or None, GEMM weights)."""
        m = self.model
        m.sync_weights()          # a sharded data-parallel trainer gathers the master weights first (collective)
        eng, acts, stage = self.buffers()
        m.refresh_shadow()
        return eng, acts, stage, m.gemm_weights(eng)

    def forward(self, eng, acts, wflat, B):
        """The DAE's Linear layers on the B rows in acts[0]; the reconstructions land in acts[-1]."""
        m = self.model
        for l, (i, o) in enumerate(m.dims):
            _C.linear_fwd(acts[l], m.aug_view(wflat, l), None, acts[l + 1], B, o, (i + 7) // 8 * 8 + 1,
                          _C.ACT_RELU if m.relu[l] else _C.ACT_NONE, eng)


class SwapScorer:
    """Scores the swap "candidate j into slot c" by || DAE(outfit_j) - outfit_j ||^2 over all io dimensions (lower
    is better) and returns the best k swaps.  Candidates are processed in chunks of `chunk` rows: codae_swap_build
    writes the swapped outfits straight into the first activation buffer, the model's Linear layers run on them,
    codae_swap_error_topk reduces each chunk to k candidates and codae_topk_merge combines chunks (and ranks)."""

    def __init__(self, model, catalog, embedding_size, k=10, inv_scale=1.0, row_offset=0, chunk=8192, process_group=None,
                 allowed=None):
        """allowed: bool / uint8 [n_local] CUDA tensor, the candidates of this shard that may be returned (None: all)."""
        if not catalog.is_cuda:
            raise RuntimeError("codae: catalog is not on a CUDA device; the B200 path has no CPU fallback")
        model._require_cuda()
        self.model, self.catalog, self.E, self.k = model, catalog, embedding_size, k
        self.inv_scale, self.row_offset, self.chunk, self.pg = float(inv_scale), int(row_offset), int(chunk), process_group
        self.io = model.dims[0][0]
        if self.io % self.E != 0 or catalog.shape[1] < self.E:
            raise Exception("Catalog width or embedding size does not fit the model input.")
        dev = catalog.device
        self.allowed = _allowed_mask(allowed, catalog.shape[0], dev)
        self._ws = _C.score_topk_workspace(dev, 1, k)
        self._dae = _DaeChunks(model, self.chunk, self.io, dev)

    def _buffers(self):
        """(engine, activations, fp32 stage or None) of the swapped-outfit chunks."""
        return self._dae.buffers()

    def topk_local(self, outfit, slot, exclude=None):
        """outfit: [io] scaled fp32 row.  Returns (errors [k], global candidate indices [k]) of this shard.  exclude: int64
        [m] CUDA tensor of global candidate indices not to return (-1 padding, m <= 256), e.g. the item already in the slot."""
        dev = self.catalog.device
        if not 0 <= slot < self.io // self.E:
            raise Exception("Slot out of range.")
        ex = _exclusions(exclude, None, dev)
        outfit = outfit.to(torch.float32).contiguous().view(-1)
        eng, acts, stage, wflat = self._dae.prepare()
        n = self.catalog.shape[0]
        n_chunks = max(1, (n + self.chunk - 1) // self.chunk)
        ls = torch.full((n_chunks, 1, self.k), float("inf"), dtype=torch.float32, device=dev)
        li = torch.full((n_chunks, 1, self.k), -1, dtype=torch.int64, device=dev)
        for c in range(n_chunks if n else 0):
            first = c * self.chunk
            B = min(self.chunk, n - first)
            if stage is None:
                _C.swap_build(outfit, self.catalog, first, B, self.E, slot, self.io, self.inv_scale, acts[0])
            else:
                _C.swap_build(outfit, self.catalog, first, B, self.E, slot, self.io, self.inv_scale, stage)
                _C.split_x3(stage, acts[0])
            self._dae.forward(eng, acts, wflat, B)
            _C.swap_error_topk(outfit, self.catalog, first, B, self.E, slot, self.io, self.inv_scale, acts[-1],
                               self.row_offset, self.k, ls[c, 0], li[c, 0], self._ws, allow=self.allowed, exclude=ex)
        out_s = torch.empty((1, self.k), dtype=torch.float32, device=dev)
        out_i = torch.empty((1, self.k), dtype=torch.int64, device=dev)
        _C.topk_merge(ls, li, _C.METRIC_SQERR, out_s, out_i)
        return out_s[0], out_i[0]

    def topk(self, outfit, slot, exclude=None):
        s, i = self.topk_local(outfit, slot, exclude)
        s, i = _gather_merge(self.pg, s.view(1, -1), i.view(1, -1), _C.METRIC_SQERR)
        return s[0], i[0]

    def _owned_positions(self, candidates):
        """Positions (ascending, int64) in the flattened [Q, m] list of the entries this shard scores: not padding, inside
        [row_offset, row_offset + n_local), allowed.  nonzero() reads the count back: one host synchronisation."""
        n = self.catalog.shape[0]
        flat = candidates.reshape(-1)
        r = flat - self.row_offset
        own = (flat >= 0) & (r >= 0) & (r < n)
        if self.allowed is not None and n > 0:
            own &= self.allowed[r.clamp(0, n - 1)].bool()
        return torch.nonzero(own).view(-1)

    def rerank_local(self, outfits, slot, candidates):
        """Re-rank per-outfit candidate lists by swap error.  outfits: [Q, io] scaled fp32 rows on the catalog's device;
        candidates: int64 [Q, m] CUDA tensor of GLOBAL catalog row ids (< 0: padding; every rank gets the same tensor).
        Returns (errors [Q, k] f32, global ids [Q, k] i64) of the listed pairs this shard holds, best first, ties -> lower id,
        unused slots (+inf, -1); rows outside the shard, padding and rows `allowed` forbids are not scored, NaN errors never
        rank, a duplicated id is returned once per listing.  The owned pairs go through the DAE in chunks of `chunk` rows,
        whatever outfits they belong to; a pair's error is computed as topk_local computes it (bit for bit when the chunk
        shapes coincide).  Synchronises once (_owned_positions)."""
        dev = self.catalog.device
        if not 0 <= slot < self.io // self.E:
            raise Exception("Slot out of range.")
        outfits, cand = _pair_lists(outfits, candidates, self.io, dev)
        Q, mm = cand.shape
        pos = self._owned_positions(cand)
        err = torch.full((Q * mm,), float("nan"), dtype=torch.float32, device=dev)
        eng, acts, stage, wflat = self._dae.prepare()      # on every rank, pairs or not: sync_weights may be a collective
        for c0 in range(0, pos.numel(), self.chunk):
            pc = pos[c0:c0 + self.chunk]
            _C.swap_build_pairs(outfits, self.catalog, self.row_offset, cand, pc, self.E, slot, self.io, self.inv_scale,
                                acts[0] if stage is None else stage)
            if stage is not None:
                _C.split_x3(stage, acts[0])
            self._dae.forward(eng, acts, wflat, pc.numel())
            _C.swap_error_pairs(outfits, self.catalog, self.row_offset, cand, pc, self.E, slot, self.io, self.inv_scale, acts[-1],
                                err)
        out_s = torch.empty((Q, self.k), dtype=torch.float32, device=dev)
        out_i = torch.empty((Q, self.k), dtype=torch.int64, device=dev)
        _C.swap_pairs_topk(err, cand, self.k, out_s, out_i)
        return out_s, out_i

    def rerank(self, outfits, slot, candidates):
        """Global rerank_local: every rank scores the listed rows it holds, then all-gather of k entries per outfit and the
        deterministic merge (codae_topk_merge)."""
        return _gather_merge(self.pg, *self.rerank_local(outfits, slot, candidates), _C.METRIC_SQERR)


def _outfit_rows(outfits, io, device):
    """CompatibilityScorer's input: outfits fp32 [Q, io], Q >= 1, on the model's device; a contiguous copy."""
    if not isinstance(outfits, torch.Tensor) or outfits.dtype != torch.float32:
        raise RuntimeError("codae: outfits must be a float32 tensor")
    if outfits.dim() != 2 or outfits.shape[1] != io or outfits.shape[0] < 1:
        raise RuntimeError("codae: outfits must have shape [Q, %d] with Q >= 1, got %s" % (io, tuple(outfits.shape)))
    if not outfits.is_cuda or outfits.device != device:
        raise RuntimeError("codae: outfits must be on the model's device %s" % device)
    return outfits.contiguous()


class CompatibilityScorer:
    """Outfit compatibility by leave-one-slot-out reconstruction: for every slot s of a complete outfit, slot s is hidden
    (multiplied by 0, as model.corrupt does), the DAE reconstructs the outfit and the squared distance of the reconstructed slot s
    from the item that was there is slot_err[s].  A compatible outfit has small errors (score = their sum); the slot of the largest
    error holds the odd item out.  Every (outfit, slot) row is an independent DAE forward: a chunk of chunk // S whole outfits is
    S codae_corrupt_fwd launches into the first activation buffer (rows slot-major), the model's Linear layers, then
    codae_outfit_loo_error (include/codae_b200.h)."""

    def __init__(self, model, embedding_size, chunk=8192, process_group=None):
        model._require_cuda()
        self.model, self.E, self.pg = model, int(embedding_size), process_group
        self.io = model.dims[0][0]
        if self.io % self.E != 0:
            raise Exception("Embedding size does not divide the model input.")
        self.S = self.io // self.E
        if chunk < self.S:
            raise Exception("chunk %d holds no whole outfit of %d slots." % (chunk, self.S))
        self.chunk_outfits = int(chunk) // self.S
        dev = self.device = model.flat.device
        S = self.S
        # codae_corrupt_fwd's tables: observation i gets mask s in run s, mask s zeroes variable s, column c is variable c / E
        self._mask_table = torch.arange(S, dtype=torch.int16, device=dev).repeat(self.chunk_outfits, 1)
        self._mask_bits = torch.bitwise_left_shift(torch.ones(S, dtype=torch.int64, device=dev), torch.arange(S, device=dev))
        self._col_var = torch.div(torch.arange(self.io, device=dev), self.E, rounding_mode="floor").to(torch.uint8)
        self._dae = _DaeChunks(model, self.chunk_outfits * S, self.io, dev)
        self._out = None

    def _outputs(self, Q):
        if self._out is None or self._out[0].shape[0] != Q:
            dev = self.device
            self._out = (torch.empty((Q, self.S), dtype=torch.float32, device=dev), torch.empty(Q, dtype=torch.float32, device=dev),
                         torch.empty(Q, dtype=torch.int64, device=dev))
        return self._out

    def score_local(self, outfits):
        """outfits: [Q, io] scaled fp32 rows on the model's device.  Returns (slot_err [Q, S] f32, score [Q] f32, odd [Q] int64):
        lower score = more compatible; odd = the slot of largest error (ties -> lower slot); an outfit with a NaN error gets a NaN
        score and odd -1.  Asynchronous (no host synchronisation); the returned tensors are reused by the next call."""
        x = _outfit_rows(outfits, self.io, self.device)
        Q, S = x.shape[0], self.S
        err, score, odd = self._outputs(Q)
        eng, acts, stage, wflat = self._dae.prepare()
        for c0 in range(0, Q, self.chunk_outfits):
            Bq = min(self.chunk_outfits, Q - c0)
            rows = x[c0:c0 + Bq]
            dst = acts[0] if stage is None else stage
            for s in range(S):
                _C.corrupt_fwd(rows, None, Bq, self._mask_table, s, self._mask_bits, self._col_var, self.io, dst[s * Bq:(s + 1) * Bq])
            if stage is not None:
                _C.split_x3(stage, acts[0])
            self._dae.forward(eng, acts, wflat, S * Bq)
            _C.outfit_loo_error(rows, S, self.E, acts[-1], err[c0:c0 + Bq], score[c0:c0 + Bq], odd[c0:c0 + Bq])
        return err, score, odd

    def score(self, outfits):
        """score_local over the ranks of the process group: every rank is given the same outfits, rank r scores its
        shard_rows(Q, G, r) slice, and the slices are all-gathered (padded to ceil(Q / G) rows) into the full results."""
        import torch.distributed as dist
        pg = self.pg
        if pg is None and not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
            return self.score_local(outfits)
        x = _outfit_rows(outfits, self.io, self.device)
        Q, S, dev = x.shape[0], self.S, self.device
        G, r = dist.get_world_size(pg), dist.get_rank(pg)
        lo, n = shard_rows(Q, G, r)
        per = (Q + G - 1) // G
        err = torch.full((per, S), float("nan"), dtype=torch.float32, device=dev)
        score = torch.full((per,), float("nan"), dtype=torch.float32, device=dev)
        odd = torch.full((per,), -1, dtype=torch.int64, device=dev)
        if n:
            e, s, o = self.score_local(x[lo:lo + n])
            err[:n], score[:n], odd[:n] = e, s, o
        else:
            self.model.sync_weights()      # a collective under a sharded data-parallel trainer: every rank takes part
        out = []
        for t in (err, score, odd):
            g = torch.empty((G * per,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
            dist.all_gather_into_tensor(g, t, group=pg)
            out.append(g[:Q])
        return tuple(out)


def compatibility_auc(pos_score, neg_score):
    """Outfit compatibility AUC: the probability that a real outfit (pos_score) scores lower -- more compatible -- than a negative
    one (neg_score), ties counting 1/2; the rank-sum (Mann-Whitney) form with average ranks for ties.  NaN scores are dropped.
    Returns a Python float (NaN when either side is empty after dropping)."""
    pos = pos_score.reshape(-1).double()
    neg = neg_score.reshape(-1).double()
    pos, neg = pos[~torch.isnan(pos)], neg[~torch.isnan(neg)]
    n_p, n_n = pos.numel(), neg.numel()
    if n_p == 0 or n_n == 0:
        return float("nan")
    # rank of every value among both sets by DESCENDING score (1 = highest), ties averaged: a real outfit below a negative one
    # gets the larger rank; U = sum of the real outfits' ranks - n_p (n_p + 1) / 2 counts the pairs (real < negative) + ties / 2
    allv = torch.cat([pos, neg])
    vals, inv, counts = torch.unique(-allv, sorted=True, return_inverse=True, return_counts=True)
    last = torch.cumsum(counts, 0).double()
    avg = last - (counts.double() - 1) / 2
    rank_pos = avg[inv[:n_p]].sum()
    u = rank_pos - n_p * (n_p + 1) / 2
    return float(u / (n_p * n_n))
