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

OutfitCompleter fills every empty slot of a partial outfit together ("I have a top, complete the outfit"): candidates per missing
slot from the slot readings, then every combination of them scored by the swap error of the completed outfit -- or, where there are
too many combinations, a beam search that fills the missing slots one at a time and keeps the best `width` partial outfits after
each (complete_beam).  For a complete outfit it answers "which one item should I replace, and with what?" (revise): candidates for
every slot from its leave-one-slot-out reading, then every single-item replacement scored by swap error against the outfit as given.
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


def predict_missing(model, outfits, missing, embedding_size):
    """Zero every missing slot (missing: bool [Q, S]) of the (scaled) outfit rows [Q, S E] through model.corrupt, run the DAE once,
    return the reconstructions [Q, S E]."""
    mask = (~missing).to(torch.float32).repeat_interleave(embedding_size, dim=1)
    with torch.no_grad():
        return model(model.corrupt(input_data=outfits, mask=mask))


def predict_slot(model, outfits, slot, embedding_size):
    """Zero slot `slot` of the (scaled) outfit rows, run the DAE, return the reconstructed slot [Q, E]."""
    E = embedding_size
    missing = torch.zeros((outfits.shape[0], outfits.shape[1] // E), dtype=torch.bool, device=outfits.device)
    missing[:, slot] = True
    return predict_missing(model, outfits, missing, E)[:, slot * E:(slot + 1) * E].contiguous()


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
        self._loo(x, lambda c0, Bq, y: _C.outfit_loo_error(x[c0:c0 + Bq], S, self.E, y, err[c0:c0 + Bq], score[c0:c0 + Bq],
                                                           odd[c0:c0 + Bq]))
        return err, score, odd

    def _loo(self, x, on_chunk):
        """The leave-one-slot-out forward of the outfit rows x [Q, io] in chunks of chunk_outfits whole outfits: on_chunk(c0, Bq, y)
        receives each chunk's reconstructions y, slot-major (row s Bq + i is outfit c0 + i with slot s hidden)."""
        Q, S = x.shape[0], self.S
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
            on_chunk(c0, Bq, acts[-1])

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


def _is_distributed(pg):
    import torch.distributed as dist
    return pg is not None or (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1)


def _exchange_pool(pool, pool_id, pg):
    """Every rank's pool rows summed into every rank with one all_reduce(SUM) over int32 views.  Each row has exactly one owner and
    every other rank holds zeros there, so the sum is the owner's bits (-0.0, NaN and inf included).  pool_id travels as id + 1, so
    a row no rank owns comes back as -1."""
    import torch.distributed as dist
    R = pool_id.numel()
    buf = torch.cat([torch.where(pool_id >= 0, pool_id + 1, 0).view(torch.int32), pool.reshape(-1).view(torch.int32)])
    dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=pg)
    return buf[2 * R:].view(torch.float32).view(pool.shape), buf[:2 * R].view(torch.int64) - 1


class OutfitCompleter:
    """Outfit completion: every empty slot of a partial outfit filled together.  Stage 1 takes, for each missing slot, the best
    `depth` catalog rows by `metric` against the DAE's reading of that slot with all missing slots hidden (predict_missing, then
    ComplementarityScorer per slot).  Stage 2 scores every combination of those candidates -- depth^m_q of them for an outfit
    missing m_q slots -- by the swap error of the completed outfit, || DAE(x') - x' ||^2 over all io columns, and keeps the best k.
    The combinations of all outfits go through the model's GEMM chain in chunks of `chunk` rows (codae_complete_build, the Linear
    layers, codae_complete_error) and are ranked by codae_swap_pairs_topk; with one missing slot this is SwapScorer.rerank's
    arithmetic, bit for bit (include/codae_b200.h: outfit completion).

    complete_beam replaces stage 2's depth^m_q combinations by a beam search of m_q W depth rows per outfit: the missing slots are
    filled one level at a time in ascending slot order, each level scores every child of the W kept partial outfits by its partial
    error (the swap error over the given slots and the slots filled so far, the later missing slots hidden as +0.0) and keeps the best
    W by (error, combination index) (include/codae_b200.h: beam completion).  When the beam holds every combination it is
    complete's search, bit for bit at chunks of <= 128 rows.

    revise takes complete outfits and returns the single-item replacements that lower the swap error: stage 1 reads every slot with
    only that slot hidden (CompatibilityScorer's pass) and takes `depth` candidates per slot; stage 2 scores the outfit as given and
    every (slot, candidate) swap through the GEMM chain (codae_revise_build, the Linear layers, codae_revise_error) and keeps the
    best k swaps below the outfit's own error (include/codae_b200.h: outfit revision)."""

    MAX_DEPTH = 128
    MAX_WIDTH = 128

    def __init__(self, model, catalogs, embedding_size, depth=8, k=10, metric="sqerr", inv_scale=1.0, row_offsets=None,
                 chunk=8192, process_group=None):
        """catalogs: S entries, entry s this rank's shard of slot s's catalog ([n_local, >= E] fp32 or bf16 CUDA tensor, rows
        row_offsets[s].. of the global catalog) or None when slot s cannot be completed.  inv_scale multiplies catalog values
        (1 / dataset.scale for un-scaled catalogs such as dataset.data_per_category).  Shards of one slot must not overlap."""
        model._require_cuda()
        if metric not in METRICS:
            raise Exception("Unknown metric.")
        self.model, self.E, self.pg = model, int(embedding_size), process_group
        self.io = model.dims[0][0]
        if self.io % self.E != 0:
            raise Exception("Embedding size does not divide the model input.")
        self.S = S = self.io // self.E
        if not 1 <= depth <= self.MAX_DEPTH:
            raise RuntimeError("codae: depth %d outside [1, %d]" % (depth, self.MAX_DEPTH))
        if not 1 <= k <= 128:
            raise RuntimeError("codae: k %d outside [1, 128]" % k)
        if chunk < 1:
            raise RuntimeError("codae: chunk %d < 1" % chunk)
        if len(catalogs) != S:
            raise RuntimeError("codae: %d catalogs for %d slots" % (len(catalogs), S))
        row_offsets = [0] * S if row_offsets is None else [int(o) for o in row_offsets]
        if len(row_offsets) != S:
            raise RuntimeError("codae: %d row offsets for %d slots" % (len(row_offsets), S))
        self.device = dev = model.flat.device
        for s, cat in enumerate(catalogs):
            if cat is None:
                continue
            if not isinstance(cat, torch.Tensor) or cat.dtype not in (torch.float32, torch.bfloat16):
                raise RuntimeError("codae: catalog %d must be a float32 or bfloat16 tensor" % s)
            if cat.dim() != 2 or cat.shape[1] < self.E:
                raise RuntimeError("codae: catalog %d must have shape [n, >= %d], got %s" % (s, self.E, tuple(cat.shape)))
            if not cat.is_cuda or cat.device != dev:
                raise RuntimeError("codae: catalog %d must be on the model's device %s" % (s, dev))
        self.catalogs, self.row_offsets = list(catalogs), row_offsets
        self.depth, self.k, self.inv_scale, self.chunk = int(depth), int(k), float(inv_scale), int(chunk)
        self._scorers = [None if cat is None else
                         ComplementarityScorer(cat, self.E, metric=metric, k=self.depth, inv_scale=inv_scale, row_offset=off,
                                               process_group=process_group)
                         for cat, off in zip(catalogs, row_offsets)]
        self._dae = _DaeChunks(model, self.chunk, self.io, dev)
        self._has_catalog = torch.tensor([cat is not None for cat in catalogs], dtype=torch.bool, device=dev)
        self._compat = None         # revise's stage 1: a CompatibilityScorer, made on first use

    def _inputs(self, outfits, missing, candidates):
        """outfits fp32 [Q, io], missing bool [Q, S] and candidates int64 [Q, S, m] (1 <= m <= 128, or None) on the model's device;
        contiguous copies."""
        x = _outfit_rows(outfits, self.io, self.device)
        Q = x.shape[0]
        return x, self._slot_mask(missing, Q, "missing"), self._candidate_lists(candidates, Q)

    def _slot_mask(self, mask, Q, name):
        """bool [Q, S] on the model's device; a contiguous copy."""
        S = self.S
        if not isinstance(mask, torch.Tensor) or mask.dtype != torch.bool:
            raise RuntimeError("codae: %s must be a bool tensor" % name)
        if tuple(mask.shape) != (Q, S):
            raise RuntimeError("codae: %s must have shape [%d, %d], got %s" % (name, Q, S, tuple(mask.shape)))
        if not mask.is_cuda or mask.device != self.device:
            raise RuntimeError("codae: %s must be on the model's device %s" % (name, self.device))
        return mask.contiguous()

    def _candidate_lists(self, candidates, Q):
        """int64 [Q, S, m] (1 <= m <= 128) on the model's device, or None; a contiguous copy."""
        S = self.S
        if candidates is not None:
            if not isinstance(candidates, torch.Tensor) or candidates.dtype != torch.int64:
                raise RuntimeError("codae: candidates must be an int64 tensor")
            if (candidates.dim() != 3 or tuple(candidates.shape[:2]) != (Q, S)
                    or not 1 <= candidates.shape[2] <= self.MAX_DEPTH):
                raise RuntimeError("codae: candidates must have shape [%d, %d, m] with 1 <= m <= %d, got %s"
                                   % (Q, S, self.MAX_DEPTH, tuple(candidates.shape)))
            if not candidates.is_cuda or candidates.device != self.device:
                raise RuntimeError("codae: candidates must be on the model's device %s" % self.device)
            candidates = candidates.contiguous()
        return candidates

    def _counts(self, missing):
        """(outfits missing each slot [S], max m_q, outfits missing nothing): one host synchronisation; RuntimeError for a missing slot
        without a catalog."""
        m_q = missing.sum(1)
        stats = torch.cat([missing.sum(0), m_q.max().view(1), (m_q == 0).sum().view(1)]).tolist()
        counts, m_max, n_full = [int(v) for v in stats[:-2]], int(stats[-2]), int(stats[-1])
        for s, n in enumerate(counts):
            if n and self.catalogs[s] is None:
                raise RuntimeError("codae: slot %d is missing in %d outfits but has no catalog" % (s, n))
        return counts, m_max, n_full

    def _limits(self, missing, depth):
        """(outfits missing each slot [S], max m_q, C = depth^max m_q): one host synchronisation; RuntimeError past a limit."""
        Q = missing.shape[0]
        counts, m_max, _ = self._counts(missing)
        C = depth ** m_max
        if C > _C.COMPLETE_MAX_COMBOS:
            raise RuntimeError("codae: %d combinations per outfit (depth %d ^ %d missing slots) exceed %d" % (C, depth, m_max,
                                                                                                        _C.COMPLETE_MAX_COMBOS))
        if Q * C > 2 ** 31 - 1:
            raise RuntimeError("codae: Q * combinations = %d exceeds 2**31 - 1" % (Q * C))
        return counts, m_max, C

    def _candidates(self, x, missing, counts):
        Q, S, E = x.shape[0], self.S, self.E
        y = predict_missing(self.model, x, missing, E)
        cand = torch.full((Q, S, self.depth), -1, dtype=torch.int64, device=self.device)
        for s in range(S):
            if not counts[s]:
                continue
            rows = torch.nonzero(missing[:, s]).view(-1)          # the slot's one host synchronisation
            query = y.index_select(0, rows)[:, s * E:(s + 1) * E]
            sc = self._scorers[s]
            _, idx = sc.topk_batched(query) if rows.numel() >= ComplementarityScorer.TC_MIN_Q else sc.topk(query)
            cand[rows, s] = idx
        return cand

    def candidates(self, outfits, missing):
        """Stage 1 alone: int64 [Q, S, depth] global row ids, for each missing slot the best `depth` rows of its catalog against
        predict_missing's reading of the slot (ComplementarityScorer.topk, or topk_batched from TC_MIN_Q outfits up), best first;
        -1 for given slots and where a catalog has fewer than `depth` rows.  A collective under a process group."""
        x, miss, _ = self._inputs(outfits, missing, None)
        counts, _, _ = self._limits(miss, self.depth)
        return self._candidates(x, miss, counts)

    def _beam_candidates(self, outfits, missing):
        """Stage 1 for complete_beam: candidates() without the exhaustive cap on depth^m_q."""
        x, miss, _ = self._inputs(outfits, missing, None)
        counts, _, _ = self._counts(miss)
        return self._candidates(x, miss, counts)

    def _pool(self, missing, cand, counts, depth):
        """The candidate rows this process holds: (slot_base [Q, S] int64, pool [R, E] f32 un-scaled, pool_id [R] int64).  The
        missing (outfit, slot) pairs are numbered slot-major; pair i owns pool rows [i depth, (i + 1) depth), one per candidate.
        Rows outside this process's shards, and padding, are zeros with pool_id -1."""
        Q, S, E, dev = missing.shape[0], self.S, self.E, self.device
        nm = sum(counts)
        t = torch.nonzero_static(missing.t().reshape(-1), size=nm).view(-1)      # s Q + q, slot-major
        pair_q, pair_s = t % Q, torch.div(t, Q, rounding_mode="floor")
        slot_base = torch.full((Q, S), -1, dtype=torch.int64, device=dev)
        slot_base[pair_q, pair_s] = torch.arange(nm, dtype=torch.int64, device=dev) * depth
        R = max(1, nm * depth)
        pool = torch.zeros((R, E), dtype=torch.float32, device=dev)
        pool_id = torch.full((R,), -1, dtype=torch.int64, device=dev)
        ids = cand[pair_q, pair_s]                                               # [nm, depth]
        off = 0
        for s in range(S):
            n = counts[s]
            if n and self.catalogs[s].shape[0]:
                cat, n_local = self.catalogs[s], self.catalogs[s].shape[0]
                g = ids[off:off + n].reshape(-1)
                r = g - self.row_offsets[s]
                own = (g >= 0) & (r >= 0) & (r < n_local)
                rows = cat[:, :E].index_select(0, r.clamp(0, n_local - 1)).to(torch.float32)   # bf16 -> fp32 is exact
                pool[off * depth:(off + n) * depth] = torch.where(own.view(-1, 1), rows, 0.0)
                pool_id[off * depth:(off + n) * depth] = torch.where(own, g, -1)
            off += n
        return slot_base, pool, pool_id

    def _through_dae(self, prep, pos, build, error):
        """The rows pos (int64 positions) through the DAE in chunks of `chunk`: build(pc, dst) writes a chunk's rows into dst, the
        fp32-parity engine splits them into its planes, the Linear layers run and error(pc, y) reads the reconstructions y.  prep is
        _DaeChunks.prepare()'s result."""
        eng, acts, stage, wflat = prep
        for c0 in range(0, pos.numel(), self.chunk):
            pc = pos[c0:c0 + self.chunk]
            build(pc, acts[0] if stage is None else stage)
            if stage is not None:
                _C.split_x3(stage, acts[0])
            self._dae.forward(eng, acts, wflat, pc.numel())
            error(pc, acts[-1])

    @staticmethod
    def _missing_bases(missing, slot_base, m_max):
        """[Q, m_max + 1] int64: pool row of candidate 0 of each outfit's j-th missing slot (-1 past its m_q)."""
        base_j = torch.full((missing.shape[0], m_max + 1), -1, dtype=torch.int64, device=missing.device)
        base_j.scatter_(1, torch.where(missing, torch.cumsum(missing, 1) - 1, m_max), slot_base)
        return base_j

    def _stage2(self, x, missing, slot_base, pool, pool_id, depth, m_max, C):
        """Every valid combination of every outfit through the DAE; (err [Q, k] f32, ids [Q, k, S] int64), best first."""
        Q, S, E, dev = x.shape[0], self.S, self.E, self.device
        R = pool_id.numel()
        base_j = self._missing_bases(missing, slot_base, m_max)
        cidx = torch.arange(C, dtype=torch.int64, device=dev)
        valid = torch.ones((Q, C), dtype=torch.bool, device=dev)
        for j in range(m_max):
            digit = torch.div(cidx, depth ** j, rounding_mode="floor") % depth
            row = base_j[:, j:j + 1] + digit
            held = (row < R) & (pool_id[row.clamp(0, R - 1)] >= 0)
            valid &= torch.where(base_j[:, j:j + 1] >= 0, held, digit == 0)
        combo = torch.where(valid, cidx, -1)
        pos = torch.nonzero(valid.view(-1)).view(-1)                  # stage 2's one host synchronisation
        err = torch.full((Q * C,), float("nan"), dtype=torch.float32, device=dev)
        prep = self._dae.prepare()      # on every rank, combinations or not: sync_weights may be a collective
        self._through_dae(prep, pos,
                          lambda pc, dst: _C.complete_build(x, S, E, slot_base, pool, pool_id, depth, C, pc, self.inv_scale, dst),
                          lambda pc, y: _C.complete_error(x, S, E, slot_base, pool, pool_id, depth, C, pc, self.inv_scale, y, err))
        out_s = torch.empty((Q, self.k), dtype=torch.float32, device=dev)
        out_c = torch.empty((Q, self.k), dtype=torch.int64, device=dev)
        _C.swap_pairs_topk(err, combo, self.k, out_s, out_c)
        return out_s, _decode_combinations(out_c, slot_base, pool_id, depth)

    def complete_local(self, outfits, missing, candidates):
        """Stage 2 for a process that holds every listed row.  outfits [Q, io] scaled fp32, missing bool [Q, S], candidates int64
        [Q, S, m] global row ids (< 0: padding; entries of given slots are ignored); depth = m.  Returns (err [Q, k] f32, ids
        [Q, k, S] int64), best first by (error, combination index); ids are -1 in given slots, unused entries (+inf, -1...).
        Combinations taking a padding id or a row outside this process's shards are not scored; NaN errors never rank."""
        x, miss, cand = self._inputs(outfits, missing, candidates)
        if cand is None:
            raise RuntimeError("codae: candidates must be an int64 tensor")
        depth = cand.shape[2]
        counts, m_max, C = self._limits(miss, depth)
        return self._stage2(x, miss, *self._pool(miss, cand, counts, depth), depth, m_max, C)

    def complete(self, outfits, missing, candidates=None):
        """Fill every missing slot: (err [Q, k] f32, ids [Q, k, S] int64) as complete_local.  Without candidates stage 1 runs first
        (depth from the constructor).  Under a process group every rank is given the same inputs: the candidate pool is assembled
        from every rank's shards (_exchange_pool), rank r scores its shard_rows(Q, G, r) outfits and the slices are all-gathered."""
        if candidates is None:
            candidates = self.candidates(outfits, missing)
        if not _is_distributed(self.pg):
            return self.complete_local(outfits, missing, candidates)
        x, miss, cand = self._inputs(outfits, missing, candidates)
        depth = cand.shape[2]
        counts, m_max, C = self._limits(miss, depth)
        slot_base, pool, pool_id = self._pool(miss, cand, counts, depth)
        pool, pool_id = _exchange_pool(pool, pool_id, self.pg)
        return self._sharded(x.shape[0], lambda lo, n: self._stage2(x[lo:lo + n], miss[lo:lo + n], slot_base[lo:lo + n], pool,
                                                                    pool_id, depth, m_max, C))

    def _sharded(self, Q, run, results=None):
        """Under a process group: run(lo, n) on this rank's shard_rows(Q, G, r) slice of the outfits, then the slices all-gathered
        (padded to ceil(Q / G) rows) into the full results.  results: (per-outfit shape, dtype, fill) of each tensor run returns,
        by default complete's (err [n, k] f32, ids [n, k, S] int64)."""
        import torch.distributed as dist
        dev = self.device
        if results is None:
            results = (((self.k,), torch.float32, float("inf")), ((self.k, self.S), torch.int64, -1))
        G, r = dist.get_world_size(self.pg), dist.get_rank(self.pg)
        lo, n = shard_rows(Q, G, r)
        per = (Q + G - 1) // G
        outs = [torch.full((per,) + shape, fill, dtype=dtype, device=dev) for shape, dtype, fill in results]
        if n:
            for t, v in zip(outs, run(lo, n)):
                t[:n] = v
        else:
            self.model.sync_weights()      # a collective under a sharded data-parallel trainer: every rank takes part
        out = []
        for t in outs:
            g = torch.empty((G * per,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
            dist.all_gather_into_tensor(g, t, group=self.pg)
            out.append(g[:Q])
        return tuple(out)

    def _check_width(self, width):
        if not 1 <= width <= self.MAX_WIDTH:
            raise RuntimeError("codae: beam width %d outside [1, %d]" % (width, self.MAX_WIDTH))
        if self.k > width:
            raise RuntimeError("codae: k %d exceeds the beam width %d" % (self.k, width))

    def _beam_limits(self, missing, depth, width):
        """complete_beam's limits: (outfits missing each slot [S], max m_q, outfits missing nothing); one host synchronisation;
        RuntimeError past a limit."""
        self._check_width(width)
        Q = missing.shape[0]
        if Q * width * depth > 2 ** 31 - 1:
            raise RuntimeError("codae: Q * width * depth = %d exceeds 2**31 - 1" % (Q * width * depth))
        counts, m_max, n_full = self._counts(missing)
        if depth ** m_max > 2 ** 62:
            raise RuntimeError("codae: depth %d ^ %d missing slots exceeds 2**62 (the beam's combination keys are int64)"
                               % (depth, m_max))
        return counts, m_max, n_full

    def _beam(self, x, missing, slot_base, pool, pool_id, depth, m_max, n_full, width):
        """Beam search over the missing slots of every outfit; (err [Q, k] f32, ids [Q, k, S] int64), best first.  n_full bounds the
        outfits missing nothing (their count, or more: extra positions are padding)."""
        Q, S, E, W, k, dev = x.shape[0], self.S, self.E, width, self.k, self.device
        R = pool_id.numel()
        inv = self.inv_scale
        m_q = missing.sum(1)
        base_j = self._missing_bases(missing, slot_base, m_max)
        prep = self._dae.prepare()      # on every rank, rows or not: sync_weights may be a collective
        err_f = torch.full((Q, k), float("inf"), dtype=torch.float32, device=dev)
        c_f = torch.full((Q, k), -1, dtype=torch.int64, device=dev)
        if n_full:
            # outfits missing nothing: complete's answer, the outfit as given scored once (a [Q, 1] combination grid)
            pos = torch.nonzero_static(m_q == 0, size=min(n_full, Q), fill_value=-1).view(-1)
            e0 = torch.full((Q,), float("nan"), dtype=torch.float32, device=dev)
            self._through_dae(prep, pos, lambda pc, dst: _C.complete_build(x, S, E, slot_base, pool, pool_id, depth, 1, pc, inv, dst),
                              lambda pc, y: _C.complete_error(x, S, E, slot_base, pool, pool_id, depth, 1, pc, inv, y, e0))
            scored = e0 == e0                                       # NaN never ranks
            err_f[:, 0] = torch.where(scored, e0, float("inf"))
            c_f[:, 0] = torch.where(scored, 0, -1)
        beam = torch.full((Q, W), -1, dtype=torch.int64, device=dev)
        beam[:, 0] = 0
        b = torch.arange(depth, dtype=torch.int64, device=dev)
        for j in range(m_max):
            # child (q, t, b) = parent beam[q, t] + b depth^j; valid while the parent is, j < m_q and candidate b's row is held
            row = base_j[:, j:j + 1] + b
            held = (base_j[:, j:j + 1] >= 0) & (row < R) & (pool_id[row.clamp(0, R - 1)] >= 0)           # [Q, depth]
            valid = (beam >= 0).unsqueeze(2) & held.unsqueeze(1)                                         # [Q, W, depth]
            key = torch.where(valid, beam.unsqueeze(2) + b * depth ** j, -1).view(Q, W * depth)
            pos = torch.nonzero(valid.view(-1)).view(-1)            # the level's one host synchronisation
            err = torch.full((Q * W * depth,), float("nan"), dtype=torch.float32, device=dev)
            parents = beam
            self._through_dae(prep, pos,
                              lambda pc, dst: _C.complete_beam_build(x, S, E, slot_base, pool, pool_id, depth, parents, j, pc, inv,
                                                                     dst),
                              lambda pc, y: _C.complete_beam_error(x, S, E, slot_base, pool, pool_id, depth, parents, j, pc, inv, y,
                                                                   err))
            out_s = torch.empty((Q, W), dtype=torch.float32, device=dev)
            beam = torch.empty((Q, W), dtype=torch.int64, device=dev)
            _C.swap_pairs_topk(err, key, W, out_s, beam)
            done = (m_q == j + 1).view(Q, 1)                        # the outfits whose last level this is
            err_f = torch.where(done, out_s[:, :k], err_f)
            c_f = torch.where(done, beam[:, :k], c_f)
        return err_f, _decode_combinations(c_f, slot_base, pool_id, depth)

    def complete_beam_local(self, outfits, missing, candidates, width):
        """complete_local by beam search of width W = `width` (1 <= k <= W <= 128): the missing slots of each outfit are filled in
        ascending slot order, and after each the best W partial outfits are kept by (partial error, combination index).  The partial
        error is the swap error over the columns of the given slots and the slots filled so far; the later missing slots are hidden
        (+0.0 in the DAE input, not in the error).  Returns (err [Q, k] f32, ids [Q, k, S] int64) as complete_local: the first k of
        the last level's selection, whose errors are complete's errors of those combinations.  With W >= depth^(m_max - 1) nothing is
        pruned and, at chunks of <= 128 rows, the result is complete_local's bit for bit.  Synchronises once for the limits and once
        per level."""
        x, miss, cand = self._inputs(outfits, missing, candidates)
        if cand is None:
            raise RuntimeError("codae: candidates must be an int64 tensor")
        depth = cand.shape[2]
        counts, m_max, n_full = self._beam_limits(miss, depth, width)
        return self._beam(x, miss, *self._pool(miss, cand, counts, depth), depth, m_max, n_full, width)

    def complete_beam(self, outfits, missing, width, candidates=None):
        """complete_beam_local for any process: without candidates stage 1 runs first (depth from the constructor).  Under a process
        group every rank is given the same inputs, the candidate pool is assembled from every rank's shards, rank r searches its
        shard_rows(Q, G, r) outfits and the slices are all-gathered -- as complete does."""
        self._check_width(width)
        if candidates is None:
            candidates = self._beam_candidates(outfits, missing)
        if not _is_distributed(self.pg):
            return self.complete_beam_local(outfits, missing, candidates, width)
        x, miss, cand = self._inputs(outfits, missing, candidates)
        depth = cand.shape[2]
        counts, m_max, n_full = self._beam_limits(miss, depth, width)
        slot_base, pool, pool_id = self._pool(miss, cand, counts, depth)
        pool, pool_id = _exchange_pool(pool, pool_id, self.pg)
        return self._sharded(x.shape[0], lambda lo, n: self._beam(x[lo:lo + n], miss[lo:lo + n], slot_base[lo:lo + n], pool, pool_id,
                                                                  depth, m_max, n_full, width))

    def _revise_inputs(self, outfits, keep, exclude, candidates):
        """revise's inputs: outfits fp32 [Q, io], keep bool [Q, S], exclude int64 [Q, S, n] (1 <= n <= 256) and candidates int64
        [Q, S, m] (1 <= m <= 128), the last three optional, on the model's device; contiguous copies.  RuntimeError unless
        Q (1 + S depth) <= 2**31 - 1, depth = m or, without candidates, the constructor's."""
        x = _outfit_rows(outfits, self.io, self.device)
        Q, S = x.shape[0], self.S
        keep = None if keep is None else self._slot_mask(keep, Q, "keep")
        if exclude is not None:
            if not isinstance(exclude, torch.Tensor) or exclude.dtype != torch.int64:
                raise RuntimeError("codae: exclude must be an int64 tensor")
            if exclude.dim() != 3 or tuple(exclude.shape[:2]) != (Q, S) or not 1 <= exclude.shape[2] <= _C.TOPK_MAX_EXCLUDE:
                raise RuntimeError("codae: exclude must have shape [%d, %d, n] with 1 <= n <= %d, got %s"
                                   % (Q, S, _C.TOPK_MAX_EXCLUDE, tuple(exclude.shape)))
            if not exclude.is_cuda or exclude.device != self.device:
                raise RuntimeError("codae: exclude must be on the model's device %s" % self.device)
            exclude = exclude.contiguous()
        cand = self._candidate_lists(candidates, Q)
        depth = self.depth if cand is None else cand.shape[2]
        if Q * (1 + S * depth) > 2 ** 31 - 1:
            raise RuntimeError("codae: Q * (1 + S * depth) = %d exceeds 2**31 - 1" % (Q * (1 + S * depth)))
        return x, keep, exclude, cand

    def _revise_candidates(self, x, keep, exclude):
        """Stage 1 of revise: for every revisable (outfit, slot), the best `depth` rows of the slot's catalog against the reconstruction
        of that slot with only that slot hidden (CompatibilityScorer's leave-one-slot-out forward); one nonzero per slot with a
        catalog."""
        Q, S, E, dev = x.shape[0], self.S, self.E, self.device
        if self._compat is None:
            self._compat = CompatibilityScorer(self.model, E, chunk=max(self.chunk, S))
            if self.chunk >= S:
                self._compat._dae = self._dae       # its chunks of whole outfits fit this completer's activation buffers
        query = torch.empty((Q, S, E), dtype=torch.float32, device=dev)

        def take(c0, Bq, y):                        # y[s Bq + i, s E:(s + 1) E]: outfit c0 + i's slot s, read with slot s hidden
            query[c0:c0 + Bq] = torch.diagonal(y[:S * Bq, :self.io].reshape(S, Bq, S, E), dim1=0, dim2=2).permute(0, 2, 1)
        self._compat._loo(x, take)
        cand = torch.full((Q, S, self.depth), -1, dtype=torch.int64, device=dev)
        for s in range(S):
            if self.catalogs[s] is None:
                continue
            if keep is None:
                rows = torch.arange(Q, dtype=torch.int64, device=dev)
            else:
                rows = torch.nonzero(~keep[:, s]).view(-1)            # the slot's one host synchronisation
                if rows.numel() == 0:
                    continue
            ex = None if exclude is None else exclude[rows, s]
            sc = self._scorers[s]
            qs = query[rows, s]
            _, idx = sc.topk_batched(qs, ex) if rows.numel() >= ComplementarityScorer.TC_MIN_Q else sc.topk(qs, ex)
            cand[rows, s] = idx
        return cand

    def revise_candidates(self, outfits, keep=None, exclude=None):
        """Stage 1 of revise alone: int64 [Q, S, depth] global row ids.  For every slot s of outfit q that keep[q, s] does not keep and
        whose catalog is not None, the best `depth` rows of catalog s by `metric` against the DAE's reconstruction of slot s with only
        slot s hidden -- predict_slot(model, outfits, s, E)'s reading, computed by CompatibilityScorer's leave-one-slot-out pass --
        never returning the global ids exclude[q, s] (< 0: padding), best first (ComplementarityScorer.topk, or topk_batched from
        TC_MIN_Q outfits up); -1 for kept slots and padding.  A collective under a process group."""
        x, keep, exclude, _ = self._revise_inputs(outfits, keep, exclude, None)
        return self._revise_candidates(x, keep, exclude)

    def _revise_limits(self, cand):
        """(revised bool [Q, S], revised outfits per slot [S]): slot s of outfit q is revised when it has a catalog and its list holds
        an id >= 0.  One host synchronisation."""
        revised = (cand >= 0).any(2) & self._has_catalog
        return revised, [int(v) for v in revised.sum(0).tolist()]

    def _revise(self, x, slot_base, pool, pool_id, depth):
        """Stage 2: the grid [Q, 1 + S depth] of every outfit -- column 0 the outfit as given, column 1 + s depth + c slot s replaced by
        its candidate c -- through the DAE; (base [Q] f32, err [Q, k] f32, slot [Q, k] int64, ids [Q, k] int64)."""
        Q, S, k, dev = x.shape[0], self.S, self.k, self.device
        R = pool_id.numel()
        G = 1 + S * depth
        row = slot_base.unsqueeze(2) + torch.arange(depth, dtype=torch.int64, device=dev)                    # [Q, S, depth]
        held = (slot_base.unsqueeze(2) >= 0) & (row < R) & (pool_id[row.clamp(0, R - 1)] >= 0)
        valid = torch.cat([torch.ones((Q, 1), dtype=torch.bool, device=dev), held.view(Q, S * depth)], 1)
        # key s depth + c of column 1 + s depth + c; the base row and the rows not held never rank
        key = torch.where(held.view(Q, S * depth), torch.arange(S * depth, dtype=torch.int64, device=dev), -1)
        key = torch.cat([torch.full((Q, 1), -1, dtype=torch.int64, device=dev), key], 1)
        pos = torch.nonzero(valid.view(-1)).view(-1)                  # stage 2's one host synchronisation
        err = torch.full((Q * G,), float("nan"), dtype=torch.float32, device=dev)
        prep = self._dae.prepare()      # on every rank, rows or not: sync_weights may be a collective
        inv = self.inv_scale
        self._through_dae(prep, pos, lambda pc, dst: _C.revise_build(x, S, self.E, slot_base, pool, pool_id, depth, pc, inv, dst),
                          lambda pc, y: _C.revise_error(x, S, self.E, slot_base, pool, pool_id, depth, pc, inv, y, err))
        out_s = torch.empty((Q, k), dtype=torch.float32, device=dev)
        out_key = torch.empty((Q, k), dtype=torch.int64, device=dev)
        _C.swap_pairs_topk(err, key, k, out_s, out_key)
        base = err.view(Q, G)[:, 0].contiguous()
        better = out_s < base.unsqueeze(1)          # every improving swap ranks first: the cut is exact; a NaN base keeps nothing
        slot = torch.div(out_key, depth, rounding_mode="floor").clamp(min=0)
        ids = pool_id[(slot_base.gather(1, slot) + out_key - slot * depth).clamp(0, R - 1)]
        return (base, torch.where(better, out_s, float("inf")), torch.where(better, slot, -1), torch.where(better, ids, -1))

    def revise_local(self, outfits, candidates):
        """Stage 2 of revise for a process that holds every listed row.  outfits [Q, io] scaled fp32; candidates int64 [Q, S, m] global
        row ids (< 0: padding), depth = m; a slot whose list holds no id >= 0, or whose catalog is None, is not revised.  Every
        outfit is scored as given (base) and with each listed candidate of each revised slot swapped in, by the swap error
        || DAE(x') - x' ||^2 over all io columns.  Returns (base [Q] f32, err [Q, k] f32, slot [Q, k] int64, ids [Q, k] int64): the
        swaps of error strictly below base, best first by (error, s depth + c) -- ties to the lower slot, then to the earlier
        candidate --, unused entries (+inf, -1, -1).  A swap that leaves the outfit as it is (the held item proposed again) never
        lists; an outfit holding a NaN has a NaN base and no swaps.  Synchronises once for the limits and once for the grid."""
        x, _, _, cand = self._revise_inputs(outfits, None, None, candidates)
        if cand is None:
            raise RuntimeError("codae: candidates must be an int64 tensor")
        depth = cand.shape[2]
        revised, counts = self._revise_limits(cand)
        return self._revise(x, *self._pool(revised, cand, counts, depth), depth)

    def revise(self, outfits, keep=None, exclude=None, candidates=None):
        """Revise complete outfits: (base, err, slot, ids) as revise_local.  keep bool [Q, S]: slots that are not changed; without
        candidates stage 1 (revise_candidates, with the exclusion lists exclude) runs first, depth from the constructor.  Under a
        process group every rank is given the same inputs: the candidate pool is assembled from every rank's shards, rank r scores its
        shard_rows(Q, G, r) outfits and the slices are all-gathered -- as complete does."""
        x, keep, exclude, cand = self._revise_inputs(outfits, keep, exclude, candidates)
        if cand is None:
            cand = self._revise_candidates(x, keep, exclude)
        elif keep is not None:
            cand = torch.where(keep.unsqueeze(2), -1, cand)
        if not _is_distributed(self.pg):
            return self.revise_local(x, cand)
        depth = cand.shape[2]
        revised, counts = self._revise_limits(cand)
        slot_base, pool, pool_id = self._pool(revised, cand, counts, depth)
        pool, pool_id = _exchange_pool(pool, pool_id, self.pg)
        k = self.k
        return self._sharded(x.shape[0], lambda lo, n: self._revise(x[lo:lo + n], slot_base[lo:lo + n], pool, pool_id, depth),
                             (((), torch.float32, float("nan")), ((k,), torch.float32, float("inf")), ((k,), torch.int64, -1),
                              ((k,), torch.int64, -1)))


def _decode_combinations(combo, slot_base, pool_id, depth):
    """combo [Q, k] (combination indices, -1 unused) -> global ids [Q, k, S]: slot s of combination c is pool row slot_base[q, s] +
    (c / depth^j) % depth for the j-th missing slot s, -1 for given slots and unused entries."""
    R = pool_id.numel()
    miss = slot_base >= 0
    pw = torch.pow(depth, (torch.cumsum(miss, 1) - 1).clamp(min=0))                        # [Q, S]
    digit = torch.div(combo.clamp(min=0).unsqueeze(2), pw.unsqueeze(1), rounding_mode="floor") % depth
    row = (slot_base.unsqueeze(1) + digit).clamp(0, R - 1)
    return torch.where(miss.unsqueeze(1) & (combo >= 0).unsqueeze(2), pool_id[row], -1)
