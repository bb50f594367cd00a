"""Batched entry point of the engine: scores of MANY splits of one alignment in one call.

This is the call that replaces the reference's per-split loops

    for split in splitp.all_splits(tree):                     # README.md:37-41, examples/playground.py:29-39
        splitp.split_score(splitp.flattening(split, aln, FlatFormat.reduced))      # or subflattening(split, aln)

and the inner loop of `erickson_SVD` (phylogenetics.py:126-140).  `score_splits` takes the alignment as HOST data
(what `parsers.fasta.read_alignment_from_file` returns, or a byte / code matrix, or the 2-bit planes written by
`pack_planes_host`), copies it to the device, and returns one float64 score per split as a numpy array:

    Method.flattening     pack -> pattern count (kernel 1) -> per split: u8 scatter (kernel 2) -> exact integer Gram on the
                          tensor cores (kernel 4) -> eigen-solver (kernel 5); scores equal those of the reduced / dense /
                          sparse flattening (dropping all-zero rows and columns does not change the singular values)
                          (up to 16 taxa; 17..64 taxa: pattern count -> engine.sparse_flattening_scores, csrc/sparse.cu)
    Method.subflattening  pack -> pair tables -> H N H^T -> per split: gather + Gram + eigenvalues (kernel 3)
    Method.mutual_information  pattern count (uint64 keys up to 31 taxa; 32..64 taxa: pack_wide + count_patterns_wide) ->
                          engine.rank1_divergence_scores (csrc/mi_batch.cu): the rank-1 divergence of every split's flattening
                          of the pattern probabilities (count / usable sites), batches of splits per launch

Under `torch.distributed` (one process per GPU) the splits are dealt to the ranks for scoring (flattening scores: contiguous
runs of the size-class-ordered list cut at equal modelled cost; subflattening and divergence scores: round-robin) and every rank receives
the scores of all splits.  The counting stage has two forms: `sites="shard"` -- every rank passes ITS contiguous site
shard (distributed.shard_range) and the pattern tables are merged -- or `sites="replicated"` -- every rank passes the
WHOLE alignment and counts it itself, with no exchange at all.  The second form wins while counting the whole alignment
is cheaper than the exchange (`replicate_sites`: 12 taxa x 10^6 sites count in 0.16 ms, the list exchange between 8
ranks takes 1.5 ms).

`PhaseTimer` collects per-phase device time (CUDA events on the launch stream) for bench.py's `phase_ms`.
"""
from __future__ import annotations

from collections import namedtuple

import numpy as np
import torch

from . import engine
from .engine import PhaseTimer, _span  # noqa: F401  (PhaseTimer is re-exported: bench.py's `phase_ms`)
from .enums import Method


# --------------------------------------------------------------------------------------------
# host-side 2-bit format (what a FASTA -> packed converter would write once)
# --------------------------------------------------------------------------------------------
def pack_planes_host(codes):
    """uint8 [n, N] codes 0..3 (anything else = unusable site, fasta.py:55-57) -> (planes uint32 [n, 2, Wp],
    valid uint32 [Wp]) in the device layout of include/splitp_b200.h: 2 bits per base instead of 8."""
    codes = np.asarray(codes, dtype=np.uint8)
    n, N = codes.shape
    Wp = int(engine.lib.spb_plane_words(N))
    pad = Wp * 32 - N
    ok = (codes <= 3).all(axis=0)
    planes = np.zeros((n, 2, Wp), dtype=np.uint32)
    for t in range(n):
        row = np.where(ok, codes[t], 0)
        for bit in range(2):
            bits = np.concatenate([(row >> bit) & 1, np.zeros(pad, np.uint8)]).astype(np.uint8)
            planes[t, bit] = np.packbits(bits, bitorder="little").view(np.uint32)
    valid = np.packbits(np.concatenate([ok, np.zeros(pad, bool)]).astype(np.uint8), bitorder="little").view(np.uint32)
    return planes, valid.copy()


class HostPlanes:
    """2-bit packed alignment on the host (pinned when `pin=True`): the e2e input format of the subflattening path."""

    def __init__(self, planes, valid, n, N, pin=False):
        self.planes = torch.from_numpy(np.ascontiguousarray(planes).view(np.int32))
        self.valid = torch.from_numpy(np.ascontiguousarray(valid).view(np.int32))
        if pin:
            self.planes, self.valid = self.planes.pin_memory(), self.valid.pin_memory()
        self.n, self.N = int(n), int(N)

    @property
    def nbytes(self):
        return self.planes.numel() * 4 + self.valid.numel() * 4

    def to_device(self):
        dev = engine.device()
        return engine.DeviceAlignment(self.n, self.N, None, self.planes.to(dev, non_blocking=True),
                                      self.valid.to(dev, non_blocking=True))


# --------------------------------------------------------------------------------------------
def _chars(alignment):
    """(uint8 [n, N] characters, is_ascii, taxa or None) of a dict, tensor or array alignment."""
    if isinstance(alignment, dict):  # {taxon: sequence string}: parsers.fasta.read_alignment_from_file
        from .parsers.fasta import _to_bytes_matrix
        return _to_bytes_matrix(list(alignment.values())), True, list(alignment.keys())
    if isinstance(alignment, torch.Tensor):
        return (alignment if alignment.is_cuda else alignment.to(engine.device(), non_blocking=True)), False, None
    arr = np.asarray(alignment)
    is_ascii = arr.dtype.kind in "SU" or (arr.dtype == np.uint8 and arr.size and arr.max() > 3 and arr.max() != 255)
    return arr.astype(np.uint8, copy=False), bool(is_ascii), None


def _as_alignment(alignment, want_sm, want_planes):
    """Anything the caller may hold -> engine.DeviceAlignment (+ taxa if known)."""
    if isinstance(alignment, engine.DeviceAlignment):
        return alignment
    if isinstance(alignment, HostPlanes):
        return alignment.to_device()
    chars, is_ascii, taxa = _chars(alignment)
    return engine.pack(chars, is_ascii=is_ascii, taxa=taxa, want_sm=want_sm, want_planes=want_planes)


def _num_taxa(alignment):
    if isinstance(alignment, (engine.DeviceAlignment, HostPlanes)):
        return alignment.n
    if isinstance(alignment, dict):
        return len(alignment)
    return int(alignment.shape[0]) if hasattr(alignment, "shape") else len(alignment)


# Flattening scores of alignments with more taxa than this go through engine.sparse_flattening_scores: the dense count
# flattenings of CountScorer (4^a x 4^b bytes per split, at least 16 per launch) stop fitting in memory at 17 taxa.
DENSE_FLATTENING_MAX_TAXA = 16


def uses_sparse_flattening(n_taxa):
    return n_taxa > DENSE_FLATTENING_MAX_TAXA


def _sparse_table(alignment):
    """Pattern table of an alignment of 17..64 taxa: uint64 keys up to 31 taxa, 128-bit keys (raw counts as values) above."""
    n = _num_taxa(alignment)
    if n <= engine.NARROW_MAX_TAXA:
        return engine.count_patterns(_as_alignment(alignment, want_sm=True, want_planes=False))
    if isinstance(alignment, (engine.DeviceAlignment, HostPlanes)):
        raise NotImplementedError(f"flattening scores of {n} taxa need the alignment as characters (dict, array or tensor): "
                                  "the packed forms hold at most 32 taxa per site word")
    chars, is_ascii, taxa = _chars(alignment)
    wide, valid, n, N = engine.pack_wide(chars, is_ascii)
    keys, counts = engine.count_patterns_wide(wide, valid, n, N).compact()
    return engine.WidePatternTable(n, keys, (counts.to(torch.int64) & 0xFFFFFFFF).to(torch.float64), taxa)


def _positions(splits, taxa):
    out = []
    for left, right in splits:
        if taxa is not None and len(left) and not isinstance(left[0], (int, np.integer)):
            out.append(engine.split_positions((left, right), taxa))
        else:
            out.append((list(left), list(right)))
    return out


# Counting n taxa x N sites costs about 1.1 ms per 1.2e9 site-taxa (count_class_kernel, B200); merging the ranks' pattern
# lists costs 0.4 ms (2 ranks) .. 1.5 ms (8 ranks) whatever the size.  Below this many site-taxa every rank counts everything.
REPLICATE_MAX_SITE_TAXA = 2.0e8


def replicate_sites(n_taxa, n_sites, world):
    """True when `SplitScorer(..., sites="replicated")` is the faster form of the counting stage (flattening scores)."""
    return world > 1 and float(n_taxa) * float(n_sites) <= REPLICATE_MAX_SITE_TAXA


class SplitScorer:
    """Reusable state of `score_splits` for one split list: encoded splits, device masks, the CountScorer's buffers.
    Keeping one per (alignment shape, split list) is what a serving loop would do; `score_splits` builds a throw-away
    one."""

    def __init__(self, splits, taxa=None, method=Method.flattening, rank=0, world=1, group=None, sites="shard", refit_steps=(2,)):
        from . import distributed as spd
        if sites not in ("shard", "replicated"):
            raise ValueError('sites must be "shard" or "replicated"')
        self.method, self.rank, self.world, self.group = method, rank, world, group
        self.count_world = 1 if sites == "replicated" else world  # ranks that share the counting stage
        self.idx_all = _positions(splits, taxa)
        self.S = len(self.idx_all)
        self.positions = None
        self._steps = 0
        self._cls = None
        # calls after which the multi-GPU split partition is re-cut from the measured rank times (the first call pays the allocations;
        # the call after a re-cut reallocates batch buffers, so two listed steps must be at least two calls apart)
        self.refit_steps = tuple(refit_steps)
        if method == Method.flattening and world > 1 and self.S:
            n = len(self.idx_all[0][0]) + len(self.idx_all[0][1])
            if uses_sparse_flattening(n):
                raise NotImplementedError(f"score_splits(Method.flattening) on several GPUs: at most {DENSE_FLATTENING_MAX_TAXA} taxa "
                                          f"(this split list covers {n}); above that score on one GPU")
            # contiguous runs of the class-ordered list, cut at equal modelled cost (distributed.partition_by_cost): most ranks
            # then score ONE size class in one batch instead of an eighth of every class
            self._n = len(self.idx_all[0][0]) + len(self.idx_all[0][1])
            self._cls = [min(len(ia), len(ib)) for ia, ib in self.idx_all]
            self._per = {a: spd.flattening_cost_us(self._n, a) for a in set(self._cls)}
            self._fixed = {a: spd.flattening_fixed_us(a) for a in self._per}
            self._cut()
        else:
            self.idx_mine = spd.shard_strided(self.idx_all, rank, world)
        self.reduce_fn = spd.make_reduce_fn(group) if self.count_world > 1 else None
        self.gather_fn = spd.make_gather_fn(group) if self.count_world > 1 else None
        self.scorer = None
        self.masks = None
        self.timer = None
        self.rank_times_us = None
        if method == Method.subflattening:
            ma, mb = engine.masks_from_splits(self.idx_mine)
            dev = engine.device()
            self.masks = (torch.from_numpy(ma.view(np.int64)).to(dev), torch.from_numpy(mb.view(np.int64)).to(dev))
        elif method not in (Method.flattening, Method.mutual_information):
            raise NotImplementedError("score_splits: Method.flattening, Method.subflattening or Method.mutual_information")

    REFIT_DAMPING = 0.5

    def _cut(self):
        """(Re)partitions the class-ordered split list from the current per-class costs."""
        from . import distributed as spd
        per, cls = self._per, self._cls
        order = sorted(range(self.S), key=lambda i: (-per[cls[i]], i))
        ranges = spd.partition_by_cost([cls[i] for i in order], [per[cls[i]] for i in order], self._fixed, self.world)
        self._held = []
        for b, e in ranges:
            held = {}
            for i in order[b:e]:
                held[cls[i]] = held.get(cls[i], 0) + 1
            self._held.append(held)
        mine = order[ranges[self.rank][0]:ranges[self.rank][1]]
        self.idx_mine = [self.idx_all[i] for i in mine]
        self.positions = mine

    def _refit(self, my_us):
        """All ranks exchange the device time of their share, re-fit the per-class costs (distributed.refit_costs) and re-cut."""
        import torch.distributed as dist

        from . import distributed as spd
        mine = torch.tensor([my_us], dtype=torch.float64, device=engine.device())
        every = [torch.zeros_like(mine) for _ in range(self.world)]
        dist.all_gather(every, mine, group=self.group)
        times = [float(x.item()) for x in every]
        self.rank_times_us = times
        # a call that paid a one-off cost (the call after a re-cut reallocates its batch buffers: measured 42 ms instead of 21 ms)
        # says nothing about the steady state: keep the partition when a rank's measured / modelled ratio is more than 30 % off the median ratio
        ratios = [t_us / (spd.RANK_BASE_US + sum(c * self._per[a] + self._fixed[a] for a, c in held.items()))
                  for held, t_us in zip(self._held, times)]
        middle = sorted(ratios)[len(ratios) // 2]
        if any(not 0.7 * middle <= r <= 1.3 * middle for r in ratios):
            return
        per, fixed = spd.refit_costs(self._per, self._fixed, self._held, times)
        # half a step towards the fitted costs: the measured call is not quite the steady state (2 GPUs: the rank holding 405 6|6
        # matrices measured 25.3 ms in its second call but runs 24.2 ms later; the full step overshot, 23.3 | 24.9 ms)
        d = self.REFIT_DAMPING
        self._per = {a: self._per[a] + d * (per[a] - self._per[a]) for a in per}
        self._fixed = {a: self._fixed[a] + d * (fixed[a] - self._fixed[a]) for a in fixed}
        self._cut()

    def device_scores(self, alignment, gram_hook=None):
        """Scores of ALL splits as a device tensor.  `alignment`: this rank's site shard, or the whole alignment when the
        scorer was built with sites="replicated" (any form _as_alignment takes)."""
        import torch.distributed as dist

        from . import distributed as spd
        t = self.timer
        self._steps += 1
        refit = self._cls is not None and self._steps in self.refit_steps
        if refit:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
        if self.method == Method.flattening and uses_sparse_flattening(_num_taxa(alignment)):
            with _span(t, "count"):
                table = _sparse_table(alignment)
            with _span(t, "sparse"):
                out = engine.sparse_flattening_scores(table, self.idx_mine)
        elif self.method == Method.flattening:
            table = self._count(alignment)
            if self.scorer is None:
                self.scorer = engine.CountScorer(table)
            self.scorer.table = table
            self.scorer.timer = t
            out = self.scorer.score_many(self.idx_mine, big_hook=gram_hook)
        elif self.method == Method.mutual_information:
            table = self._count(alignment) if _num_taxa(alignment) <= engine.NARROW_MAX_TAXA else self._count_wide(alignment)
            with _span(t, "mi"):
                out = engine.rank1_divergence_scores(table, self.idx_mine)
        else:
            with _span(t, "h2d+pack"):
                aln = _as_alignment(alignment, want_sm=False, want_planes=True)
            with _span(t, "pairs"):
                raw = engine.pair_raw(aln)
            if self.count_world > 1:
                with _span(t, "allreduce"):
                    dist.all_reduce(raw, group=self.group)
            with _span(t, "subflatten+score"):
                pt = engine.pair_finalize(raw, aln.n, -1.0)  # divisor = usable sites, read on the device: no host sync
                out = engine.subflatten_scores(pt, self.masks[0], self.masks[1])
        if refit:
            ev1.record()
        with _span(t, "gather"):
            if self.positions is not None:
                if not isinstance(self.positions, torch.Tensor):
                    self.positions = torch.tensor(self.positions, dtype=torch.int64, device=out.device)
                res = spd.gather_by_position(out, self.positions, self.S, self.group)
            else:
                res = spd.gather_strided(out, self.S, self.rank, self.world, self.group)
        if refit:
            ev1.synchronize()
            self._refit(ev0.elapsed_time(ev1) * 1e3)
        return res

    def _count(self, alignment):
        """Pattern table (uint64 keys, up to 31 taxa) of the whole alignment from this rank's part of it."""
        from . import distributed as spd
        t = self.timer
        with _span(t, "h2d+pack"):
            aln = _as_alignment(alignment, want_sm=True, want_planes=False)
        with _span(t, "count"):
            if aln.n <= engine.DIRECT_MAX_TAXA:
                return engine.count_patterns(aln, gather_fn=self._timed_gather if self.gather_fn else None)
            if self.count_world > 1:  # hashed tables: gather + hash merge on every rank
                return spd.count_patterns_sharded(aln, self.rank, self.world, self.group, local=True)
            return engine.count_patterns(aln)

    def _count_wide(self, alignment):
        """engine.WideTable (128-bit keys, 32..64 taxa; divisor = usable sites) of the whole alignment from this rank's part."""
        from . import distributed as spd
        if isinstance(alignment, (engine.DeviceAlignment, HostPlanes)):
            raise NotImplementedError(f"scores of {alignment.n} taxa need the alignment as characters (dict, array or tensor): "
                                      "the packed forms hold at most 32 taxa per site word")
        with _span(self.timer, "h2d+pack"):
            chars, is_ascii, taxa = _chars(alignment)
            wide, valid, n, N = engine.pack_wide(chars, is_ascii)
        with _span(self.timer, "count"):
            if self.count_world > 1:
                return spd.count_patterns_wide_sharded(wide, valid, n, N, self.rank, self.world, self.group, local=True)
            return engine.count_patterns_wide(wide, valid, n, N, taxa=taxa)

    def _timed_gather(self, keys, counts):
        with _span(self.timer, "exchange"):
            return self.gather_fn(keys, counts)

    def __call__(self, alignment):
        return self.device_scores(alignment).cpu().numpy()


def score_splits(alignment, splits, method=Method.flattening, taxa=None):
    """One float64 score per split (numpy array, order of `splits`).

    alignment  {taxon: sequence} dict, uint8 [n_taxa, n_sites] matrix of ASCII bytes or codes 0..3 (host or device),
               `HostPlanes`, or `engine.DeviceAlignment`
    splits     pairs (left, right) of taxon labels (with `taxa`, or the dict's key order) or of taxon positions
    method     Method.flattening (scores of the flattening, constructions.py:7-102 + phylogenetics.py:280-300),
               Method.subflattening (constructions.py:108-198) or Method.mutual_information (rank-1 divergence of the
               flattening of the pattern probabilities, count / usable sites, phylogenetics.py:136-140 + 364-373: what
               erickson_SVD(..., method=Method.mutual_information) scores per candidate; 2..64 taxa, every split must place
               every taxon on exactly one side, a split with an empty side scores 0.0)
    """
    if taxa is None and isinstance(alignment, dict):
        taxa = list(alignment.keys())
    rank = world = None
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        rank, world = dist.get_rank(), dist.get_world_size()
    return SplitScorer(splits, taxa, method, rank or 0, world or 1)(alignment)


def _bootstrap_checks(name, replicates, seed):
    """The replicate count and seed checks of the bootstrap entry points and their one-process rule; returns the seed."""
    if isinstance(replicates, bool) or not isinstance(replicates, (int, np.integer)) or replicates < 1:
        raise ValueError(f"{name}: replicates must be an integer >= 1 (got {replicates!r})")
    if replicates > engine.BOOTSTRAP_MAX_REPLICATES:
        raise ValueError(f"{name}: at most {engine.BOOTSTRAP_MAX_REPLICATES} replicates")
    seed = engine.bootstrap_seed(seed)
    _one_process(name)
    return seed


def _one_process(name):
    """NotImplementedError inside a torch.distributed group of several processes: `name` runs on one GPU."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        raise NotImplementedError(f"{name} runs on one GPU: call it outside a torch.distributed group of several processes")


def bootstrap_scores(alignment, splits, method=Method.flattening, replicates=100, seed=0, taxa=None):
    """Nonparametric bootstrap of split scores: numpy float64 [replicates, len(splits)], row b = the scores `score_splits`
    gives for bootstrap replicate b of the alignment.

    A replicate draws N sites with replacement from the N usable sites; as sites with the same pattern are exchangeable it
    is drawn on the device as N patterns of the pattern table, each with probability count / N (engine.bootstrap_tables,
    csrc/bootstrap.cu).  Row b depends on the alignment, `seed` and b only: two calls with the same arguments return equal
    arrays.  `alignment`, `splits`, `method` and `taxa` have the meaning they have in `score_splits` (2..64 taxa).

    The alignment is counted once; every replicate's table then goes through the scorer `score_splits` uses:
      Method.flattening     up to 16 taxa: one engine.CountScorer for all replicates; above: engine.sparse_flattening_scores
      Method.subflattening  pair tables of the replicate's counts (engine.pair_tables_from_table) + engine.subflatten_scores
      Method.mutual_information  engine.rank1_divergence_scores (counts / N)
    The scores stay on the device until the last replicate is scored."""
    seed = _bootstrap_checks("bootstrap_scores", replicates, seed)
    if taxa is None and isinstance(alignment, dict):
        taxa = list(alignment.keys())
    # one process: the SplitScorer holds the split positions, the subflattening masks and the counting stage of score_splits
    ss = SplitScorer(splits, taxa, method)
    idx, n = ss.idx_all, _num_taxa(alignment)
    table = ss._count(alignment) if n <= engine.NARROW_MAX_TAXA else ss._count_wide(alignment)
    out = engine._empty((int(replicates), len(idx)), torch.float64)
    scorer = None
    for b, tb in enumerate(engine.bootstrap_tables(table, replicates, seed)):
        if not idx:
            continue
        if method == Method.flattening and uses_sparse_flattening(n):
            out[b] = engine.sparse_flattening_scores(tb, idx)
        elif method == Method.flattening:
            if scorer is None:
                scorer = engine.CountScorer(tb)
            else:
                scorer.table = tb
            out[b] = scorer.score_many(idx)
        elif method == Method.subflattening:
            out[b] = engine.subflatten_scores(engine.pair_tables_from_table(tb, as_counts=True), *ss.masks)
        else:
            out[b] = engine.rank1_divergence_scores(tb, idx)
    return out.cpu().numpy()


BootstrapTrees = namedtuple("BootstrapTrees", "tree support replicate_trees")


def _default_taxa(n):
    """erickson_SVD's leaf names of an alignment without names, in row order."""
    return [str(np.base_repr(i, base=max(i + 1, 2))) if n <= 36 else f"t{i}" for i in range(n)]


def _side_mask(side, index, n):
    m = 0
    for name in side:
        if name not in index:
            raise ValueError(f"bootstrap_trees: unknown leaf {name!r} in a split")
        m |= 1 << index[name]
    return m


def _split_of_mask(m, taxa):
    """erickson_SVD's form of the bipartition whose joined side is the bit mask m over the rows of `taxa`."""
    m, n = int(m), len(taxa)
    joined = tuple(sorted(taxa[i] for i in range(n) if m >> i & 1))
    rest = tuple(sorted(taxa[i] for i in range(n) if not m >> i & 1))
    return tuple(sorted((joined, rest)))


def bootstrap_trees(alignment, replicates=100, seed=0, taxa=None, method=Method.subflattening, splits=None):
    """Bootstrap support of the splits of an erickson_SVD tree.  Returns BootstrapTrees(tree, support, replicate_trees):

      tree             the n - 2 splits erickson_SVD(Method.subflattening) chooses for the alignment, in its format (a sorted
                       2-tuple of sorted leaf-name tuples per step)
      replicate_trees  the same for every bootstrap replicate; replicate b is the table engine.bootstrap_tables yields at
                       index b, so also row b of bootstrap_scores with the same seed
      support          numpy float64: entry i is the fraction of replicate trees that contain split i as a bipartition
                       (orientation ignored); split i is splits[i] (a pair of leaf-name sequences) or, by default, tree[i]

    Each tree is what erickson_SVD(Alignment(mapping, taxa), taxa=taxa, method=Method.subflattening) computes on its table:
    candidates in combinations order over the current clusters (merged cluster appended), the first minimum wins, and every
    bipartition is scored in the orientation score_canonical gives it (the side with the smallest leaf name first).  Scores
    come from pair tables of the table's integer counts, so the result is bit-reproducible.  Every replicate is agglomerated
    on the device at once (engine.bootstrap_tree_masks, csrc/agglomerate.cu): about three launches per step and no host
    synchronisation until the trees are read back.

    `alignment`, `replicates`, `seed` and `taxa` are as in bootstrap_scores; 2..64 taxa.  Leaf names are the dict's keys or
    `taxa`, else erickson_SVD's default names in row order.  Only Method.subflattening is supported."""
    if method in (Method.flattening, Method.mutual_information):
        raise NotImplementedError(f"bootstrap_trees supports Method.subflattening only: the {method} scorers take one pattern "
                                  "table per launch, so the replicates cannot be agglomerated in lockstep")
    if method != Method.subflattening:
        raise NotImplementedError("bootstrap_trees supports Method.subflattening only")
    seed = _bootstrap_checks("bootstrap_trees", replicates, seed)
    n = _num_taxa(alignment)
    if not 2 <= n <= engine._lib.SPB_MAX_TAXA:
        raise ValueError(f"bootstrap_trees: 2 to {engine._lib.SPB_MAX_TAXA} taxa (got {n})")
    if taxa is None:
        taxa = list(alignment.keys()) if isinstance(alignment, dict) else _default_taxa(n)
    taxa = list(taxa)
    if len(taxa) != n or len(set(taxa)) != n:
        raise ValueError(f"bootstrap_trees: taxa must be {n} distinct names, one per row")
    index = {t: i for i, t in enumerate(taxa)}
    full = (1 << n) - 1
    if splits is not None:
        wanted = []
        for side_a, side_b in splits:
            ma, mb = _side_mask(side_a, index, n), _side_mask(side_b, index, n)
            if ma & mb or ma | mb != full or len(side_a) + len(side_b) != n:
                raise ValueError("bootstrap_trees: every split must place every taxon on exactly one side")
            wanted.append(ma)
    first = min(range(n), key=lambda i: taxa[i])
    ss = SplitScorer([], taxa, Method.subflattening)  # the counting stage of bootstrap_scores: the same replicate tables
    table = ss._count(alignment) if n <= engine.NARROW_MAX_TAXA else ss._count_wide(alignment)
    masks, _ = engine.bootstrap_tree_masks(table, int(replicates), seed, first)

    trees = [[_split_of_mask(m, taxa) for m in row] for row in masks]
    if splits is None:
        wanted = [int(m) for m in masks[0]]
    # a bipartition as the mask of the side without taxon 0: orientation-free
    canon = lambda m: m if not m & 1 else full & ~m  # noqa: E731
    have = [{canon(int(m)) for m in row} for row in masks[1:]]
    support = np.array([sum(canon(w) in h for h in have) / len(have) for w in wanted], dtype=np.float64)
    return BootstrapTrees(trees[0], support, trees[1:])


# --------------------------------------------------------------------------------------------
# site windows
# --------------------------------------------------------------------------------------------
def sliding_windows(n_sites, width, step=None):
    """Every full window [k step, k step + width) of an alignment of n_sites sites, in order: int64 numpy [W, 2] (W = 0 when
    width > n_sites).  `step` defaults to `width` (adjacent windows)."""
    step = width if step is None else step
    for name, v, least in (("n_sites", n_sites, 0), ("width", width, 1), ("step", step, 1)):
        if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or v < least:
            raise ValueError(f"sliding_windows: {name} must be an integer >= {least} (got {v!r})")
    if width > n_sites:
        return np.zeros((0, 2), np.int64)
    k = np.arange((int(n_sites) - int(width)) // int(step) + 1, dtype=np.int64) * int(step)
    return np.stack([k, k + int(width)], axis=1)


def _num_sites(alignment):
    if isinstance(alignment, (engine.DeviceAlignment, HostPlanes)):
        return alignment.N
    if isinstance(alignment, dict):
        return len(next(iter(alignment.values()))) if alignment else 0
    return int(alignment.shape[1]) if hasattr(alignment, "shape") else len(alignment[0])


def _check_windows(name, windows, n_sites):
    """`windows` as int64 numpy [W, 2]; ValueError unless it is an integer [W, 2] array-like with 0 <= begin < end <= n_sites."""
    try:
        arr = np.asarray(windows)
    except ValueError as e:  # ragged nested sequences
        raise ValueError(f"{name}: windows must be an integer [W, 2] array ({e})") from None
    if arr.size == 0 and (arr.ndim == 1 or (arr.ndim == 2 and arr.shape[1] == 2)):
        return np.zeros((0, 2), np.int64)
    if arr.dtype.kind not in "iu":
        raise ValueError(f"{name}: windows must hold integers (got dtype {arr.dtype})")
    if arr.ndim != 2 or arr.shape[1] != 2:
        raise ValueError(f"{name}: windows must have shape [W, 2] (got {list(arr.shape)})")
    if arr.dtype.kind == "u" and (arr > np.iinfo(np.int64).max).any():
        raise ValueError(f"{name}: every window needs 0 <= begin < end <= {n_sites}")
    arr = arr.astype(np.int64)
    if ((arr[:, 0] < 0) | (arr[:, 1] > n_sites) | (arr[:, 0] >= arr[:, 1])).any():
        raise ValueError(f"{name}: every window needs 0 <= begin < end <= {n_sites}")
    return arr


def _window_inputs(name, alignment, windows):
    """(n_taxa, windows as int64 numpy [W, 2]) after the checks both window entry points share."""
    _one_process(name)
    n = _num_taxa(alignment)
    if not 2 <= n <= engine._lib.SPB_MAX_TAXA:
        raise ValueError(f"{name}: 2 to {engine._lib.SPB_MAX_TAXA} taxa (got {n})")
    return n, _check_windows(name, windows, _num_sites(alignment))


def window_scores(alignment, splits, windows, method=Method.flattening, taxa=None):
    """Split scores along site windows: numpy float64 [len(windows), len(splits)], row w = the scores `score_splits` gives
    for the alignment restricted to the sites [windows[w][0], windows[w][1]).

    windows    integer [W, 2] array-like of (begin, end) with 0 <= begin < end <= n_sites, in any order (windows may overlap
               or repeat; sliding_windows builds the usual scan); anything else raises ValueError before any device work
    alignment, splits, method, taxa   as in score_splits (2..64 taxa; above 31 taxa Method.flattening and
               Method.mutual_information need the alignment as characters)

    Method.subflattening packs the alignment once and reads it once: one segment pass cuts it at every window end
    (spb_pair_tables_segments), each window's pair tables are exact integer sums of its segments (engine.window_tables) and
    every window is scored by the multi-table scorer; the scores are bitwise those of score_splits on each slice.
    Method.flattening and Method.mutual_information pack once and count each window's patterns from the packed sites
    (count_patterns / count_patterns_wide with a site range), then score each table with the scorer score_splits uses.

    A window without usable sites scores what score_splits gives for such a slice: subflattening NaN for splits whose sides
    both hold at least two taxa and 0.0 for the others (all-zero pair tables); flattening up to 16 taxa the same (empty count
    flattening), above 16 taxa 0.0; mutual information 0.0.
    Runs on one GPU: inside a torch.distributed group of several processes it raises NotImplementedError."""
    n, wins = _window_inputs("window_scores", alignment, windows)
    if taxa is None and isinstance(alignment, dict):
        taxa = list(alignment.keys())
    ss = SplitScorer(splits, taxa, method)  # split positions and subflattening masks, as score_splits builds them
    idx, W = ss.idx_all, int(wins.shape[0])
    if W == 0 or not idx:
        return np.zeros((W, len(idx)), np.float64)
    if method == Method.subflattening:
        aln = _as_alignment(alignment, want_sm=False, want_planes=True)
        return engine.window_subflatten_scores(aln, wins, *ss.masks).cpu().numpy()
    if n <= engine.NARROW_MAX_TAXA:
        aln = _as_alignment(alignment, want_sm=True, want_planes=False)

        def table_of(b, e):
            return engine.count_patterns(aln, b, e)
    else:
        if isinstance(alignment, (engine.DeviceAlignment, HostPlanes)):
            raise NotImplementedError(f"scores of {n} taxa need the alignment as characters (dict, array or tensor): "
                                      "the packed forms hold at most 32 taxa per site word")
        chars, is_ascii, names = _chars(alignment)
        wide, valid, _, N = engine.pack_wide(chars, is_ascii)

        def table_of(b, e):
            return engine.count_patterns_wide(wide, valid, n, N, b, e, taxa=names)
    out = engine._empty((W, len(idx)), torch.float64)
    scorer = None
    for w, (b, e) in enumerate(wins.tolist()):
        tb = table_of(b, e)
        if method == Method.flattening and uses_sparse_flattening(n):
            if isinstance(tb, engine.WideTable):  # the table _sparse_table builds above 31 taxa
                keys, counts = tb.compact()
                tb = engine.WidePatternTable(n, keys, (counts.to(torch.int64) & 0xFFFFFFFF).to(torch.float64), names)
            out[w] = engine.sparse_flattening_scores(tb, idx)
        elif method == Method.flattening:
            if scorer is None:
                scorer = engine.CountScorer(tb)
            else:
                scorer.table = tb
            out[w] = scorer.score_many(idx)
        else:
            out[w] = engine.rank1_divergence_scores(tb, idx)
    return out.cpu().numpy()


def window_trees(alignment, windows, taxa=None):
    """erickson_SVD trees along site windows: tree w is the list of n - 2 splits erickson_SVD(..., method=
    Method.subflattening) chooses for the alignment restricted to the sites [windows[w][0], windows[w][1]), in its format
    (a sorted 2-tuple of sorted leaf-name tuples per step).

    Every window is agglomerated on the device at once (engine.window_tree_masks): the tables are those of window_scores
    (Method.subflattening), so every score the agglomeration compares equals the window_scores entry of that split bit for
    bit, and the candidates are oriented as bootstrap_trees orients them.  `windows` and `alignment` are as in
    window_scores; leaf names are the dict's keys or `taxa`, else erickson_SVD's default names in row order.  Runs on one
    GPU: inside a torch.distributed group of several processes it raises NotImplementedError."""
    n, wins = _window_inputs("window_trees", alignment, windows)
    if taxa is None:
        taxa = list(alignment.keys()) if isinstance(alignment, dict) else _default_taxa(n)
    taxa = list(taxa)
    if len(taxa) != n or len(set(taxa)) != n:
        raise ValueError(f"window_trees: taxa must be {n} distinct names, one per row")
    if wins.shape[0] == 0:
        return []
    first = min(range(n), key=lambda i: taxa[i])
    aln = _as_alignment(alignment, want_sm=False, want_planes=True)
    masks, _ = engine.window_tree_masks(aln, wins, first)
    return [[_split_of_mask(m, taxa) for m in row] for row in masks]
