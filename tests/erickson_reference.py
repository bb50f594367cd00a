"""A Python restatement of erickson_SVD's agglomeration loop (splitp_b200/phylogenetics.py, reference
splitp/phylogenetics.py:99-171) with the scorer passed in, for the bootstrap-tree tests.

`score_many(splits)` receives the bipartitions a step has not scored yet, each once and in the orientation score_canonical
gives it (the side holding the smallest leaf name first), and returns one score per split.  Candidates are formed with
`combinations` over the current cluster list, the first minimum wins, the merged cluster is appended.
"""
from itertools import combinations

M64 = (1 << 64) - 1


def _leaves(cluster):
    return (cluster,) if isinstance(cluster, str) else tuple(cluster)


def agglomerate(taxa, score_many):
    """(chosen splits as erickson_SVD returns them, per-step {split: score} of the candidates)."""
    taxa = list(taxa)
    num_taxa = len(taxa)
    known, canonical_scores = {}, {}
    chosen, trace = [], []
    while len(chosen) < num_taxa - 2:
        candidates = []
        for pair in combinations(taxa, 2):
            joined = tuple(sorted(leaf for cluster in pair for leaf in _leaves(cluster)))
            rest = tuple(sorted(leaf for cluster in taxa for leaf in _leaves(cluster) if leaf not in joined))
            candidates.append((pair, (joined, rest)))
        todo = []
        for _, split in candidates:
            c = split if split[0] <= split[1] else (split[1], split[0])
            if c not in canonical_scores and c not in todo:
                todo.append(c)
        if todo:
            canonical_scores.update(zip(todo, score_many(todo)))
        for _, split in candidates:
            known[split] = canonical_scores[split if split[0] <= split[1] else (split[1], split[0])]
        best_pair, best_split = min(candidates, key=lambda c: known[c[1]])
        trace.append({split: known[split] for _, split in candidates})
        chosen.append(tuple(sorted(best_split)))
        merged = best_split[0]
        taxa = [c for c in taxa if c not in merged and not set(c).issubset(merged)] + [merged]
    return chosen, trace


def hashed_score(ma, mb, r):
    """An integer-valued fake score of the oriented split (ma, mb) of replicate r, 0..4: many exact ties."""
    h = ((ma * 0x9E3779B97F4A7C15) ^ (mb * 0xC2B2AE3D27D4EB4F) ^ (r * 0x94D049BB133111EB)) & M64
    return float((h >> 40) % 5)


def mask_of(side, index):
    m = 0
    for name in side:
        m |= 1 << index[name]
    return m


def split_of_mask(m, taxa):
    """erickson_SVD's form of the bipartition (bit i set = taxa[i] on the joined side)."""
    n = len(taxa)
    joined = tuple(sorted(taxa[i] for i in range(n) if m >> i & 1))
    rest = tuple(sorted(taxa[i] for i in range(n) if not m >> i & 1))
    return tuple(sorted((joined, rest)))
