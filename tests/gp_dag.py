"""TEST INFRASTRUCTURE: a subsplit-DAG and GP op-program generator.

From a list of rooted bifurcating trees on n taxa it builds the subsplit DAG (every subsplit
the trees use, and every parent-subsplit -> child-subsplit edge, a GPCSP, that they use) and
emits what sbn.GPEngine and gp.GPEngineOracle take: PLV and GPCSP counts, an SBN prior q,
unconditional node probabilities, the inverted prior, and the five op programs in the flat
int32 encoding of include/sbn_b200_gp.h.

Conventions are the reference GPDAG's (visible in tests/golden/gp_*.npz):
- node ids: leaves 0..n-1, then the subsplits in order of clade size, so that every child has
  a smaller id than its parents and the rootsplits come last;
- six PLVs per node: p, p-hat, p-hat-tilde, r-hat, r, r-tilde at kind * node_count + node.
  p-hat sums the children of a subsplit's first clade, p-hat-tilde those of its second;
  r = r-hat * p-hat-tilde feeds the first clade's children, r-tilde = r-hat * p-hat the second's;
- GPCSPs: the rootsplits first, then one contiguous group per (parent, clade), so that
  UpdateSBNProbabilities(start, stop) covers one group;
- PrepForMarginalization comes before a PLV receives increments.
The generator does not reproduce GPDAG op for op: tests/test_gp_reference_cpu.py checks that
the programs compute the exact marginal of the trees the DAG holds (tests/gp_reference.py).

A tree is a dict {clade bitmask: (first, second)} with one entry per clade of two or more
taxa; `first` is the half that holds the clade's lowest taxon.
"""
import numpy as np

P_PLV, PHAT, PHAT_TILDE, RHAT, R_PLV, R_TILDE = range(6)


def _ordered(a, b):
    return (a, b) if (a & -a) < (b & -b) else (b, a)


def random_tree(taxon_count, rng):
    """A coalescent-shaped random rooted tree: random pairs of clades merged until one is left."""
    clades, tree = [1 << i for i in range(taxon_count)], {}
    while len(clades) > 1:
        i, j = sorted(rng.choice(len(clades), size=2, replace=False))
        a, b = clades[i], clades[j]
        tree[a | b] = _ordered(a, b)
        clades = [c for k, c in enumerate(clades) if k not in (i, j)] + [a | b]
    return tree


def ladder_tree(order):
    """The caterpillar that adds the taxa of `order` one at a time: (((o0, o1), o2), ...)."""
    clade, tree = 1 << order[0], {}
    for taxon in order[1:]:
        tree[clade | (1 << taxon)] = _ordered(clade, 1 << taxon)
        clade |= 1 << taxon
    return tree


def caterpillar_resolution(clade):
    """Every clade of `clade` resolved one fixed way: its lowest taxon against the rest."""
    tree = {}
    while clade & (clade - 1):
        low = clade & -clade
        tree[clade] = (low, clade ^ low)
        clade ^= low
    return tree


def rootsplit_tree(first, second):
    """The tree with root subsplit (first, second) and both halves resolved as caterpillars."""
    tree = {first | second: _ordered(first, second)}
    tree.update(caterpillar_resolution(first))
    tree.update(caterpillar_resolution(second))
    return tree


class SubsplitDAG:
    def __init__(self, taxon_count, trees, seed=0, dirichlet_alpha=1.0):
        n = self.taxon_count = int(taxon_count)
        full = (1 << n) - 1
        subsplits, pcsps = set(), set()
        for tree in trees:
            assert tree, "a tree needs at least two taxa"
            for clade, (a, b) in tree.items():
                assert a | b == clade and not a & b and (a & -a) < (b & -b)
                subsplits.add((a, b))
                for side, half in enumerate((a, b)):
                    if half & (half - 1):
                        pcsps.add(((a, b), side, tree[half]))
                    else:
                        pcsps.add(((a, b), side, half.bit_length() - 1))
        internal = sorted(subsplits, key=lambda s: (bin(s[0] | s[1]).count("1"), s[0] | s[1], s[0]))
        self.subsplits = [None] * n + internal
        node_of = {s: n + i for i, s in enumerate(internal)}
        self.node_count = len(self.subsplits)
        self.plv_count = 6 * self.node_count
        self.rootsplit_nodes = [node_of[s] for s in internal if s[0] | s[1] == full]
        # GPCSPs: rootsplits, then (parent, side) groups in node order
        edges = [(None, None, v) for v in self.rootsplit_nodes]
        self.groups = [(0, len(edges))]
        self.children = {}  # (node, side) -> [(gpcsp, child)]
        by_side = {}
        for parent, side, child in pcsps:
            child = node_of[child] if isinstance(child, tuple) else child
            by_side.setdefault((node_of[parent], side), []).append(child)
        for v in range(n, self.node_count):
            for side in (0, 1):
                start = len(edges)
                for child in sorted(by_side[(v, side)]):
                    self.children.setdefault((v, side), []).append((len(edges), child))
                    edges.append((v, side, child))
                self.groups.append((start, len(edges)))
        self.edges = edges
        self.gpcsp_count = len(edges)
        self.rootsplit_count = len(self.rootsplit_nodes)
        self.parents = {}  # node -> [(gpcsp, parent, side)]
        for g, (v, side, child) in enumerate(edges):
            if v is not None:
                self.parents.setdefault(child, []).append((g, v, side))
        rng = np.random.default_rng(seed)
        self.q = np.empty(self.gpcsp_count)
        for start, stop in self.groups:
            self.q[start:stop] = rng.dirichlet(np.full(stop - start, dirichlet_alpha))
        self.q = np.maximum(self.q, 1e-12)
        for start, stop in self.groups:
            self.q[start:stop] /= self.q[start:stop].sum()
        # unconditional node probabilities (top-down) and P(parent | child)
        node_probability = np.zeros(self.node_count)
        for g, v in enumerate(self.rootsplit_nodes):
            node_probability[v] = self.q[g]
        for v in range(self.node_count - 1, -1, -1):
            for side in (0, 1):
                for g, child in self.children.get((v, side), []):
                    node_probability[child] += node_probability[v] * self.q[g]
        self.unconditional_node_probabilities = node_probability
        self.inverted_sbn_prior = np.ones(self.gpcsp_count)
        for g, (v, side, child) in enumerate(edges):
            if v is not None:
                self.inverted_sbn_prior[g] = node_probability[v] * self.q[g] / node_probability[child]
        self.programs = {name: np.array(words, dtype=np.int32) for name, words in self._programs().items()}

    def plv(self, kind, node):
        return kind * self.node_count + node

    def is_leaf(self, node):
        return node < self.taxon_count

    # ---- the five programs
    def _programs(self):
        n, N = self.taxon_count, self.node_count
        populate = []
        for v in range(n, N):
            for kind in (P_PLV, PHAT, PHAT_TILDE):
                populate += [0, self.plv(kind, v)]
        for v in range(N):
            for kind in (RHAT, R_PLV, R_TILDE):
                populate += [0, self.plv(kind, v)]
        for g, v in enumerate(self.rootsplit_nodes):
            populate += [1, self.plv(RHAT, v), g]
        for v in range(n, N):  # leafward, children before parents
            for side, kind in ((0, PHAT), (1, PHAT_TILDE)):
                children = self.children[(v, side)]
                populate += [9, self.plv(kind, v), len(children)] + [self.plv(P_PLV, c) for _, c in children]
                for g, c in children:
                    populate += [2, self.plv(kind, v), g, self.plv(P_PLV, c)]
            populate += [3, self.plv(P_PLV, v), self.plv(PHAT, v), self.plv(PHAT_TILDE, v)]
        for v in range(N - 1, -1, -1):  # rootward, parents before children
            parents = self.parents.get(v, [])
            if parents:
                sources = [self.plv(R_PLV if side == 0 else R_TILDE, u) for _, u, side in parents]
                populate += [9, self.plv(RHAT, v), len(sources)] + sources
                for (g, _, _), src in zip(parents, sources):
                    populate += [2, self.plv(RHAT, v), g, src]
            if not self.is_leaf(v):
                populate += [3, self.plv(R_PLV, v), self.plv(RHAT, v), self.plv(PHAT_TILDE, v)]
                populate += [3, self.plv(R_TILDE, v), self.plv(RHAT, v), self.plv(PHAT, v)]
        marginal = [7]
        for g, v in enumerate(self.rootsplit_nodes):
            marginal += [8, self.plv(RHAT, v), g, self.plv(P_PLV, v)]
        likelihoods, optimization = [], []
        for g in range(self.rootsplit_count, self.gpcsp_count):
            leafward, rootward = self.edge_plvs(g)
            likelihoods += [4, g, leafward, rootward]
            optimization += [5, leafward, rootward, g]
        sbn = []
        for start, stop in self.groups:
            if stop - start > 1:
                sbn += [6, start, stop]
        return {"populate_plvs": populate, "compute_likelihoods": likelihoods + marginal,
                "marginal_likelihood": marginal, "branch_length_optimization": optimization,
                "optimize_sbn_parameters": sbn}

    def edge_plvs(self, g):
        """(leafward, rootward) PLVs of a non-rootsplit GPCSP: the OptimizeBranchLength fields."""
        v, side, child = self.edges[g]
        return self.plv(P_PLV, child), self.plv(R_PLV if side == 0 else R_TILDE, v)

    # ---- the trees the DAG holds
    def tree_count(self):
        count = [1] * self.node_count
        for v in range(self.taxon_count, self.node_count):
            count[v] = 1
            for side in (0, 1):
                count[v] *= sum(count[c] for _, c in self.children[(v, side)])
        return sum(count[v] for v in self.rootsplit_nodes)

    def trees(self, limit=5000):
        """Every tree the DAG holds, as a sorted tuple of GPCSP indices (its rootsplit first)."""
        assert self.tree_count() <= limit, f"{self.tree_count()} trees: more than the enumeration's cap of {limit}"
        below = [[()] for _ in range(self.node_count)]
        for v in range(self.taxon_count, self.node_count):
            options = [()]
            for side in (0, 1):
                options = [o + (g,) + sub for o in options for g, c in self.children[(v, side)] for sub in below[c]]
            below[v] = options
        return [tuple(sorted((g,) + sub)) for g, v in enumerate(self.rootsplit_nodes) for sub in below[v]]

    def tree_shape(self, tree, branch_lengths):
        """(parent_ids, lengths) of a tree in subst_reference.prune's convention (children have smaller
        ids than parents, the root last, one length per node) and the node of each GPCSP's child."""
        nodes = sorted({self.edges[g][2] for g in tree})
        index = {v: i for i, v in enumerate(nodes)}
        assert nodes[:self.taxon_count] == list(range(self.taxon_count))
        parent_ids = np.zeros(len(nodes) - 1, dtype=np.int64)
        lengths = np.zeros(len(nodes))
        child_of = {}
        for g in tree:
            v, _, child = self.edges[g]
            if v is None:
                assert index[child] == len(nodes) - 1
                continue
            parent_ids[index[child]] = index[v]
            lengths[index[child]] = branch_lengths[g]
            child_of[g] = index[child]
        return parent_ids, lengths, child_of


def simulate_states(dag, tree, branch_lengths, pattern_count, rng, gap_fraction=0.0):
    """[taxon][pattern] states evolved down one tree of the DAG under JC69 (for alignments with
    signal, so that branch-length optima are interior), with a fraction of gaps (4)."""
    parent_ids, lengths, _ = dag.tree_shape(tree, branch_lengths)
    node_count = len(parent_ids) + 1
    states = np.zeros((node_count, pattern_count), dtype=np.int64)
    states[-1] = rng.integers(0, 4, pattern_count)
    for node in range(node_count - 2, -1, -1):
        keep = rng.random(pattern_count) < np.exp(-4.0 * lengths[node] / 3.0)
        states[node] = np.where(keep, states[parent_ids[node]], rng.integers(0, 4, pattern_count))
    tips = states[:dag.taxon_count].astype(np.uint8)
    tips[rng.random(tips.shape) < gap_fraction] = 4
    return tips


# ---- the shapes the tests use
def hybrid_dag(taxon_count, tree_count, seed):
    """The union of `tree_count` random trees: holds more trees than went in."""
    rng = np.random.default_rng(seed)
    return SubsplitDAG(taxon_count, [random_tree(taxon_count, rng) for _ in range(tree_count)], seed=seed)


def one_tree_dag(taxon_count, shape, seed):
    rng = np.random.default_rng(seed)
    tree = ladder_tree([int(x) for x in rng.permutation(taxon_count)]) if shape == "ladder" else random_tree(taxon_count, rng)
    return SubsplitDAG(taxon_count, [tree], seed=seed)


def wide_root_dag(taxon_count, rootsplit_count, seed):
    """`rootsplit_count` trees, each with its own rootsplit and every clade resolved as a caterpillar:
    the root group has `rootsplit_count` children and the DAG holds exactly these trees."""
    rng = np.random.default_rng(seed)
    full, chosen = (1 << taxon_count) - 1, set()
    while len(chosen) < rootsplit_count:
        first = int(rng.integers(1, full)) | 1  # (the half holding taxon 0)
        if first != full:
            chosen.add(first)
    return SubsplitDAG(taxon_count, [rootsplit_tree(first, full ^ first) for first in sorted(chosen)], seed=seed)
