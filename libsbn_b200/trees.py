"""Host-side topology utilities: synthetic random trees in the reference's id
convention, and Newick export for the reference arm of the benchmark.

Id convention (reference src/node.cpp:341-357 `Node::Polish`): leaves are
0..n-1, internal nodes are numbered in post-order with the children of every
node sorted by their maximum leaf id (src/node.cpp:36-44), the root is last.
A topology is its `Node::ParentIdVector` (src/node.cpp:413-424).
"""
import numpy as np


def _canonical(children, root, taxon_count):
    """Relabels an arbitrary rooted tree (dict node -> child list, leaves are
    0..n-1) into the reference convention; returns (parent_ids, old->new map)."""
    max_leaf, order, stack = {}, [], [(root, False)]
    while stack:  # iterative post-order (ladder trees are deep)
        node, done = stack.pop()
        kids = children.get(node, [])
        if not kids:
            max_leaf[node] = node
        elif done:
            kids.sort(key=lambda k: max_leaf[k])
            max_leaf[node] = max_leaf[kids[-1]]
        else:
            stack.append((node, True))
            stack.extend((k, False) for k in kids)
    new_id, next_id, stack = {}, taxon_count, [(root, False)]
    while stack:
        node, done = stack.pop()
        kids = children.get(node, [])
        if not kids:
            new_id[node] = node
        elif done:
            new_id[node] = next_id
            next_id += 1
        else:
            stack.append((node, True))
            stack.extend((k, False) for k in reversed(kids))
    parent_ids = np.full(next_id - 1, -1, dtype=np.int32)
    for node, kids in children.items():
        for k in kids:
            parent_ids[new_id[k]] = new_id[node]
    return parent_ids, new_id


def random_unrooted_topology(taxon_count, rng):
    """Uniform random stepwise addition; trifurcating root; 2n-3 parent ids."""
    assert taxon_count >= 3
    root = taxon_count
    children = {root: [0, 1, 2]}
    parent = {0: root, 1: root, 2: root}
    next_label = taxon_count + 1
    edges = [0, 1, 2]  # an edge is named by its child node
    for leaf in range(3, taxon_count):
        target = edges[rng.integers(len(edges))]
        up = parent[target]
        inner = next_label
        next_label += 1
        children[up][children[up].index(target)] = inner
        children[inner] = [target, leaf]
        parent[inner], parent[target], parent[leaf] = up, inner, inner
        edges.extend([inner, leaf])
    return _canonical(children, root, taxon_count)[0]


def random_rooted_topology(taxon_count, rng):
    """Random bifurcating rooted topology; 2n-2 parent ids."""
    assert taxon_count >= 2
    root = taxon_count
    children = {root: [0, 1]}
    parent = {0: root, 1: root}
    next_label = taxon_count + 1
    edges = [0, 1]
    for leaf in range(2, taxon_count):
        target = edges[rng.integers(len(edges))]
        up = parent[target]
        inner = next_label
        next_label += 1
        children[up][children[up].index(target)] = inner
        children[inner] = [target, leaf]
        parent[inner], parent[target], parent[leaf] = up, inner, inner
        edges.extend([inner, leaf])
    return _canonical(children, root, taxon_count)[0]


def ladder_topology(taxon_count, unrooted=True):
    """Caterpillar tree: the deepest possible traversal (n-2 dependent levels)."""
    root = 10 * taxon_count
    if unrooted:
        children, spine = {root: [0, 1, None]}, root
        slot, first = 2, 2
    else:
        children, spine = {root: [0, None]}, root
        slot, first = 1, 1
    label = taxon_count
    for leaf in range(first, taxon_count - 1):
        children[spine][slot] = label
        children[label] = [leaf, None]
        spine, slot = label, 1
        label += 1
    children[spine][slot] = taxon_count - 1
    return _canonical(children, root, taxon_count)[0]


def random_tree_batch(taxon_count, tree_count, seed, mean_branch_length=0.1, rooted=False):
    """(parent_ids [T][nodes-1], branch_lengths [T][nodes]) ~ Exp(mean), clipped >= 1e-6."""
    rng = np.random.default_rng(seed)
    make = random_rooted_topology if rooted else random_unrooted_topology
    parent_ids = np.stack([make(taxon_count, rng) for _ in range(tree_count)])
    node_count = parent_ids.shape[1] + 1
    lengths = np.maximum(rng.exponential(mean_branch_length, size=(tree_count, node_count)), 1e-6)
    lengths[:, -1] = 0.0  # the root has no branch
    return parent_ids, lengths


def random_time_trees(taxon_count, tree_count, seed, epochs=4, relaxed=False, ladder=False, topology_count=None):
    """Seeded dated (time) trees: a dict of everything TreeBatch takes.

    Tips are sampled at `epochs` dates, so internal nodes both share their bound with an
    internal child and sit above a child of an older epoch; internal bounds are the
    largest bound of their children.  A non-root node d internal nodes above its deepest
    tip has ratio (d + u) / (d + 1), u uniform in [-0.5, 0.5], clipped to [1e-3, 0.999]:
    the ratios on a path then multiply to about (d + 1) / (depth + 1), so even a 1000-taxon
    ladder keeps every branch far from 0 (a product of independent ratios would shrink
    geometrically, and fp64 transition matrices of branches near 1e-9 are only good to
    ~1e-16 / length, which decides the likelihood of alignments with a change on every
    branch).  Then
    heights follow top-down as h = b + r (h_parent - b) (the float64 expression any
    reference must repeat to see the same heights); height_ratios[n - 2] is the root
    height, branch_lengths[e] = h_parent - h_e with the root's entry 0.  Strict clock:
    one rate c != 1 on every edge (rate_count 1); relaxed: lognormal rates per edge
    (rate_count 2n - 2).  topology_count: reuse that many topologies cyclically, each
    tree with its own dates, ratios and rates; ladder: caterpillar topologies."""
    rng = np.random.default_rng(seed)
    n, N = taxon_count, 2 * taxon_count - 1
    shapes = topology_count or tree_count
    topologies = [ladder_topology(n, unrooted=False) if ladder else random_rooted_topology(n, rng)
                  for _ in range(shapes)]
    out = {name: np.zeros((tree_count, width)) for name, width in (
        ("branch_lengths", N), ("rates", N - 1), ("node_heights", N), ("node_bounds", N), ("height_ratios", n - 1))}
    out["parent_ids"] = np.stack([topologies[t % shapes] for t in range(tree_count)])
    out["rate_count"] = N - 1 if relaxed else 1
    for t in range(tree_count):
        parent = out["parent_ids"][t]
        children = [[] for _ in range(N)]
        for child, p in enumerate(parent):
            children[p].append(child)
        dates = np.concatenate([[0.0], np.cumsum(rng.uniform(0.02, 0.1, size=epochs - 1))])
        for _ in range(100):  # until both sides of the epoch test occur (where the shape allows)
            bounds = np.zeros(N)
            bounds[:n] = dates[rng.integers(0, epochs, size=n)]
            for node in range(n, N):
                bounds[node] = max(bounds[c] for c in children[node])
            pairs = [(bounds[node] == bounds[c]) for node in range(n, N - 1) for c in children[node] if c >= n]
            if epochs < 2 or (any(pairs) and not all(pairs)):
                break
        above = np.zeros(N)
        for node in range(n, N):
            above[node] = 1 + max(above[c] for c in children[node])
        ratios = np.clip((above[n:] + rng.uniform(-0.5, 0.5, size=n - 1)) / (above[n:] + 1), 1e-3, 0.999)
        ratios[n - 2] = bounds[N - 1] + rng.uniform(0.2, 0.6)
        heights = bounds.copy()
        heights[N - 1] = ratios[n - 2]
        for node in range(N - 2, n - 1, -1):
            heights[node] = bounds[node] + ratios[node - n] * (heights[parent[node]] - bounds[node])
        out["branch_lengths"][t, :N - 1] = heights[parent] - heights[:N - 1]
        clock = rng.choice([rng.uniform(0.4, 0.9), rng.uniform(1.1, 1.6)])
        out["rates"][t] = clock * (rng.lognormal(0.0, 0.4, size=N - 1) if relaxed else 1.0)
        out["node_heights"][t], out["node_bounds"][t], out["height_ratios"][t] = heights, bounds, ratios
    return out


def random_alignment(taxon_count, pattern_count, seed, gap_fraction=0.01):
    """iid uniform {A,C,G,T} with a fraction of gap states; every column is kept
    as its own pattern with weight 1 (BASELINE config 4/5 shape)."""
    rng = np.random.default_rng(seed)
    states = rng.integers(0, 4, size=(taxon_count, pattern_count), dtype=np.uint8)
    states[rng.random((taxon_count, pattern_count)) < gap_fraction] = 4
    return states, np.ones(pattern_count)


def random_masked_alignment(taxon_count, pattern_count, seed, ambiguous_fraction=0.05, gap_fraction=0.01):
    """Nucleotide masks (bit 0 = A .. bit 3 = T): iid uniform single states, a fraction
    of missing characters (15) and a fraction of ambiguous ones drawn uniformly from the
    ten two- and three-state masks; every column its own pattern with weight 1."""
    rng = np.random.default_rng(seed)
    masks = (1 << rng.integers(0, 4, size=(taxon_count, pattern_count))).astype(np.uint8)
    draw = rng.random((taxon_count, pattern_count))
    masks[draw < gap_fraction] = 15
    ambiguous = (draw >= gap_fraction) & (draw < gap_fraction + ambiguous_fraction)
    choices = np.array([3, 5, 6, 7, 9, 10, 11, 12, 13, 14], dtype=np.uint8)
    masks[ambiguous] = choices[rng.integers(0, len(choices), size=int(ambiguous.sum()))]
    return masks, np.ones(pattern_count)


def states_to_masks(states):
    """States (0..3, >= 4 gap) -> the equivalent nucleotide masks (1, 2, 4, 8, 15)."""
    states = np.asarray(states)
    return np.where(states < 4, np.left_shift(1, np.minimum(states, 3)), 15).astype(np.uint8)


def masks_to_states(masks):
    """Masks -> states, every ambiguous mask turned into a gap (what the state table keeps)."""
    masks = np.asarray(masks)
    single = {1: 0, 2: 1, 4: 2, 8: 3}
    out = np.full(masks.shape, 4, dtype=np.uint8)
    for mask, state in single.items():
        out[masks == mask] = state
    return out


def newick(parent_ids, branch_lengths, taxon_names=None):
    """Newick string of one tree (children in id order, lengths by node id)."""
    node_count = len(parent_ids) + 1
    kids = [[] for _ in range(node_count)]
    for child, parent in enumerate(parent_ids):
        kids[parent].append(child)
    text = {}
    for node in range(node_count):  # children precede parents
        if kids[node]:
            label = "(" + ",".join(text.pop(k) for k in kids[node]) + ")"
        else:
            label = taxon_names[node] if taxon_names else f"t{node}"
        if node != node_count - 1:
            label += f":{float(branch_lengths[node])!r}"
        text[node] = label
    return text[node_count - 1] + ";"
