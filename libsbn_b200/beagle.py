"""ctypes binding of the inner boundary: include/libhmsbeagle/beagle.h as implemented on the device by
libsbn_b200/lib/libhmsbeagle_b200.so (libsbn_b200/csrc/beagle_shim.cu), driven with the call sequence the
reference's FatBeagle makes (src/fat_beagle.cpp:50-70, 119-175, 207-362).  The same class runs over any
other library with the same ABI (the tests pass the CPU restatement's path to compare call by call)."""
import ctypes
import os

import numpy as np

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libhmsbeagle_b200.so")
OP_NONE = -1
_I, _D = ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_double)


class Beagle:
    """The BEAGLE calls of fat_beagle.cpp over one of the two libraries."""

    def __init__(self, path, n, P, C, use_tip_states):
        self.lib = ctypes.CDLL(path or os.environ.get("SBNB_BEAGLE_LIBRARY") or LIB_PATH)
        self.n, self.P, self.C, self.N = n, P, C, 2 * n - 1
        partials = 3 * n - 2 + (0 if use_tip_states else n)  # fat_beagle.cpp:207-256
        self.handle = self.lib.beagleCreateInstance(n, partials, n if use_tip_states else 0, 4, P, 1, 2 * self.N, C,
                                                    partials + 1, None, 0, 0, 1 << 6, None)
        assert self.handle >= 0, self.handle

    def ok(self, code):
        assert code == 0, code

    def _d(self, a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        return a, a.ctypes.data_as(_D)

    def _i(self, a):
        a = np.ascontiguousarray(a, dtype=np.int32)
        return a, a.ctypes.data_as(_I)

    def set_tips(self, states, weights, use_tip_states, masks=False):
        """Tip states (use_tip_states) or tip partials built from them; masks=True: `states`
        are nucleotide masks, and each tip's partial is the indicator vector of its bits."""
        for tip in range(self.n):
            if masks:
                bits = np.asarray(states[tip], dtype=np.int64)
                partial = np.ascontiguousarray(((bits[:, None] >> np.arange(4)) & 1).astype(np.float64))
                keep, ptr = self._d(partial)
                self.ok(self.lib.beagleSetTipPartials(self.handle, tip, ptr))
                continue
            if use_tip_states:
                keep, ptr = self._i(states[tip])
                self.ok(self.lib.beagleSetTipStates(self.handle, tip, ptr))
            else:
                partial = np.zeros((self.P, 4))
                for k, s in enumerate(states[tip]):
                    partial[k, :] = 1.0 if s >= 4 else 0.0
                    if s < 4:
                        partial[k, s] = 1.0
                keep, ptr = self._d(partial)
                self.ok(self.lib.beagleSetTipPartials(self.handle, tip, ptr))
        keep, ptr = self._d(weights)
        self.ok(self.lib.beagleSetPatternWeights(self.handle, ptr))

    def set_model(self, evec, ivec, evals, freqs, rates, proportions):
        keeps = [self._d(x) for x in (evec, ivec, evals, freqs, rates, proportions)]
        self.ok(self.lib.beagleSetStateFrequencies(self.handle, 0, keeps[3][1]))
        self.ok(self.lib.beagleSetEigenDecomposition(self.handle, 0, keeps[0][1], keeps[1][1], keeps[2][1]))
        self.ok(self.lib.beagleSetCategoryWeights(self.handle, 0, keeps[5][1]))
        self.ok(self.lib.beagleSetCategoryRates(self.handle, keeps[4][1]))

    def log_likelihood_and_gradient(self, post_ops, pre_ops, lengths, q, rates, freqs, rescaling, per_site=True):
        """FatBeagle::BranchGradientInternals (fat_beagle.cpp:119-175).  per_site=False asks for what
        FatBeagle asks for (the sums only: fat_beagle.cpp:157-166 passes NULL for the per-site
        derivatives and the sums of squares); the default also fetches those two, for the tests."""
        n, N = self.n, self.N
        keep_i, idx = self._i(np.arange(N - 1))
        keep_l, lens = self._d(lengths[:N - 1])
        self.ok(self.lib.beagleUpdateTransitionMatrices(self.handle, 0, idx, None, None, lens, N - 1))
        dq = np.stack([r * q for r in rates])
        keep_q, dq_ptr = self._d(dq)
        self.ok(self.lib.beagleSetDifferentialMatrix(self.handle, N - 1, dq_ptr))
        cumulative = 0 if rescaling else OP_NONE
        if rescaling:
            self.ok(self.lib.beagleResetScaleFactors(self.handle, 0))
        keep_a, ops = self._i(post_ops)
        self.ok(self.lib.beagleUpdatePartials(self.handle, ops, len(post_ops), cumulative))
        root_pre = np.tile(freqs, self.C * self.P)
        keep_r, root_ptr = self._d(root_pre)
        self.ok(self.lib.beagleSetPartials(self.handle, 2 * N - 1, root_ptr))
        keep_b, ops = self._i(pre_ops)
        self.ok(self.lib.beagleUpdatePrePartials(self.handle, ops, len(pre_ops), OP_NONE))
        keep_1, post_idx = self._i(np.arange(N - 1))
        keep_2, pre_idx = self._i(np.arange(N - 1) + N)
        keep_3, dm_idx = self._i(np.full(N - 1, N - 1))
        keep_4, zero = self._i([0])
        sums, squares = np.zeros(N - 1), np.zeros(N - 1)
        per_site_values = np.zeros((N - 1, self.P)) if per_site else None
        self.ok(self.lib.beagleCalculateEdgeDerivatives(
            self.handle, post_idx, pre_idx, dm_idx, zero, N - 1,
            per_site_values.ctypes.data_as(_D) if per_site else None, sums.ctypes.data_as(_D),
            squares.ctypes.data_as(_D) if per_site else None))
        keep_5, root = self._i([N - 1])
        keep_6, cum = self._i([cumulative])
        logl = ctypes.c_double()
        self.ok(self.lib.beagleCalculateRootLogLikelihoods(self.handle, root, zero, zero, cum, 1, ctypes.byref(logl)))
        return logl.value, sums, squares, per_site_values

    def close(self):
        self.ok(self.lib.beagleFinalizeInstance(self.handle))


def random_tree_operations(n, rng, rescaling, order="libsbn"):
    """A random rooted binary tree as the op lists of fat_beagle.cpp:327-362.

    order = "libsbn": libsbn's numbering AND order -- leaves 0..n-1, internal nodes numbered by a depth-first
    post-order traversal (root 2n-2); the post-order list in that traversal's order (Node::Postorder,
    node.cpp:205-211), the pre-order list as Node::TriplePreorderBifurcating emits it (node.cpp:226-261:
    a node's first child, that child's subtree, then its second child and its subtree).
    order = "node_id": internal nodes numbered in the order of the random joins and the lists in id order
    (children before parents, but not depth-first: consecutive ops are rarely parent and child)."""
    N = 2 * n - 1
    roots, joined, next_id = list(range(n)), {}, n
    while len(roots) > 1:
        a, b = (roots.pop(int(rng.integers(len(roots)))) for _ in range(2))
        joined[next_id] = (a, b)
        roots.append(next_id)
        next_id += 1
    if order == "node_id":
        children = joined
        post_order = sorted(children)
        pre_pairs = [(v, child, sister) for v in sorted(children, reverse=True)
                     for child, sister in (children[v], children[v][::-1])]
    else:
        # renumber the internal nodes by a depth-first post-order traversal
        new_id, visit_order, stack = {t: t for t in range(n)}, [], [(next_id - 1, False)]
        while stack:
            v, expanded = stack.pop()
            if v < n:
                continue
            if expanded:
                new_id[v] = n + len(visit_order)
                visit_order.append(v)
            else:
                stack.append((v, True))
                stack.append((joined[v][1], False))
                stack.append((joined[v][0], False))
        children = {new_id[v]: (new_id[joined[v][0]], new_id[joined[v][1]]) for v in visit_order}
        post_order = sorted(children)
        pre_pairs, stack = [], [(N - 1, False)]
        while stack:  # Node::TriplePreorderBifurcating
            v, visited = stack.pop()
            c0, c1 = children[v]
            if visited:
                pre_pairs.append((v, c1, c0))
                if c1 >= n:
                    stack.append((c1, False))
            else:
                pre_pairs.append((v, c0, c1))
                stack.append((v, True))
                if c0 >= n:
                    stack.append((c0, False))
    post = [[v, (v - n + 1) if rescaling else OP_NONE, OP_NONE, children[v][0], children[v][0], children[v][1],
             children[v][1]] for v in post_order]
    pre = [[child + N, (child + 1 + n - 1) if rescaling else OP_NONE, OP_NONE, v + N, child, sister, sister]
           for v, child, sister in pre_pairs]
    return np.array(post, dtype=np.int32), np.array(pre, dtype=np.int32)


def depth_first_operations(post, n):
    """The same ops, children before parents in depth-first order (libsbn's traversal order: the
    destination of an op is a child of the next one, which the device kernel keeps in registers)."""
    by_dest = {int(op[0]): op for op in post}
    order, stack = [], [(int(post[-1][0]), False)]
    while stack:  # (no recursion: a 1000-taxon ladder is 999 ops deep)
        v, expanded = stack.pop()
        if v < n:
            continue
        if expanded:
            order.append(by_dest[v])
        else:
            stack.append((v, True))
            stack.append((int(by_dest[v][5]), False))
            stack.append((int(by_dest[v][3]), False))
    return np.array(order, dtype=np.int32)


def gtr_eigensystem():
    rates = np.array([0.05, 0.1, 0.15, 0.20, 0.25, 0.25])
    freqs = np.array([0.1, 0.2, 0.3, 0.4])
    q = np.zeros((4, 4))
    index = 0
    for i in range(4):
        for j in range(i + 1, 4):
            q[i, j], q[j, i] = rates[index] * freqs[j], rates[index] * freqs[i]
            index += 1
    q -= np.diag(q.sum(axis=1))
    q /= -np.sum(np.diag(q) * freqs)
    root = np.sqrt(freqs)
    values, vectors = np.linalg.eigh(root[:, None] * q / root[None, :])
    return vectors / root[:, None], vectors.T * root[None, :], values, freqs, q
