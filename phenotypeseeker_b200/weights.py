"""Mash/GSC sample weights (`-w`): host-side replacement for `Samples.get_mash_sketches` /
`Samples.get_weights` (modeling.py:386-503), for installations without the `mash` binary,
Biopython and ete3. SURVEY.md §8f row 2. The weights are an INPUT VECTOR of the GPU test kernels
(modeling.py:812-822, 734-736); computing them is O(N L) sketching + O(N^2) distances + O(N^3)
neighbour joining on the host and is outside the timed hot path.

What the reference does, step by step, and what is restated here:

  mash sketch -r <sample>         -> sketch(): the 1000 smallest distinct 64-bit hashes
      (mash 2.2: k = 21, MurmurHash3_x64_128 seed 42, first 8 bytes, canonical = the
      alphabetically smaller of a k-mer and its reverse complement, k-mers with a letter outside
      ACGT skipped, case folded).                      PINNED against the shipped binary
      (`mash info -d`), tests/golden/mash.json.
  mash paste + mash dist          -> mash_distance(): merge walk over the two sorted sketches up
      to 1000 union elements, j = shared/denom, d = -ln(2j/(1+j))/k, printed by mash with 6
      significant digits (the reference parses that text, modeling.py:421).        PINNED (same).
  Bio.Phylo DistanceTreeConstructor.nj + phyloxml -> newick (modeling.py:446-458)
                                  -> neighbor_joining(), newick(): restated from the published
      algorithm of Biopython 1.76 (`TreeConstruction.py`), including its tie-breaking order, its
      rooting (the last two nodes are joined by hanging one under the other) and the Newick
      writer's "%1.5f" branch lengths. Biopython is not installed here and not vendored by the
      reference: PARITY UNPINNED for this step.
  GSC weights on the ete3 tree (modeling.py:460-503) -> gsc_weights(): clip branch lengths to
      [1e-9, 1e9], post-order branch sums, pre-order weights w_child = w_parent (dist +
      BranchSum) / parent.BranchSum, leaves x N.        PINNED against the reference's own
      methods run on a minimal ete3 stand-in (tests/test_weights.py).

Reference quirk kept: `mash paste reference.msh K-mer_lists/*.msh` orders the sketches by shell
glob (sorted file names) while `_mash_output_to_distance_matrix` labels the rows with the
data.pheno order (modeling.py:414-428) — the two differ when data.pheno is not sorted by sample
name. `gsc_weights_for_samples(..., keep_glob_quirk=True)` reproduces that; the default labels
the distances correctly.
"""
import math
import sys

import numpy as np

MASH_K = 21
MASH_S = 1000
MASH_SEED = 42

_M = np.uint64(0xFFFFFFFFFFFFFFFF)
_C1 = np.uint64(0x87C37B91114253D5)
_C2 = np.uint64(0x4CF5AD432745937F)


def _rotl(x, r):
    return (x << np.uint64(r)) | (x >> np.uint64(64 - r))


def _fmix(k):
    k = k ^ (k >> np.uint64(33))
    k = k * np.uint64(0xFF51AFD7ED558CCD)
    k = k ^ (k >> np.uint64(33))
    k = k * np.uint64(0xC4CEB9FE1A85EC53)
    k = k ^ (k >> np.uint64(33))
    return k


def murmur3_x64_128_h1(data, seed=MASH_SEED):
    """First 64 bits of MurmurHash3_x64_128 of every row of `data` (n x len uint8), vectorised.
    (Appleby's public-domain algorithm; mash hashes the k-mer string with it, Sketch.cpp getHash.)"""
    data = np.ascontiguousarray(data, dtype=np.uint8)
    n, length = data.shape
    h1 = np.full(n, seed, dtype=np.uint64)
    h2 = np.full(n, seed, dtype=np.uint64)
    with np.errstate(over="ignore"):
        def le64(cols):
            v = np.zeros(n, dtype=np.uint64)
            for j in range(cols.shape[1]):
                v |= cols[:, j].astype(np.uint64) << np.uint64(8 * j)
            return v
        nblocks = length // 16
        for b in range(nblocks):
            k1 = le64(data[:, 16 * b:16 * b + 8])
            k2 = le64(data[:, 16 * b + 8:16 * b + 16])
            k1 = k1 * _C1; k1 = _rotl(k1, 31); k1 = k1 * _C2; h1 = h1 ^ k1
            h1 = _rotl(h1, 27); h1 = h1 + h2; h1 = h1 * np.uint64(5) + np.uint64(0x52DCE729)
            k2 = k2 * _C2; k2 = _rotl(k2, 33); k2 = k2 * _C1; h2 = h2 ^ k2
            h2 = _rotl(h2, 31); h2 = h2 + h1; h2 = h2 * np.uint64(5) + np.uint64(0x38495AB5)
        tail = data[:, 16 * nblocks:]
        t = tail.shape[1]
        if t > 8:
            k2 = le64(tail[:, 8:])
            k2 = k2 * _C2; k2 = _rotl(k2, 33); k2 = k2 * _C1; h2 = h2 ^ k2
        if t > 0:
            k1 = le64(tail[:, :min(t, 8)])
            k1 = k1 * _C1; k1 = _rotl(k1, 31); k1 = k1 * _C2; h1 = h1 ^ k1
        h1 = h1 ^ np.uint64(length); h2 = h2 ^ np.uint64(length)
        h1 = h1 + h2; h2 = h2 + h1
        h1 = _fmix(h1); h2 = _fmix(h2)
        h1 = h1 + h2
    return h1


_COMP = np.zeros(256, dtype=np.uint8)
for _a, _b in zip(b"ACGT", b"TGCA"):
    _COMP[_a] = _b
_VALID = np.zeros(256, dtype=bool)
_VALID[list(b"ACGT")] = True


def _records(text):
    """FASTA / FASTQ bytes -> list of upper-cased sequence byte arrays (one per record)."""
    text = bytes(text)
    recs = []
    if text[:1] == b"@":
        lines = text.split(b"\n")
        for i in range(1, len(lines), 4):
            recs.append(lines[i].strip())
    else:
        for chunk in text.split(b">")[1:]:
            nl = chunk.find(b"\n")
            recs.append(b"" if nl < 0 else chunk[nl + 1:].replace(b"\n", b"").replace(b"\r", b""))
    return [np.frombuffer(r.upper(), dtype=np.uint8) for r in recs if len(r)]


def sketch(text, k=MASH_K, s=MASH_S, seed=MASH_SEED, chunk=1 << 20):
    """`mash sketch -r -k k -s s -S seed`: ascending array of the <= s smallest distinct hashes."""
    best = np.empty(0, dtype=np.uint64)
    for seq in _records(text):
        if len(seq) < k:
            continue
        for c0 in range(0, len(seq) - k + 1, chunk):
            part = seq[c0:c0 + chunk + k - 1]
            win = np.lib.stride_tricks.sliding_window_view(part, k)
            ok = _VALID[part]
            bad = np.concatenate(([0], np.cumsum(~ok)))
            good = (bad[k:] - bad[:-k]) == 0                     # windows made of ACGT only
            win = win[good]
            if not len(win):
                continue
            rc = _COMP[win[:, ::-1]]
            # alphabetical minimum of forward / reverse complement (first differing letter decides)
            diff = win != rc
            first = diff.argmax(axis=1)
            rows = np.arange(len(win))
            use_rc = diff.any(axis=1) & (rc[rows, first] < win[rows, first])
            canon = np.where(use_rc[:, None], rc, win)
            h = np.unique(murmur3_x64_128_h1(canon, seed))
            best = np.union1d(best, h[:s])[:s]
    return best


def mash_distance(a, b, k=MASH_K, s=MASH_S):
    """`mash dist` on two sketches (ascending hash arrays) -> (distance, shared, denom)
    (mash 2.2 CommandDistance.cpp compareSketches)."""
    i = j = common = denom = 0
    na, nb = len(a), len(b)
    while denom < s and i < na and j < nb:
        if a[i] < b[j]:
            i += 1
        elif b[j] < a[i]:
            j += 1
        else:
            i += 1; j += 1; common += 1
        denom += 1
    if denom < s:
        if i < na:
            denom += na - i
        if j < nb:
            denom += nb - j
        if denom > s:
            denom = s
    return distance_from_counts(common, denom, k), common, denom


def distance_from_counts(common, denom, k=MASH_K):
    """The Mash distance of a sketch pair with `common` of its `denom` smallest union hashes shared."""
    if denom == 0 or common == denom:
        return 0.0
    if common == 0:
        return 1.0
    jac = common / denom
    return -math.log(2.0 * jac / (1.0 + jac)) / k


def printed(x):
    """The value the reference reads back: mash prints distances with 6 significant digits
    (C++ ostream default) and modeling.py:421 parses that text."""
    return float("%g" % x)


def printed_distances(shared_denom, k=MASH_K):
    """N x N array of shared << 16 | denom (ps_mash_pairs) -> the printed distance matrix, through a table of
    printed(distance) over the (shared, denom) pairs that occur: the same values as distance_matrix()."""
    sd = np.asarray(shared_denom, dtype=np.uint32)
    vals, inv = np.unique(sd, return_inverse=True)
    table = np.array([printed(distance_from_counts(int(v) >> 16, int(v) & 0xFFFF, k)) for v in vals], dtype=np.float64)
    dm = table[inv].reshape(sd.shape)
    np.fill_diagonal(dm, 0.0)
    return dm


def distance_matrix(sketches, k=MASH_K, s=MASH_S):
    n = len(sketches)
    dm = np.zeros((n, n))
    for i in range(n):
        for j in range(i):
            dm[i, j] = dm[j, i] = printed(mash_distance(sketches[i], sketches[j], k, s)[0])
    return dm


class Node:
    __slots__ = ("name", "dist", "children", "up", "BranchSum", "NodeWeight")

    def __init__(self, name=None, dist=0.0):
        self.name, self.dist, self.children, self.up = name, dist, [], None
        self.BranchSum = 0.0
        self.NodeWeight = 0.0

    def add(self, child):
        child.up = self
        self.children.append(child)


def _compensated_sum(xs):
    """Python >= 3.12's sum() of floats (start 0): Neumaier's compensated summation, the compensation added at the
    end when it is non-zero and finite. Restated for older interpreters, whose sum() adds left to right."""
    it = iter(xs)
    f, c = 0 + next(it), 0.0
    for x in it:
        t = f + x
        if abs(f) >= abs(x):
            c += (f - t) + x
        else:
            c += (x - t) + f
        f = t
    if c and math.isfinite(c):
        f += c
    return f


# neighbour joining's row sums: what sum() gives on Python >= 3.12 (ps_neighbor_joining does the same on the device)
_row_sum = sum if sys.version_info >= (3, 12) else _compensated_sum


def nj_joins(dm):
    """The loop of Biopython 1.76 DistanceTreeConstructor.nj (see module docstring: unpinned) on an N x N symmetric
    matrix, N >= 3 -> (join, branch): join[t] = the list positions (mi, mj) joined at step t, branch[2t], branch[2t+1]
    = their branch lengths, branch[-1] = the distance left between the last two nodes. Row sums are Python 3.12's
    sum() on every interpreter (_row_sum). ps_neighbor_joining restates this bit for bit."""
    dm = [list(map(float, row)) for row in np.asarray(dm, dtype=np.float64)]
    n = len(dm)
    join = np.empty((n - 2, 2), dtype=np.int32)
    branch = np.empty(2 * (n - 2) + 1, dtype=np.float64)
    step = 0
    while len(dm) > 2:
        m = len(dm)
        nd = [_row_sum(dm[i]) / (m - 2) for i in range(m)]
        min_dist = dm[1][0] - nd[1] - nd[0]
        mi, mj = 0, 1
        for i in range(1, m):
            for j in range(i):
                t = dm[i][j] - nd[i] - nd[j]
                if min_dist > t:
                    min_dist, mi, mj = t, i, j
        c1 = (dm[mi][mj] + nd[mi] - nd[mj]) / 2.0
        join[step] = mi, mj
        branch[2 * step], branch[2 * step + 1] = c1, dm[mi][mj] - c1
        for x in range(m):
            if x != mi and x != mj:
                dm[mj][x] = dm[x][mj] = (dm[mi][x] + dm[mj][x] - dm[mi][mj]) / 2.0
        del dm[mi]
        for row in dm:
            del row[mi]
        step += 1
    branch[-1] = dm[1][0]
    return join, branch


def tree_from_joins(names, join, branch):
    """Replays the list operations of nj_joins on the clades: inner nodes "Inner1", "Inner2", ... and the rooting of
    the last two nodes (the last inner node stays the root when it is first in the list). Returns the root Node."""
    clades = [Node(nm) for nm in names]
    inner = None
    for t, (mi, mj) in enumerate(np.asarray(join).tolist()):
        c1, c2 = clades[mi], clades[mj]
        inner = Node("Inner" + str(t + 1))
        inner.add(c1); inner.add(c2)
        c1.dist = float(branch[2 * t])
        c2.dist = float(branch[2 * t + 1])
        clades[mj] = inner
        del clades[mi]
    last = float(branch[-1])
    if clades[0] is inner:
        clades[0].dist = 0.0
        clades[1].dist = last
        clades[0].add(clades[1])
        return clades[0]
    clades[0].dist = last
    clades[1].dist = 0.0
    clades[1].add(clades[0])
    return clades[1]


def neighbor_joining(names, dm):
    """Biopython 1.76 DistanceTreeConstructor.nj restated (see module docstring: unpinned).
    names: N labels; dm: N x N symmetric. Returns the root Node (branch lengths in .dist)."""
    n = len(names)
    if n == 1:
        return Node(names[0])
    if n == 2:
        d = float(np.asarray(dm, dtype=np.float64)[1][0])
        c1, c2 = Node(names[1]), Node(names[0])
        c1.dist = d / 2.0
        c2.dist = d - c1.dist
        root = Node("Inner")
        root.add(c1); root.add(c2)
        return root
    return tree_from_joins(names, *nj_joins(dm))


def newick(node):
    """Bio.Phylo's Newick writer: names + "%1.5f" branch lengths (the reference converts the
    phyloxml tree to Newick before handing it to ete3, modeling.py:454-458). Iterative, so that
    trees thousands of levels deep (a caterpillar from N = 5,000 samples) can be written."""
    out, stack = [], [node]
    while stack:
        it = stack.pop()
        if isinstance(it, str):
            out.append(it)
            continue
        label = (it.name or "") + ":%1.5f" % it.dist
        if not it.children:
            out.append(label)
            continue
        out.append("(")
        stack.append(")" + label)
        for i in range(len(it.children) - 1, -1, -1):
            stack.append(it.children[i])
            if i:
                stack.append(",")
    return "".join(out)


def parse_newick(text):
    """Minimal Newick reader (names + branch lengths, ete3 format=1 subset) -> root Node. Iterative, like newick()."""
    text = text.strip().rstrip(";")
    pos = 0

    def label(node):
        nonlocal pos
        start = pos
        while pos < len(text) and text[pos] not in ",():":
            pos += 1
        node.name = text[start:pos]
        if pos < len(text) and text[pos] == ":":
            pos += 1
            start = pos
            while pos < len(text) and text[pos] not in ",()":
                pos += 1
            node.dist = float(text[start:pos])

    open_nodes, root = [], None
    while True:
        node = Node()                      # a node begins at pos
        if open_nodes:
            open_nodes[-1].add(node)
        else:
            root = node
        if text[pos] == "(":
            pos += 1
            open_nodes.append(node)
            continue
        label(node)
        while True:                        # after a finished node: a sibling follows, or parents close
            if not open_nodes:
                return root
            if text[pos] == ",":
                pos += 1
                break
            pos += 1                       # ')'
            label(open_nodes.pop())


def gsc_weights(root, normalize="mean1", min_val=1e-9, max_val=1e9):
    """GSC_weights_from_newick + clip_branch_lengths + set_branch_sum + set_node_weight
    (modeling.py:460-503) on a Node tree -> {leaf name: weight}. ete3 gives a root without a branch
    length dist = 0.0, which the clip raises to 1e-9 (unused by the sums)."""
    order, stack = [], [root]
    while stack:                                      # pre-order
        nd = stack.pop()
        order.append(nd)
        stack.extend(reversed(nd.children))
    for nd in order:
        if nd.dist > max_val:
            nd.dist = max_val
        elif nd.dist < min_val:
            nd.dist = min_val
    for nd in reversed(order):                        # children before parents
        total = 0.0
        for ch in nd.children:
            total += ch.BranchSum
            total += ch.dist
        nd.BranchSum = total
    weights = {}
    for nd in order:                                  # parents before children
        if nd.up is None:
            nd.NodeWeight = 1.0
        else:
            nd.NodeWeight = nd.up.NodeWeight * (nd.dist + nd.BranchSum) / nd.up.BranchSum
        if not nd.children:
            weights[nd.name] = nd.NodeWeight
    if normalize == "mean1":
        weights = {k: v * len(weights) for k, v in weights.items()}
    return weights


def gsc_weights_for_samples(names, texts, keep_glob_quirk=False, k=MASH_K, s=MASH_S):
    """names / texts in data.pheno order -> weights in the same order (what `get_weights` leaves in
    Input.samples[name].weight, modeling.py:392-402)."""
    sk = {nm: sketch(t, k, s) for nm, t in zip(names, texts)}
    # shell glob order of K-mer_lists/<name>.msh in the C locale (other locales collate differently)
    order = sorted(names, key=lambda nm: nm + ".msh") if keep_glob_quirk else list(names)
    dm = distance_matrix([sk[nm] for nm in order], k, s)
    root = neighbor_joining(list(names), dm)          # rows are labelled in data.pheno order either way
    w = gsc_weights(parse_newick(newick(root) + ";"))
    return np.array([w[nm] for nm in names], dtype=np.float64)


def gsc_weights_on_device(ctx, names, first_idx=0, keep_glob_quirk=False, k=MASH_K, s=MASH_S, seed=MASH_SEED):
    """gsc_weights_for_samples for samples first_idx.. of a libpskmer context that already holds them (decoded by
    ps_add_samples): sketches, pair counts and neighbour joining on the device, the distance table, the tree replay,
    Newick and GSC here. Bit-identical to the host path on well-formed FASTA / FASTQ; the device reads the text as
    the k-mer counter does (DESIGN.md "Reader semantics"), which differs on bytes 1-31 inside a sequence and on U."""
    n = len(names)
    h, nh = ctx.mash_sketch(first_idx, n, k, s, seed)
    if keep_glob_quirk:                               # see gsc_weights_for_samples
        order = sorted(range(n), key=lambda i: names[i] + ".msh")
        h, nh = h[order], nh[order]
    dm = printed_distances(ctx.mash_pairs(h, nh), k)
    if n >= 3:
        root = tree_from_joins(list(names), *ctx.neighbor_joining(dm))
    else:
        root = neighbor_joining(list(names), dm)
    w = gsc_weights(parse_newick(newick(root) + ";"))
    return np.array([w[nm] for nm in names], dtype=np.float64)
