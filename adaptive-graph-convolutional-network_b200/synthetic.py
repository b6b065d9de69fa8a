"""Synthetic inputs of the BASELINE.json shapes (SURVEY.md section 8d), host side, numpy only.

Used by bench.py and tools/ as the product-side input generator (the CPU oracle under oracle/ has its own copy of
the molecule generator for the tests; tests/test_host_logic.py checks that both produce the same batch).  Every
batch comes back in the reference's wire layout (models/tf_modules/graph_topology.py:84-98): zero-padded
X [B, Nmax, F], L [B, Nmax, Nmax] float32 and n_nodes [B] int32.

  C1 / C2  molecules        75-d one-hot-ish atom features (utils/feature/graph_features.py:156-180), random
                            spanning tree + ring closures, degree <= 4, Laplacian by Graph.compute_laplacian
  C3       ModelNet40-shape N = 1024 points, xyz normalised to the unit sphere, rotated + jittered like
                            utils/provider.py:33-85, adjacency d_ij < mean distance (meshloader.py:264-285)
  C4       Sydney-shape     ragged n ~ loguniform[13, 1024], xyz + intensity, adjacency by the cut-off rule of
                            pointcloudloader.py:240-263
"""
import numpy as np

from .graph_structure import Graph


# ---- molecules (C1 Tox21-shape, C2 ToxCast-shape) -----------------------------------------------------------------
def tox21_like_features(rng, n):
    """75-d atom features: one-hot blocks of 44, 11, 5, 7, formal charge, radical electrons, one-hot 5, aromatic flag
    (graph_features.py:156-180).  Rows repeat exactly on purpose (SURVEY Q7: duplicate rows have distance 0)."""
    x = np.zeros((n, 75), np.float32)
    col = 0
    for width, conc in ((44, 4), (11, 4), (5, 3), (7, 3)):
        idx = np.minimum(rng.geometric(1.0 / conc, n) - 1, width - 1)
        x[np.arange(n), col + idx] = 1.0
        col += width
    x[:, col] = rng.choice([-1.0, 0.0, 1.0], n, p=[0.03, 0.94, 0.03]); col += 1
    col += 1  # radical electrons: 0
    x[np.arange(n), col + np.minimum(rng.geometric(0.5, n) - 1, 4)] = 1.0; col += 5
    x[:, col] = rng.random(n) < 0.4
    return x


def molecule_like_adjacency(rng, n):
    """Adjacency lists of a random spanning tree plus a few ring closures, degree <= 4."""
    deg = np.zeros(n, np.int32)
    adj = [[] for _ in range(n)]

    def link(a, b):
        if a != b and b not in adj[a] and deg[a] < 4 and deg[b] < 4:
            adj[a].append(b), adj[b].append(a)
            deg[a] += 1; deg[b] += 1
            return True
        return False

    for v in range(1, n):
        for _ in range(16):
            if link(v, int(rng.integers(max(0, v - 6), v))):
                break
        else:
            cands = [u for u in range(v) if deg[u] < 4]
            link(v, cands[-1])
    for _ in range(max(1, n // 6)):
        a = int(rng.integers(0, n)); b = int(min(n - 1, a + rng.integers(3, 7)))
        link(a, b)
    return adj


def tox21_like_sizes(rng, B, Nmax=132):
    n = np.clip(np.round(rng.lognormal(np.log(17.0), 0.55, B)), 4, Nmax).astype(np.int32)
    n[0] = Nmax                                            # one forced maximum-size molecule
    return n


def molecule_batch(B, Nmax=132, seed=1234):
    """X [B,Nmax,75], L [B,Nmax,Nmax] (Graph.compute_laplacian, the drop-in of graph_structure.py:85-130), n_nodes."""
    rng = np.random.default_rng(seed)
    n_nodes = tox21_like_sizes(rng, B, Nmax)
    X = np.zeros((B, Nmax, 75), np.float32)
    L = np.zeros((B, Nmax, Nmax), np.float32)
    for g, n in enumerate(n_nodes):
        X[g, :n] = tox21_like_features(rng, n)
        graph = Graph(X[g, :n], molecule_like_adjacency(rng, n), max_deg=4, min_deg=0)
        L[g, :n, :n] = np.asarray(graph.Laplacian.todense(), dtype=np.float32)      # graph_topology.py:92-98
    return X, L, n_nodes


# ---- point clouds (C3 ModelNet40-shape, C4 Sydney-shape) -------------------------------------------------------------
def laplacian_from_dense_adjacency(A):
    """Graph.compute_laplacian (graph_structure.py:85-130) on a dense symmetric 0/1 adjacency without self loops:
    A^ = D~^-1/2 (A + I) D~^-1/2, then L = I - D^-1/2 A^ D^-1/2 with D from the column sums of A^.  float64."""
    n = A.shape[0]
    At = A.astype(np.float64) + np.eye(n)
    dinv = 1.0 / np.sqrt(At.sum(1))
    An = (At * dinv[None, :]) * dinv[:, None]
    d = An.sum(axis=0) + np.spacing(np.array(0, An.dtype))
    d = 1.0 / np.sqrt(d)
    return np.eye(n) - (d[:, None] * An) * d[None, :]


def pairwise_distances(P):
    P = P.astype(np.float32)
    diff = P[:, None, :] - P[None, :, :]
    return np.sqrt(np.einsum("ijk,ijk->ij", diff, diff)).astype(np.float32)


def adjacency_mean_rule(P):
    """meshloader.py:264-285: d_lim = mean of ||p_i - p_j|| over the pairs j <= i (the n zero self-distances
    included); i ~ j iff i != j and d_ij < d_lim."""
    D = pairwise_distances(P)
    n = D.shape[0]
    d_lim = D[np.tril_indices(n)].astype(np.float32).mean(dtype=np.float32)
    A = D < d_lim
    np.fill_diagonal(A, False)
    return A


def adjacency_cutoff_rule(P, sparse_ratio=0.1):
    """pointcloudloader.py:240-263: d_lim = the int(n * sparse_ratio)-th LARGEST of the distances over the pairs
    j <= i (np.sort(all_dist)[-cut_off_idx]; cut_off_idx == 0 selects the smallest, a zero self-distance, i.e. no
    edge at all); i ~ j iff i != j and d_ij < d_lim."""
    D = pairwise_distances(P)
    n = D.shape[0]
    all_dist = np.sort(D[np.tril_indices(n)])
    d_lim = all_dist[-int(n * sparse_ratio)]
    A = D < d_lim
    np.fill_diagonal(A, False)
    return A


def _rotate_jitter(rng, P, sigma=0.01, clip=0.05):
    """utils/provider.py:33-85: random rotation about the up axis, then clipped Gaussian jitter."""
    a = rng.uniform(0, 2 * np.pi)
    c, s = np.cos(a), np.sin(a)
    Rm = np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]], np.float32)
    P = P @ Rm
    return (P + np.clip(sigma * rng.standard_normal(P.shape), -clip, clip)).astype(np.float32)


def modelnet_like_batch(B=32, N=1024, seed=1236):
    """C3: B clouds of N points (no padding), F = 3."""
    rng = np.random.default_rng(seed)
    X = np.zeros((B, N, 3), np.float32)
    L = np.zeros((B, N, N), np.float32)
    for g in range(B):
        P = rng.standard_normal((N, 3)).astype(np.float32) * rng.uniform(0.3, 1.0, 3).astype(np.float32)
        P = P - P.mean(0)
        P = P / np.abs(P).max()
        P = _rotate_jitter(rng, P)
        X[g] = P
        L[g] = laplacian_from_dense_adjacency(adjacency_mean_rule(P)).astype(np.float32)
    return X, L, np.full(B, N, np.int32)


def sydney_like_sizes(rng, B, lo=13, hi=1024):
    return np.exp(rng.uniform(np.log(lo), np.log(hi), B)).round().astype(np.int32)


def sydney_like_batch(B=128, Nmax=1024, seed=1237):
    """C4: ragged clouds, F = 4 (xyz + intensity in [0, 1], pointcloudloader.py:233), padded to Nmax."""
    rng = np.random.default_rng(seed)
    n_nodes = np.minimum(sydney_like_sizes(rng, B, 13, Nmax), Nmax).astype(np.int32)
    n_nodes[0] = Nmax
    X = np.zeros((B, Nmax, 4), np.float32)
    L = np.zeros((B, Nmax, Nmax), np.float32)
    for g, n in enumerate(n_nodes):
        P = rng.standard_normal((n, 3)).astype(np.float32) * rng.uniform(0.5, 3.0, 3).astype(np.float32)
        feat = np.hstack([P, (rng.integers(0, 256, (n, 1)) / 255.0).astype(np.float32)])
        X[g, :n] = feat
        L[g, :n, :n] = laplacian_from_dense_adjacency(adjacency_cutoff_rule(feat)).astype(np.float32)
    return X, L, n_nodes


def knn_like_batch(B, N, F, seed=1238, deg=16):
    """C5 sweep point: n_g = N, X ~ N(0, 1), L = normalised Laplacian of a random ~deg-neighbour graph."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((B, N, F)).astype(np.float32)
    L = np.zeros((B, N, N), np.float32)
    for g in range(B):
        A = np.zeros((N, N), bool)
        idx = rng.integers(0, N, (N, min(deg, N - 1)))
        A[np.repeat(np.arange(N), idx.shape[1]), idx.reshape(-1)] = True
        A |= A.T
        np.fill_diagonal(A, False)
        L[g] = laplacian_from_dense_adjacency(A).astype(np.float32)
    return X, L, np.full(B, N, np.int32)


# ---- per-node labels (the part labels of a segmentation batch) -------------------------------------------------------
def synthetic_node_labels(batch, X, C, seed):
    """One class out of C per node, learnable from the node's own features, in the packed row order.

    batch: a GraphBatch, or its n_nodes array; X: the padded features [B, Nmax, F] of the batch (wire layout).
      point clouds (F <= 8, xyz in the first three columns): the angular sector of (x, z) around the up axis y times
      the height band of y within the cloud, S sectors x H bands with H = ceil(sqrt(C)), S = ceil(C / H), label
      (sector * H + band) mod C;
      molecules (75-d atom features): the index of the atom-type one-hot block (the first 44 columns) mod C.
    Returns (targets [R, C] one-hot float32, weights [R] float32 of 0 / 1 with about 10 % zeros: unlabelled nodes)."""
    n_nodes = np.asarray(getattr(batch, "n_nodes", batch), np.int64)
    X = np.asarray(X)
    rows = np.concatenate([X[g, :n] for g, n in enumerate(n_nodes)]).astype(np.float32)
    if X.shape[-1] == 75:
        label = rows[:, :44].argmax(1) % C
    else:
        H = int(np.ceil(np.sqrt(C)))
        S = int(np.ceil(C / H))
        ang = np.arctan2(rows[:, 2], rows[:, 0]) + np.pi                       # [0, 2 pi]
        sector = np.minimum((ang * (S / (2 * np.pi))).astype(np.int64), S - 1)
        band = np.empty(len(rows), np.int64)
        off = 0
        for n in n_nodes:
            y = rows[off:off + n, 1]
            lo, span = y.min(), max(float(y.max() - y.min()), 1e-12)
            band[off:off + n] = np.minimum(((y - lo) * (H / span)).astype(np.int64), H - 1)
            off += n
        label = (sector * H + band) % C
    targets = np.zeros((len(rows), C), np.float32)
    targets[np.arange(len(rows)), label] = 1.0
    weights = (np.random.default_rng(seed).random(len(rows)) >= 0.1).astype(np.float32)
    return targets, weights
