"""Parity of the CUDA path (through the C ABI) against the CPU oracle.  Tolerance: 1e-4 relative
(max-abs error over max-abs reference, BASELINE.md section 5); padding rows must be exactly +0.0."""
import numpy as np
import pytest
import torch

from oracle import sgcll_oracle as O
from util_cases import TOL, compare, cuda_run, make_batch, oracle_run, random_prev_laps

pytestmark = pytest.mark.gpu

SIZES = [132, 4, 5, 18, 33, 64, 65, 17, 96, 31]


def _cot(shape, seed):
    return np.random.default_rng(seed).standard_normal(shape).astype(np.float32)


@pytest.mark.parametrize("laplacian", ["reference_literal", "paper"])
@pytest.mark.parametrize("K", [1, 2, 3, 5])
def test_sgc_ll_forward_backward(laplacian, K):
    F, Fo = 75, 64
    X, L, n = make_batch(SIZES, F, 132, seed=K, kind="tox")
    p = O.make_params(F, Fo, K, "SGC_LL", seed=10 + K, dtype=torch.float64)
    cY = _cot((len(SIZES), 132, Fo), 5)
    orc = oracle_run(X, L, n, p, K, "SGC_LL", laplacian, "reference", cot_Y=cY)
    cu = cuda_run(X, L, n, p, K, "SGC_LL", laplacian, "reference", cot_Y=cY)
    errs = compare(cu, orc)
    print(laplacian, K, errs)


@pytest.mark.parametrize("laplacian", ["reference_literal", "paper"])
@pytest.mark.parametrize("with_prev", [False, True])
def test_reslap_forward_backward(laplacian, with_prev):
    F, Fo, K = 64, 128, 3
    X, L, n = make_batch(SIZES, F, 132, seed=3, kind="relu")
    p = O.make_params(F, Fo, K, "SGC_LL_Reslap", seed=21, dtype=torch.float64)
    Lprev = random_prev_laps(n, 4) if with_prev else None
    cY = _cot((len(SIZES), 132, Fo), 6)
    cL = [_cot((int(k), int(k)), 70 + i) for i, k in enumerate(n)]
    orc = oracle_run(X, L, n, p, K, "SGC_LL_Reslap", laplacian, "reference", Lprev, cot_Y=cY, cot_L=cL)
    cu = cuda_run(X, L, n, p, K, "SGC_LL_Reslap", laplacian, "reference", Lprev, cot_Y=cY, cot_L=cL)
    errs = compare(cu, orc)
    print(laplacian, with_prev, errs)


@pytest.mark.parametrize("variant", ["SGC_LL", "SGC_LL_Reslap"])
def test_paper_full_metric_gradient(variant):
    F, Fo, K = 32, 16, 3
    sizes = [40, 4, 9, 23, 64, 70]
    X, L, n = make_batch(sizes, F, 72, seed=8)
    X *= 0.5
    p = O.make_params(F, Fo, K, variant, seed=31, dtype=torch.float64)
    Lprev = random_prev_laps(n, 5) if variant == "SGC_LL_Reslap" else None
    cY = _cot((len(sizes), 72, Fo), 7)
    cL = [_cot((int(k), int(k)), 90 + i) for i, k in enumerate(n)] if variant == "SGC_LL_Reslap" else None
    orc = oracle_run(X, L, n, p, K, variant, "paper", "full", Lprev, cot_Y=cY, cot_L=cL)
    cu = cuda_run(X, L, n, p, K, variant, "paper", "full", Lprev, cot_Y=cY, cot_L=cL)
    errs = compare(cu, orc)
    assert float(orc["dM_L"].abs().max()) > 0
    print(variant, errs)


def test_full_gradient_with_duplicate_rows():
    """Exactly duplicated rows (dist == 0): sub-gradient 0 (SURVEY H5), no NaN."""
    F, Fo, K = 75, 8, 2
    X, L, n = make_batch([18, 30, 7], F, 30, seed=12, kind="tox")
    p = O.make_params(F, Fo, K, "SGC_LL", seed=2, dtype=torch.float64)
    cY = _cot((3, 30, Fo), 9)
    orc = oracle_run(X, L, n, p, K, "SGC_LL", "paper", "full", cot_Y=cY)
    cu = cuda_run(X, L, n, p, K, "SGC_LL", "paper", "full", cot_Y=cY)
    for k, v in cu.items():
        if isinstance(v, torch.Tensor):
            assert torch.isfinite(v).all(), k
    compare(cu, orc)


@pytest.mark.parametrize("F,Fo,K", [(3, 32, 3), (4, 16, 2), (128, 128, 3), (256, 32, 2), (64, 617, 2)])
def test_feature_shapes(F, Fo, K):
    sizes = [50, 13, 100, 4, 29]
    X, L, n = make_batch(sizes, F, 100, seed=F)
    p = O.make_params(F, Fo, K, "SGC_LL", seed=F + 1, dtype=torch.float64)
    cY = _cot((len(sizes), 100, Fo), 11)
    for lap in ("reference_literal", "paper"):
        orc = oracle_run(X, L, n, p, K, "SGC_LL", lap, "reference", cot_Y=cY)
        cu = cuda_run(X, L, n, p, K, "SGC_LL", lap, "reference", cot_Y=cY)
        compare(cu, orc)


def test_padding_rows_are_positive_zero_and_pack_roundtrip():
    import agcn_b200
    F, Fo, K = 75, 64, 3
    X, L, n = make_batch(SIZES, F, 132, seed=1, kind="tox")
    p = O.make_params(F, Fo, K, "SGC_LL", seed=1, dtype=torch.float64)
    cu = cuda_run(X, L, n, p, K, "SGC_LL", "reference_literal", "reference")
    Y = cu["Y"].numpy()
    for g, k in enumerate(n):
        pad = Y[g, k:]
        assert np.array_equal(pad.view(np.uint32), np.zeros_like(pad).view(np.uint32))  # bit-exact +0.0
    batch = cu["batch"]
    Xd, Ld = torch.tensor(X, device="cuda"), torch.tensor(L, device="cuda")
    assert torch.equal(batch.unpack_nodes(batch.pack_nodes(Xd)), Xd)
    assert torch.equal(batch.unpack_lap(batch.pack_lap(Ld)), Ld)


def test_metric_block_against_reference_golden():
    """res_W / res_L of the CUDA path against the outputs of the reference's own `func`
    (tests/golden/metric_block.npz, produced by executing the reference source)."""
    import os
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "metric_block.npz"))
    names = sorted({k.split("/")[0] for k in gold.files})
    for name in names:
        x, M = gold[name + "/x"], gold[name + "/M"]
        n, F = x.shape
        X = x[None].copy()
        L = np.zeros((1, n, n), np.float32)
        p = O.make_params(F, 8, 2, "SGC_LL", seed=0, dtype=torch.float64, perturb=False)
        p["M_L"] = torch.tensor(M, dtype=torch.float64)
        cu = cuda_run(X, L, np.array([n], np.int32), p, 2, "SGC_LL", "reference_literal", "reference")
        W_ref, L_ref = gold[name + "/W_ll"], gold[name + "/L_ll"]
        err = O.rel_err(cu["res_W"][0], W_ref) if W_ref.max() > 0 else float(cu["res_W"][0].abs().max())
        assert err <= TOL, (name, err)
        # alpha = 1, clip_by_average_norm(I) = I  => res_L == I exactly
        assert torch.equal(cu["res_L"][0], torch.tensor(L_ref)), name


def test_layer_api_matches_oracle():
    """SGC_LL / SGC_LL_Reslap called like the reference's graph containers call them
    (tf_graphs.py:45-54,178-194), with the reference's padded list inputs."""
    import agcn_b200
    from agcn_b200.layers import SGC_LL, SGC_LL_Reslap
    F, Fo, K = 75, 32, 2
    sizes = [20, 4, 9, 50]
    X, L, n = make_batch(sizes, F, 50, seed=3, kind="tox")
    dev = torch.device("cuda:0")
    x = {"node_features": [torch.tensor(X[g], device=dev) for g in range(4)],
         "original_laplacian": [torch.tensor(L[g], device=dev) for g in range(4)],
         "data_slice": np.stack([[k, -1] for k in n]).astype(np.int32),
         "lap_slice": np.stack([[k, k] for k in n]).astype(np.int32)}
    layer = SGC_LL(Fo, F, 4, K=K, activation="relu")
    out, res_L, res_W = layer(x)
    assert len(out) == 4 and tuple(out[0].shape) == (50, Fo)
    p = {k: v.detach().double().cpu() for k, v in layer.vars.items()}
    orc = oracle_run(X, L, n, p, K, "SGC_LL", "reference_literal", "reference")
    assert O.rel_err(out.padded().detach().cpu(), orc["Y"]) <= TOL
    assert tuple(res_W[1].shape) == (4, 4) and O.rel_err(res_W[3].cpu(), orc["res_W"][3]) <= TOL
    assert torch.equal(res_L[0].cpu(), torch.eye(20))
    # Reslap stack: second layer consumes the first layer's saved Laplacians
    l1 = SGC_LL_Reslap(Fo, F, 4, K=K, save_lap=True)
    l2 = SGC_LL_Reslap(16, Fo, 4, K=K)
    x["res_lap"] = []
    o1, _, _, La1 = l1(x)
    x2 = dict(x, node_features=o1, res_lap=list(La1)[-4:])
    o2, _, _, La2 = l2(x2)
    p1 = {k: v.detach().double().cpu() for k, v in l1.vars.items()}
    p2 = {k: v.detach().double().cpu() for k, v in l2.vars.items()}
    r1 = oracle_run(X, L, n, p1, K, "SGC_LL_Reslap", "reference_literal", "reference")
    r2 = oracle_run(r1["Y"].numpy(), L, n, p2, K, "SGC_LL_Reslap", "reference_literal", "reference",
                    [t.numpy() for t in r1["L_all"]])
    assert O.rel_err(o2.padded().detach().cpu(), r2["Y"]) <= TOL
    assert O.rel_err(La2[3].detach().cpu(), r2["L_all"][3]) <= TOL
    (o2.data.sum() + La2.data.sum()).backward()
    assert l1.vars["beta"].grad is not None and torch.isfinite(l1.vars["weight"].grad).all()
    with pytest.raises(TypeError):
        SGC_LL(8, 8, 4, bogus=1)
    with pytest.raises(ValueError):
        SGC_LL(8, 8, 4, activation="nope")


def test_host_buffer_entry_point():
    """agcn_sgcll_forward_host: padded host arrays in, padded host array out."""
    import ctypes
    import agcn_b200
    from agcn_b200 import _lib
    from agcn_b200.functional import make_desc
    F, Fo, K = 75, 64, 3
    X, L, n = make_batch([30, 4, 17, 60], F, 64, seed=2, kind="tox")
    p = O.make_params(F, Fo, K, "SGC_LL", seed=4, dtype=torch.float64)
    dev = torch.device("cuda:0")
    batch = agcn_b200.GraphBatch(n, 64, device=dev)
    desc = make_desc(F, Fo, K, "SGC_LL", "reference_literal", "reference", "relu", 0)
    nbytes = ctypes.c_size_t()
    _lib.check(_lib.lib().agcn_sgcll_host_scratch_bytes(ctypes.byref(desc), batch.handle, ctypes.byref(nbytes)))
    scratch = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
    pd = {k: v.float().to(dev) for k, v in p.items()}
    Xh, Lh = torch.tensor(X).pin_memory(), torch.tensor(L).pin_memory()
    Yh = torch.empty(4, 64, Fo).pin_memory()
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    _lib.check(_lib.lib().agcn_sgcll_forward_host(ctypes.byref(desc), batch.handle, vp(Xh), vp(Lh), vp(pd["M_L"]),
                                                  vp(pd["weight"]), vp(pd["bias"]), vp(pd["alpha"]), vp(Yh),
                                                  vp(scratch), scratch.numel(),
                                                  ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    orc = oracle_run(X, L, n, p, K, "SGC_LL", "reference_literal", "reference")
    assert O.rel_err(Yh, orc["Y"]) <= TOL


def test_full_size_properties_toxcast_batch():
    """BASELINE full size (B = 1024, Nmax = 132, 75 -> 64, K = 3): size-independent properties --
    linearity in the weights, zero padding, and exact agreement with the oracle on a sample of graphs."""
    F, Fo, K, B = 75, 64, 3, 1024
    X, L, n = O.synthetic_molecule_batch(B, 132, seed=1235)
    p = O.make_params(F, Fo, K, "SGC_LL", seed=5, dtype=torch.float64)
    p["bias"] = torch.zeros_like(p["bias"])
    cu1 = cuda_run(X, L, n, p, K, "SGC_LL", "reference_literal", "reference", activation="linear", want_res=False)
    p2 = dict(p, weight=p["weight"] * 2.0)
    cu2 = cuda_run(X, L, n, p2, K, "SGC_LL", "reference_literal", "reference", activation="linear", want_res=False)
    assert O.rel_err(cu2["Y"], 2.0 * cu1["Y"]) <= 1e-6                 # linear in the weights
    idx = [0, 1, 2, 511, 1023]
    orc = oracle_run(X[idx], L[idx], n[idx], p, K, "SGC_LL", "reference_literal", "reference", activation="linear")
    assert O.rel_err(cu1["Y"][idx], orc["Y"]) <= TOL
    rows = torch.arange(132)[None, :] >= torch.tensor(n.astype(np.int64))[:, None]
    assert float(cu1["Y"][rows].abs().max()) == 0.0


def _dense_laplacians(n_list, Nmax, seed):
    """Dense symmetric normalised Laplacians like the thresholded point-cloud graphs (~50 % fill)."""
    rng = np.random.default_rng(seed)
    L = np.zeros((len(n_list), Nmax, Nmax), np.float32)
    for g, n in enumerate(n_list):
        A = (rng.random((n, n)) < 0.5).astype(np.float64)
        A = np.triu(A, 1); A = A + A.T + np.eye(n)
        d = 1.0 / np.sqrt(A.sum(1))
        L[g, :n, :n] = (np.eye(n) - d[:, None] * A * d[None, :]).astype(np.float32)
    return L


@pytest.mark.parametrize("sizes,F,Fo,K", [([1024, 1024, 1024], 3, 32, 3),          # ModelNet40-shape
                                          ([13, 700, 145, 1024, 64, 144, 333], 4, 26, 3),   # Sydney-shape, ragged
                                          ([2048, 150], 32, 32, 2),              # sweep point
                                          ([513, 200], 64, 128, 5),
                                          ([300, 145, 257, 1000], 256, 32, 3),   # two 128-column blocks, ragged n
                                          ([161, 450], 96, 48, 4),               # three 32-column boxes
                                          ([200, 150, 333], 5, 16, 3),           # thin path, F in 5..8
                                          ([129, 192, 128], 128, 128, 3)])       # tile edges: n = 128 k + 1, 64-row remainder
def test_large_graphs_row_tiled_path(sizes, F, Fo, K):
    """Graphs that do not fit in shared memory (n > 144) run through the grouped-GEMM path; small and large
    graphs mix freely in one batch (SURVEY C3 / C4 / C5)."""
    Nmax = max(sizes)
    X, _, n = make_batch(sizes, F, Nmax, seed=F + K)
    L = _dense_laplacians(sizes, Nmax, seed=K)
    p = O.make_params(F, Fo, K, "SGC_LL", seed=F, dtype=torch.float64)
    cY = _cot((len(sizes), Nmax, Fo), 13)
    orc = oracle_run(X, L, n, p, K, "SGC_LL", "reference_literal", "reference", cot_Y=cY)
    cu = cuda_run(X, L, n, p, K, "SGC_LL", "reference_literal", "reference", cot_Y=cY, want_res=False)
    errs = compare(cu, orc, skip=("res_L", "res_W", "L_all"))
    print(sizes, errs)


@pytest.mark.parametrize("F,Fo,K", [(32, 16, 3), (4, 8, 4)])
def test_nonsymmetric_laplacian_transpose_paths(F, Fo, K):
    """The backward recurrence multiplies by L^T: a non-symmetric intrinsic matrix tells L from L^T in every size
    class (fused tiles, per-graph shared-memory kernels, row-tiled / tensor-core / thin kernels)."""
    sizes = [150, 70, 20, 300, 129]
    Nmax = max(sizes)
    X, _, n = make_batch(sizes, F, Nmax, seed=8)
    L = _dense_laplacians(sizes, Nmax, seed=2)
    rng = np.random.default_rng(77)
    for g, k in enumerate(sizes):
        L[g, :k, :k] += (rng.standard_normal((k, k)) * 0.02).astype(np.float32)
    p = O.make_params(F, Fo, K, "SGC_LL", seed=5, dtype=torch.float64)
    cY = _cot((len(sizes), Nmax, Fo), 21)
    orc = oracle_run(X, L, n, p, K, "SGC_LL", "reference_literal", "reference", cot_Y=cY)
    cu = cuda_run(X, L, n, p, K, "SGC_LL", "reference_literal", "reference", cot_Y=cY, want_res=False)
    print(compare(cu, orc, skip=("res_L", "res_W", "L_all")))


@pytest.mark.parametrize("sizes,F,Fo,K,laplacian,metric_grad", [
    ([256, 256, 256], 64, 32, 3, "reference_literal", "reference"),
    ([384, 384], 128, 128, 2, "reference_literal", "reference"),     # two 128-column... one column block, 3 row tiles
    ([256, 256], 160, 16, 3, "reference_literal", "reference"),      # two column blocks (128 + 32)
    ([256, 256], 32, 32, 3, "paper", "full"),                        # dense L_all, dL, the RowScale product
    ([1024], 16, 16, 2, "reference_literal", "reference"),
    ([1024] * 19, 32, 16, 2, "reference_literal", "reference")])     # 152 row tiles > 148 SMs: bt::grouped_tcu_kernel
def test_equal_size_graphs_row_tiled_products(sizes, F, Fo, K, laplacian, metric_grad):
    """Batches of equal-size graphs with n % 128 == 0 (ModelNet40-shape point clouds), whole layer forward + backward.
    A non-symmetric intrinsic matrix tells L from L^T (forward recurrence against the reverse one).  (Grids above one
    CTA per SM take bt::grouped_tcu_kernel: the 19-cloud case below and test_uniform_tensor_core_product.)"""
    Nmax = max(sizes)
    X, _, n = make_batch(sizes, F, Nmax, seed=F + K)
    X *= 0.5
    L = _dense_laplacians(sizes, Nmax, seed=K + 3)
    rng = np.random.default_rng(19)
    for g, k in enumerate(sizes):
        L[g, :k, :k] += (rng.standard_normal((k, k)) * 0.01).astype(np.float32)
    p = O.make_params(F, Fo, K, "SGC_LL", seed=F + 2, dtype=torch.float64)
    cY = _cot((len(sizes), Nmax, Fo), 17)
    orc = oracle_run(X, L, n, p, K, "SGC_LL", laplacian, metric_grad, cot_Y=cY, compute_similarity=(laplacian == "paper"))
    cu = cuda_run(X, L, n, p, K, "SGC_LL", laplacian, metric_grad, cot_Y=cY, want_res=False)
    print(sizes, compare(cu, orc, skip=("res_L", "res_W", "L_all")))


@pytest.mark.parametrize("variant,laplacian,metric_grad,with_prev", [
    ("SGC_LL", "paper", "reference", False),
    ("SGC_LL", "paper", "full", False),
    ("SGC_LL", "reference_literal", "reference", False),      # shortcut + optional outputs
    ("SGC_LL_Reslap", "reference_literal", "reference", True),
    ("SGC_LL_Reslap", "paper", "reference", False),
    ("SGC_LL_Reslap", "paper", "full", True)])
def test_big_graphs_all_modes(variant, laplacian, metric_grad, with_prev):
    """Graphs with more than 144 nodes (row-tiled sweeps, agcn_graph_big.cu) mixed with small ones, in every
    variant / semantics, including the optional res_L / res_W / L_all outputs and all gradients."""
    F, Fo, K = 16, 24, 3
    sizes = [150, 333, 20, 513, 64, 145, 4]
    Nmax = max(sizes)
    X, _, n = make_batch(sizes, F, Nmax, seed=41)
    X *= 0.6
    L = _dense_laplacians(sizes, Nmax, seed=5)
    p = O.make_params(F, Fo, K, variant, seed=17, dtype=torch.float64)
    Lprev = random_prev_laps(n, 6) if with_prev else None
    cY = _cot((len(sizes), Nmax, Fo), 3)
    cL = [_cot((int(k), int(k)), 50 + i) * 0.1 for i, k in enumerate(n)] if variant == "SGC_LL_Reslap" else None
    orc = oracle_run(X, L, n, p, K, variant, laplacian, metric_grad, Lprev, cot_Y=cY, cot_L=cL)
    cu = cuda_run(X, L, n, p, K, variant, laplacian, metric_grad, Lprev, cot_Y=cY, cot_L=cL)
    errs = compare(cu, orc)
    if metric_grad == "full":
        assert float(orc["dM_L"].abs().max()) > 0
    print(variant, laplacian, metric_grad, errs)


def test_big_graph_point_cloud_shape_paper_full():
    """ModelNet40-like first layer (xyz features, F = 3, n = 1024) with the differentiable metric, K = 2."""
    sizes = [1024, 700]
    F, Fo, K = 3, 32, 2
    X, _, n = make_batch(sizes, F, 1024, seed=2)
    L = _dense_laplacians(sizes, 1024, seed=9)
    p = O.make_params(F, Fo, K, "SGC_LL", seed=4, dtype=torch.float64)
    cY = _cot((2, 1024, Fo), 1)
    orc = oracle_run(X, L, n, p, K, "SGC_LL", "paper", "full", cot_Y=cY)
    cu = cuda_run(X, L, n, p, K, "SGC_LL", "paper", "full", cot_Y=cY)
    print(compare(cu, orc))


@pytest.mark.parametrize("laplacian,metric_grad", [("reference_literal", "reference"), ("paper", "reference"),
                                                   ("paper", "full")])
@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("sizes,F,Fo", [([132, 4, 5, 18, 33, 64, 65, 17, 96, 31], 75, 64),     # molecules: fused tiles
                                        ([300, 20, 145, 513], 16, 24)])                       # big graphs
def test_first_layer_backward_without_input_gradient(laplacian, metric_grad, K, sizes, F, Fo):
    """d_dX == NULL (the first layer of every training step: atom features have no gradient): the fused backward is
    off, the whole dYpre branch runs on the side stream and, in paper mode, dX is scratch aliasing G_0.  The
    parameter gradients must not change."""
    Nmax = max(sizes)
    X, L, n = make_batch(sizes, F, Nmax, seed=K + F, kind="tox" if F == 75 else "normal")
    if F != 75:
        X *= 0.6
        L = _dense_laplacians(sizes, Nmax, seed=4)
    p = O.make_params(F, Fo, K, "SGC_LL", seed=3 + K, dtype=torch.float64)
    cY = _cot((len(sizes), Nmax, Fo), 17)
    orc = oracle_run(X, L, n, p, K, "SGC_LL", laplacian, metric_grad, cot_Y=cY)
    if metric_grad == "full":
        # the library needs d_dX with a differentiable metric (the gradient reaches M_L through X M_L); the autograd
        # bridge allocates it even when X itself needs none
        cu = cuda_run(X, L, n, p, K, "SGC_LL", laplacian, metric_grad, cot_Y=cY, want_res=False, x_grad=False)
    else:
        cu = cuda_run(X, L, n, p, K, "SGC_LL", laplacian, metric_grad, cot_Y=cY, want_res=False, x_grad=False)
    assert "dX" not in cu
    errs = compare(cu, orc, skip=("res_L", "res_W", "L_all", "dX"))
    for k in ("dweight", "dbias", "dM_L", "dalpha"):
        assert k in errs, k
    print(laplacian, metric_grad, K, errs)


@pytest.mark.parametrize("sizes,F,Fo,K,laplacian,metric_grad", [
    ([1024, 1024, 700], 128, 128, 3, "reference_literal", "reference"),   # the shape grouped_tc_kernel is profiled on
    ([1024, 300], 128, 128, 3, "paper", "full"),
    ([4096, 50], 32, 32, 3, "reference_literal", "reference"),            # largest sweep size
    ([132, 20, 64, 9, 100, 31], 256, 256, 3, "reference_literal", "reference"),   # F = Fo = 256 on molecules
    ([132, 20, 64, 9, 100, 31], 256, 256, 2, "paper", "full"),
    ([600, 130], 256, 256, 3, "reference_literal", "reference")])          # F = Fo = 256 on big graphs
def test_named_baseline_shapes(sizes, F, Fo, K, laplacian, metric_grad):
    """Shapes BASELINE.json names that no other case reaches: N = 1024 with F = 128, N = 4096, F = Fo = 256
    (the widths the fused tile kernels hand to the split path)."""
    Nmax = max(sizes)
    X, _, n = make_batch(sizes, F, Nmax, seed=F + K)
    X *= 0.3
    L = _dense_laplacians(sizes, Nmax, seed=K + 1)
    p = O.make_params(F, Fo, K, "SGC_LL", seed=F + 2, dtype=torch.float64)
    cY = _cot((len(sizes), Nmax, Fo), 23)
    literal = laplacian == "reference_literal"
    orc = oracle_run(X, L, n, p, K, "SGC_LL", laplacian, metric_grad, cot_Y=cY, compute_similarity=not literal)
    cu = cuda_run(X, L, n, p, K, "SGC_LL", laplacian, metric_grad, cot_Y=cY, want_res=False)
    errs = compare(cu, orc, skip=("res_L", "res_W", "L_all"))
    print(sizes, F, Fo, K, laplacian, errs)


@pytest.mark.parametrize("Fh,Fm,Nt,kind", [(64, 256, 1234, "sigmoid_ce"), (32, 64, 40, "sigmoid_ce"),
                                           (128, 132, 50, "sigmoid_ce"), (64, 256, 24, "sigmoid_ce"),
                                           (64, 256, 40, "softmax_ce"), (64, 128, 26, "softmax_ce"),
                                           (256, 64, 6, "softmax_ce")])
def test_head_loss_and_gradients_match_oracle(Fh, Fm, Nt, kind):
    """agcn_head_loss_grad_ex (DenseMol + GraphGatherMol + logits + loss, SURVEY.md section 8f rows 1 and 3) against
    oracle/network_oracle.py in fp64: the multitask sigmoid heads (incl. Tox21's 12 tasks = 24 logits, below one
    tensor-core k-block) and the single-task softmax head of the point-cloud networks."""
    import agcn_b200
    from agcn_b200.functional import head_loss
    from oracle import network_oracle as NO
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(Fh + Nt)
    n = np.array(SIZES + [7, 1, 20, 19, 44], np.int32)
    B, R = len(n), int(n.sum())
    batch = agcn_b200.GraphBatch(n, 132, device=dev)
    H64 = torch.tensor(np.maximum(rng.standard_normal((R, Fh)), 0) * 0.3, dtype=torch.float64)
    p64 = [torch.tensor(rng.standard_normal(s) * sc, dtype=torch.float64)
           for s, sc in (((Fh, Fm), 0.1), ((Fm,), 0.05), ((Fm, Nt), 0.1), ((Nt,), 0.1))]
    scale, up = 1.0 / 37.0, 1.7
    Hr = H64.clone().requires_grad_(True)
    pr = [t.clone().requires_grad_(True) for t in p64]
    off = np.concatenate([[0], np.cumsum(n)])
    H_list = [Hr[off[g]:off[g + 1]] for g in range(B)]
    if kind == "sigmoid_ce":
        y = torch.tensor((rng.random((B, Nt)) < 0.3).astype(np.float64))
        w = torch.tensor(rng.random((B, Nt)) + 0.5)
        loss_ref = NO.head_loss(H_list, pr[0], pr[1], pr[2], pr[3], y, w, scale)
    else:
        y = torch.zeros(B, Nt, dtype=torch.float64)
        y[torch.arange(B), torch.tensor(rng.integers(0, Nt, B))] = 1.0
        w = torch.tensor(rng.random(B) + 0.5)
        mol = torch.tanh(torch.stack([(h @ pr[0] + pr[1]).sum(0) for h in H_list]))
        logits = mol @ pr[2] + pr[3]
        loss_ref = ((torch.logsumexp(logits, 1) - (logits * y).sum(1)) * w).sum() * scale
    (loss_ref * up).backward()
    Hc = H64.float().to(dev).requires_grad_(True)
    pc = [t.float().to(dev).requires_grad_(True) for t in p64]
    loss = head_loss(Hc, pc[0], pc[1], pc[2], pc[3], y.float().to(dev), w.float().to(dev), batch, scale,
                     loss_kind=kind)
    (loss * up).backward()
    torch.cuda.synchronize()
    assert abs(float(loss) - float(loss_ref)) <= TOL * abs(float(loss_ref))
    assert O.rel_err(Hc.grad.cpu(), Hr.grad) <= TOL
    for a, b, name in zip(pc, pr, ("dense_W", "dense_b", "head_W", "head_b")):
        assert O.rel_err(a.grad.cpu(), b.grad) <= TOL, name


_UNIFORM_SHAPES = [([256, 256, 256], 64), ([384, 384], 160), ([256], 16), ([1024, 1024], 128)]


@pytest.mark.parametrize("sizes,F,impl", [(s, F, impl) for s, F in _UNIFORM_SHAPES for impl in (1, 2, 4)] +
                         [([256, 256], 8, impl) for impl in (1, 3)])
def test_uniform_tensor_core_product(sizes, F, impl):
    """Each row-tiled product kernel on equal-size graphs, chosen through the debug entry: impl 1 = the SIMT kernel
    (grouped_lap_gemm_kernel), 2 = bt::grouped_tc_kernel, 3 = the streaming kernel for F <= 8 (bt::grouped_thin_kernel),
    4 = bt::grouped_tcu_kernel (TMA-staged L tiles, A operand in tensor memory) forced whatever the grid size.  Every
    op(L) variant, against a float64 product on the device."""
    import ctypes
    import agcn_b200
    from agcn_b200 import _lib
    from agcn_b200.batch import _ptr, _stream_ptr
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(5)
    batch = agcn_b200.GraphBatch(sizes, max(sizes), device=dev)
    R = batch.total_nodes
    L = torch.randn(batch.total_lap, device=dev, generator=gen) * 0.1
    X = torch.randn(R, F, device=dev, generator=gen)
    for transL in (0, 1):
        for add_identity in (0, 1):
            ref = torch.zeros(R, F, device=dev, dtype=torch.float64)
            for g, n in enumerate(sizes):
                Lg = batch.lap_view(L, g).double()
                Lg = Lg.t() if transL else Lg
                if add_identity:
                    Lg = Lg + torch.eye(n, device=dev, dtype=torch.float64)
                r0 = int(batch.node_off[g])
                ref[r0:r0 + n] = 2.0 * (Lg @ X[r0:r0 + n].double())
            out = torch.full((R, F), float("nan"), device=dev)
            _lib.check(_lib.lib().agcn_debug_grouped_product(batch.handle, _ptr(L), _ptr(X), _ptr(out), F, transL,
                                                             add_identity, 2.0, impl, _stream_ptr()))
            torch.cuda.synchronize()
            assert torch.isfinite(out).all()
            err = float((out.double() - ref).abs().max() / ref.abs().max())
            assert err <= 1e-5, (sizes, F, impl, transL, add_identity, err)


@pytest.mark.parametrize("metric_grad", ["reference", "full"])
def test_equal_size_big_graphs_metric_block_with_near_duplicates(metric_grad):
    """Paper semantics on equal-size big graphs: the pair matrices come from bt::pair_tcu_kernel (Gram tiles on the tensor
    cores).  Exact duplicates, near-duplicates (0.04 .. 0.8 apart at norms of ~3, where the Gram expansion cancels: SURVEY Q7) and far
    rows in one batch: similarity, Laplacian and every gradient within the layer's budget."""
    sizes, F, Fo, K = [256, 256], 64, 32, 3
    Nmax = max(sizes)
    X, _, n = make_batch(sizes, F, Nmax, seed=23)
    X *= 0.4
    rng = np.random.default_rng(4)
    for g in range(len(sizes)):
        X[g, 9] = X[g, 5]                                                   # exact duplicates
        X[g, 200] = X[g, 5]
        # (closer pairs than ~5e-3 make 1 / dist amplify the fp32 error of ANY dL by > 1e3: not a layer-budget case)
        for a, b, eps in ((11, 7, 1e-2), (40, 41, 3e-2), (100, 180, 1e-1), (33, 250, 5e-3)):
            X[g, a] = X[g, b] + (rng.standard_normal(F) * eps).astype(np.float32)
    L = _dense_laplacians(sizes, Nmax, seed=6)
    p = O.make_params(F, Fo, K, "SGC_LL", seed=3, dtype=torch.float64)
    cY = _cot((len(sizes), Nmax, Fo), 29)
    orc = oracle_run(X, L, n, p, K, "SGC_LL", "paper", metric_grad, cot_Y=cY)
    cu = cuda_run(X, L, n, p, K, "SGC_LL", "paper", metric_grad, cot_Y=cY)
    errs = compare(cu, orc)
    print(metric_grad, errs)
