"""The node GEMMs of include/agcn_sgcll.h against a float64 product on the device, on every engine they dispatch to.

agcn_node_gemm  C (+)= act(scale * A op(B) + bias) over M packed rows:
                  tcgen05 3xTF32  Kd >= 32, A 16-byte aligned, lda % 4 == 0;
                  gemm_rows, vector loads   otherwise, when Kd, lda, ldb (and N unless transB) are multiples of 4 and
                                            A / B are 16-byte aligned;
                  gemm_rows, scalar loads   everything else (here: A offset by one float).
agcn_gemm_tn    out[(f*S + s)*N + c] = sum_r A_s[r, f] D[r, c], tcgen05 (use_tensor_cores = 1) or CUDA cores (0), both
                a chunked contraction over the rows followed by a fixed-order reduction of the chunks; -1 takes the
                library's choice (tcgen05 for M >= 32, Kd <= 128, Kd and N multiples of 4, aligned operands).

Shapes are the ones where tiles go wrong: M = 1 and M just off a 128-row tile, N above 128 and not a multiple of 128,
Kd not a multiple of 4 on the tensor cores, row pitches larger than the width (lda > Kd, ldc > N), transB, S > 1 and
row counts that are not a multiple of 32.  C is pre-filled with a sentinel: the pitch columns beyond N and the rows
beyond M must still hold it, bit for bit.  The scratch buffers are filled with NaN bytes first.

Budget: max-abs error over max-abs reference <= 1e-5 (test_uniform_tensor_core_product's).  Worst case observed on
one NVIDIA B200 (1000 W power limit) over the whole grid, as the tests print it per engine:

    agcn_node_gemm  tcgen05 4.2e-6, gemm_rows vector 1.5e-7, gemm_rows scalar 3.1e-6
    agcn_gemm_tn    tcgen05 2.0e-6, CUDA cores 4.8e-7

The engine a case is labelled with is checked against the kernels the CUDA profiler sees, so that a change of the
dispatch rules cannot quietly move the grid off an engine.
"""
import re

import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
BUDGET = 1e-5
SENTINEL = 0x7FC0FFEE       # a quiet-NaN bit pattern no kernel computes

NODE_M = (1, 31, 128, 129, 1000)
NODE_N = (1, 30, 64, 65, 160, 257)
NODE_KD = (16, 30, 32, 33, 75, 128, 160)
EPILOGUES = ("plain", "bias_relu", "scale_accumulate")


def _lib():
    from agcn_b200 import _lib
    return _lib


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr() if t is not None else 0)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)


def _operand(shape, gen):
    """Uniform in [-0.75, 1.25): signs of both kinds (relu clips), but no output is a near-cancelling sum."""
    return (torch.rand(shape, generator=gen, dtype=torch.float64) * 2 - 0.75).float()


def _place(t, pitch, offset):
    """t [rows, cols] copied into a fresh device buffer with row pitch `pitch`, starting `offset` floats in (a nonzero
    offset leaves the operand 4-byte but not 16-byte aligned); the pitch columns hold NaN.  Returns the buffer from
    the operand's first element on."""
    rows, cols = t.shape
    buf = torch.full((offset + rows * pitch + 8,), float("nan"), device=DEV)
    view = buf[offset:offset + rows * pitch].view(rows, pitch)
    view[:, :cols] = t.to(DEV)
    return buf[offset:]


def node_engine(M, N, Kd, lda, ldb, transB, a_offset):
    """The engine agcn_node_gemm dispatches to (tc_gemm_supported / gemm_rows in the sources)."""
    a_aligned = a_offset % 4 == 0
    if Kd >= 32 and a_aligned and lda % 4 == 0:
        return "tcgen05"
    vec = Kd % 4 == 0 and lda % 4 == 0 and a_aligned and ldb % 4 == 0 and (transB or N % 4 == 0)
    return "gemm_rows vector" if vec else "gemm_rows scalar"


def _node_case(M, N, Kd, transB, epilogue, pitched, a_offset, gen, scratch):
    lib = _lib().lib()
    lda = ((Kd + 1 + 3) // 4) * 4 if pitched else Kd            # Kd = 33 -> 36, 75 -> 76
    ldc = (N + 4 if N % 4 == 0 else N + 3) if pitched else N
    ldb = Kd if transB else N
    A = _operand((M, Kd), gen)
    Bm = _operand((N, Kd) if transB else (Kd, N), gen)
    A_dev = _place(A, lda, a_offset)
    B_dev = Bm.to(DEV).contiguous()
    bias = _operand((N,), gen).to(DEV) if epilogue == "bias_relu" else None
    scale = torch.tensor([0.625], device=DEV) if epilogue == "scale_accumulate" else None
    accumulate = epilogue == "scale_accumulate"
    act = "relu" if epilogue == "bias_relu" else "linear"
    # C: M rows of pitch ldc and two guard rows after them, all holding the sentinel; the accumulated block starts
    # from values of its own
    C = torch.full(((M + 2) * ldc,), SENTINEL, dtype=torch.int32, device=DEV).view(torch.float32).view(M + 2, ldc)
    C0 = _operand((M, N), gen).to(DEV)
    if accumulate:
        C[:M, :N] = C0
    scratch.view(torch.uint8).fill_(0xFF)
    _lib().check(lib.agcn_node_gemm(_ptr(A_dev), lda, _ptr(B_dev), ldb, transB, _ptr(C), ldc, M, N, Kd, _ptr(bias),
                                    _ptr(scale), 1 if accumulate else 0, _lib().ACT[act], _ptr(scratch), _stream()))
    ref = A.to(DEV).double() @ (Bm.to(DEV).double().t() if transB else Bm.to(DEV).double())
    if scale is not None:
        ref = ref * scale.double()
    if bias is not None:
        ref = ref + bias.double()
    if accumulate:
        ref = ref + C0.double()
    if act == "relu":
        ref = ref.clamp_min(0.0)
    got = C[:M, :N].double()
    err = float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30))
    bits = C.view(torch.int32)
    untouched = bool((bits[M:] == SENTINEL).all()) and bool((bits[:M, N:] == SENTINEL).all())
    return err, untouched, node_engine(M, N, Kd, lda, ldb, transB, a_offset)


@pytest.mark.parametrize("epilogue", EPILOGUES)
@pytest.mark.parametrize("transB", (0, 1))
def test_node_gemm_matches_fp64(transB, epilogue):
    """Every M x N x Kd of the grid, contiguous and pitched (lda > Kd, ldc > N), with A 16-byte aligned and offset by
    one float: on tcgen05 where the shape allows it, on gemm_rows (vector and scalar loads) otherwise."""
    lib = _lib().lib()
    gen = torch.Generator().manual_seed(17 + 2 * transB + EPILOGUES.index(epilogue))
    scratch = torch.empty(lib.agcn_node_gemm_scratch_bytes(max(NODE_N), max(NODE_KD)) // 4 + 1, device=DEV)
    worst, bad = {}, []
    for M in NODE_M:
        for N in NODE_N:
            for Kd in NODE_KD:
                for pitched in (False, True):
                    for a_offset in (0, 1):
                        err, untouched, engine = _node_case(M, N, Kd, transB, epilogue, pitched, a_offset, gen,
                                                            scratch)
                        worst[engine] = max(worst.get(engine, 0.0), err)
                        if not (err <= BUDGET and untouched):
                            bad.append((M, N, Kd, "pitched" if pitched else "contiguous", a_offset, engine,
                                        "%.2e" % err, "sentinel ok" if untouched else "SENTINEL OVERWRITTEN"))
    torch.cuda.synchronize()
    print("transB", transB, epilogue, {k: "%.2e" % v for k, v in sorted(worst.items())})
    assert sorted(worst) == ["gemm_rows scalar", "gemm_rows vector", "tcgen05"]
    assert not bad, "%d failing shapes (M, N, Kd, pitch, A offset, engine, error, C pad): %s" % (len(bad), bad[:20])


TN_TC = dict(M=(32, 33, 100, 4097), Kd=(4, 36, 64, 128), N=(4, 60, 64, 68, 132, 260))
TN_CUDA = dict(M=(1, 32, 33, 100, 4097), Kd=(4, 36, 64, 75, 128, 200), N=(4, 30, 60, 64, 68, 132, 260))


def _tn_case(M, Kd, N, S, use_tc, gen):
    lib = _lib().lib()
    A = _operand((S * M, Kd), gen).to(DEV)          # A_0 = rows [0, M), the S - 1 extra slices contiguous after it
    D = _operand((M, N), gen).to(DEV)
    A1 = A[M:] if S > 1 else None
    scratch = torch.empty(lib.agcn_gemm_tn_scratch_bytes(M, Kd, N, S), dtype=torch.uint8, device=DEV)
    outs = []
    for _ in range(2):
        scratch.fill_(0xFF)
        out = torch.full((Kd * S * N,), float("nan"), device=DEV)
        _lib().check(lib.agcn_gemm_tn(_ptr(A), _ptr(A1), _ptr(D), _ptr(out), M, Kd, N, S, _ptr(scratch), use_tc,
                                      _stream()))
        outs.append(out)
    ref = torch.einsum("srf,rc->fsc", A.double().view(S, M, Kd), D.double()).reshape(-1)
    err = float((outs[0].double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))
    return err, torch.equal(outs[0], outs[1]), outs[0]


@pytest.mark.parametrize("use_tc", (1, 0), ids=("tcgen05", "cuda_cores"))
def test_gemm_tn_matches_fp64_and_is_deterministic(use_tc):
    """Both engines over their grids at S = 1 and S = 3: within budget, and two identical calls give the same bits."""
    grid = TN_TC if use_tc else TN_CUDA
    gen = torch.Generator().manual_seed(29 + use_tc)
    worst, bad = 0.0, []
    for M in grid["M"]:
        for Kd in grid["Kd"]:
            for N in grid["N"]:
                for S in (1, 3):
                    err, same, _ = _tn_case(M, Kd, N, S, use_tc, gen)
                    worst = max(worst, err)
                    if not (err <= BUDGET and same):
                        bad.append((M, Kd, N, S, "%.2e" % err, "deterministic" if same else "NOT DETERMINISTIC"))
    torch.cuda.synchronize()
    print("gemm_tn", "tcgen05" if use_tc else "cuda cores", "worst %.2e" % worst)
    assert not bad, "%d failing shapes (M, Kd, N, S, error, repeat): %s" % (len(bad), bad[:20])


def _kernels(fn):
    """Names of the library's GEMM kernels that fn() launches, as the CUDA profiler reports them."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.key for e in prof.key_averages() if re.search(r"gemm_rows_kernel|gemm_tn_kernel|tc_gemm_kernel", e.key)}


def _engine_of(names):
    found = set()
    for n in names:
        if "tc_gemm_kernel" in n or "tc_gemm_tn_kernel" in n:
            found.add("tcgen05")
        elif re.search(r"gemm_rows_kernel(<true|ILb1)", n):
            found.add("gemm_rows vector")
        elif re.search(r"gemm_rows_kernel(<false|ILb0)", n):
            found.add("gemm_rows scalar")
        elif "gemm_tn_kernel" in n:
            found.add("cuda cores")
    return found


ENGINE_CASES = [
    # M, N, Kd, transB, pitched, A offset
    (129, 257, 33, 1, True, 0),     # tcgen05: Kd % 4 != 0 with lda = 36, transB, N > 128 off a 128-column tile
    (31, 160, 75, 0, True, 0),      # tcgen05: lda = 76
    (129, 64, 16, 0, False, 0),     # gemm_rows vector loads
    (1000, 30, 16, 1, True, 0),     # gemm_rows vector loads, transB
    (129, 65, 75, 0, True, 1),      # gemm_rows scalar loads: A misaligned
    (128, 64, 30, 1, False, 0),     # gemm_rows scalar loads: Kd % 4 != 0 below 32
]

TN_ENGINE_CASES = [
    # M, Kd, N, S, engine of use_tensor_cores = -1 (the library's choice)
    (100, 36, 68, 3, "tcgen05"),
    (100, 132, 68, 1, "cuda cores"),   # Kd > 128
    (100, 36, 66, 1, "cuda cores"),    # N % 4 != 0
    (31, 36, 68, 1, "cuda cores"),     # M < 32
]


def test_engines_are_the_ones_the_grid_is_labelled_with():
    lib = _lib().lib()
    gen = torch.Generator().manual_seed(3)
    scratch = torch.empty(lib.agcn_node_gemm_scratch_bytes(max(NODE_N), max(NODE_KD)) // 4 + 1, device=DEV)
    for M, N, Kd, transB, pitched, off in ENGINE_CASES:
        label = []
        names = _kernels(lambda: label.append(_node_case(M, N, Kd, transB, "plain", pitched, off, gen, scratch)[2]))
        assert _engine_of(names) == {label[0]}, (M, N, Kd, transB, pitched, off, label[0], names)
    # agcn_gemm_tn on each engine it takes; the library's choice must give the bits of the engine it names
    for M, Kd, N, S, auto in TN_ENGINE_CASES:
        outs = {}
        for use_tc, want in ((1, "tcgen05"), (0, "cuda cores"), (-1, auto)):
            run = lambda: outs.setdefault(use_tc, _tn_case(M, Kd, N, S, use_tc, torch.Generator().manual_seed(M + Kd))[2])
            if use_tc == 1 and auto != "tcgen05":
                with pytest.raises(_lib().AgcnError, match="not supported by the tensor-core kernel"):
                    run()
                continue
            names = _kernels(run)
            assert _engine_of(names) == {want}, (M, Kd, N, S, use_tc, names)
        same = outs[1 if auto == "tcgen05" else 0]
        assert torch.equal(outs[-1].view(torch.int32), same.view(torch.int32)), (M, Kd, N, S)
