"""tcgen05 dense transform (TF32x3 and BF16 modes) vs the exact fp32 SIMT path, through the C ABI."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _dense(lib, a, w, b, act, precision, accumulate=None):
    from bikg_graph_explainability_public_b200 import _lib

    m, k = a.shape
    n = w.shape[0]
    out = torch.zeros((m, n), device="cuda") if accumulate is None else accumulate.clone()
    _lib.check(lib.xpgnn_dense_rows(a.data_ptr(), m, k, k, w.data_ptr(), _lib.dptr(b), n, act, out.data_ptr(), n,
                                    int(accumulate is not None), precision, _lib.stream_ptr()))
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("m,k,n", [(1000, 128, 128), (4096, 64, 16), (300, 32, 40), (129, 256, 64), (70000, 128, 128)])
def test_tensor_core_dense_matches_fp32(lib, m, k, n):
    g = torch.Generator(device="cuda").manual_seed(m + k + n)
    a = torch.randn(m, k, device="cuda", generator=g)
    w = torch.randn(n, k, device="cuda", generator=g) / k ** 0.5
    b = torch.randn(n, device="cuda", generator=g)
    ref = (a.double() @ w.double().T + b.double())
    simt = _dense(lib, a, w, b, 0, 0)
    assert torch.allclose(simt.double(), ref, rtol=1e-5, atol=1e-5)
    scale = float(ref.abs().max())
    x3 = _dense(lib, a, w, b, 0, 2)
    err3 = float((x3.double() - ref).abs().max()) / scale
    assert err3 < 2e-6, "TF32x3 error %g" % err3
    bf = _dense(lib, a, w, b, 0, 1)
    errb = float((bf.double() - ref).abs().max()) / scale
    assert errb < 2e-2, "bf16 error %g" % errb
    # fused epilogue: accumulate + ReLU, no bias
    prev = torch.randn(m, n, device="cuda", generator=g)
    ref2 = torch.relu(prev.double() + a.double() @ w.double().T)
    y = _dense(lib, a, w, None, 1, 2, accumulate=prev)
    assert float((y.double() - ref2).abs().max()) / scale < 2e-6


SENTINEL = -12345.0
BARS = {0: 2e-6, 2: 2e-6, 1: 2e-2}  # SIMT (exact fp32 FMAs), TF32x3, bf16: error / max |reference|


def _dense_strided(lib, rows, k, n, ld_in, ld_out, act, precision, seed, accumulate=False):
    """in [rows, ld_in] with NaN in the columns k .. ld_in (a read past k poisons the result), out [rows, ld_out] with a
    sentinel in the columns n .. ld_out (a write past n_out overwrites it).  Returns (rc, out, float64 reference)."""
    from bikg_graph_explainability_public_b200 import _lib

    g = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.full((max(rows, 1), ld_in), float("nan"), device="cuda")
    a[:, :k] = torch.randn(max(rows, 1), k, device="cuda", generator=g)
    w = torch.randn(n, k, device="cuda", generator=g) / k ** 0.5
    b = torch.randn(n, device="cuda", generator=g)
    out = torch.full((max(rows, 1), ld_out), SENTINEL, device="cuda")
    prev = torch.randn(max(rows, 1), n, device="cuda", generator=g)
    if accumulate:
        out[:, :n] = prev
    ref = a[:, :k].double() @ w.double().T + b.double() + (prev.double() if accumulate else 0.0)
    ref = {0: ref, 1: torch.relu(ref), 2: torch.sigmoid(ref)}[act]
    rc = lib.xpgnn_dense_rows(a.data_ptr(), rows, k, ld_in, w.data_ptr(), b.data_ptr(), n, act, out.data_ptr(), ld_out,
                              int(accumulate), precision, _lib.stream_ptr())
    torch.cuda.synchronize()
    return rc, out[:max(rows, 1)], ref[:rows]


@pytest.mark.parametrize("precision", [0, 2, 1])
@pytest.mark.parametrize("rows,k,n,act", [(1, 64, 64, 2), (127, 32, 8, 0), (128, 64, 255, 2), (129, 32, 256, 1),
                                          (1000, 160, 8, 2), (3000, 64, 256, 0)])
def test_dense_rows_strides_edges_and_sigmoid(lib, rows, k, n, act, precision):
    """ld_in > k and ld_out > n_out, rows around one 128-row tile, n_out 8 / 255 / 256 (tensor-core limits; at 256
    columns the TF32x3 weight image fits shared memory up to k = 64), sigmoid:
    against float64 a @ w.T + b; the padding columns of the input are never read, the guard columns never written."""
    rc, out, ref = _dense_strided(lib, rows, k, n, k + 4, n + 4, act, precision, seed=rows + k + n)
    assert rc == 0, lib.xpgnn_last_error()
    assert bool(torch.isfinite(out[:, :n]).all()), "a padding column of the input was read"
    assert bool((out[:, n:] == SENTINEL).all()), "a guard column of the output was written"
    err = float((out[:, :n].double() - ref).abs().max()) / max(float(ref.abs().max()), 1e-30)
    assert err < BARS[precision], (precision, err)


@pytest.mark.parametrize("precision", [2, 1])
def test_dense_rows_accumulate(lib, precision):
    """accumulate = 1: out = act(out + in w^T + b) in the tensor-core modes (bf16 included), strided."""
    rc, out, ref = _dense_strided(lib, 300, 64, 40, 68, 44, 1, precision, seed=5, accumulate=True)
    assert rc == 0, lib.xpgnn_last_error()
    assert bool((out[:, 40:] == SENTINEL).all())
    err = float((out[:, :40].double() - ref).abs().max()) / float(ref.abs().max())
    assert err < BARS[precision], (precision, err)


@pytest.mark.parametrize("k,n", [(64, 257), (48, 64), (100, 16)])
def test_dense_rows_shapes_outside_the_tensor_core_path(lib, k, n):
    """n_out > 256 or k % 32 != 0: the tensor-core modes refuse the call with an error and write nothing; the SIMT
    mode computes it."""
    for precision in (2, 1):
        rc, out, _ = _dense_strided(lib, 200, k, n, k + 4, n + 4, 0, precision, seed=k + n)
        assert rc != 0
        assert bool((out == SENTINEL).all()), "a refused call wrote its output"
    rc, out, ref = _dense_strided(lib, 200, k, n, k + 4, n + 4, 0, 0, seed=k + n)
    assert rc == 0, lib.xpgnn_last_error()
    assert bool((out[:, n:] == SENTINEL).all())
    assert float((out[:, :n].double() - ref).abs().max()) / float(ref.abs().max()) < BARS[0]


@pytest.mark.parametrize("precision", [0, 2, 1])
def test_dense_rows_zero_rows_is_a_no_op(lib, precision):
    """rows = 0 is a valid empty call in every mode: success, nothing written."""
    rc, out, _ = _dense_strided(lib, 0, 64, 64, 68, 68, 0, precision, seed=1)
    assert rc == 0, lib.xpgnn_last_error()
    assert bool((out == SENTINEL).all())
