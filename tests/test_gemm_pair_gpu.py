"""GPU parity of the cases the CTA-pair split of the GEMM introduces: each 256 x BN output tile is computed by two SMs (the even CTA
owns rows 0-127, the odd CTA rows 128-255, each loads half of B), so the odd CTA's rows may be partly or wholly beyond M, the grid
can be smaller than the number of pair slots, split-K divides K per pair unit, and the persistent state of the epilogue (bias slice
rotation, cross-tile aux prefetch) runs over several pair tiles per cluster.  Checked against fp32 torch with the tolerances of
test_gemm_gpu.py."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _k():
    from deeplearningexamples_b200 import kernels, _lib
    return kernels, _lib


def _rand(shape, scale=1.0, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(shape, generator=g, device="cuda") * scale).to(torch.bfloat16)


def _close(got, want, rtol=1e-2, atol=None):
    want = want.float(); got = got.float()
    atol = atol if atol is not None else 1e-2 * want.abs().max().item() + 1e-6
    torch.testing.assert_close(got, want, rtol=rtol, atol=atol)


def _operand(rows, K, mn, scale, seed):
    """[rows, K] (K-major) or [K, rows] (MN-major) as a view of a wider buffer whose row stride is a multiple of 8 elements, so that
    any `rows` is allowed; returns (tensor for the kernel, the [rows, K] matrix it stands for)."""
    if not mn:
        t = _rand((rows, K), scale, seed)
        return t, t.float()
    wide = _rand((K, (rows + 7) // 8 * 8), scale, seed)
    t = wide[:, :rows]
    return t, t.float().t()


@pytest.mark.parametrize("M", [128, 384, 130])
@pytest.mark.parametrize("a_mn,b_mn", [(False, False), (False, True), (True, False), (True, True)])
@pytest.mark.parametrize("N", [128, 384])
def test_odd_cta_rows_out_of_range(M, a_mn, b_mn, N):
    """M = 128: the odd CTA's rows are all beyond M; 384: the second pair tile has only the even CTA's rows; 130: two rows for the
    odd CTA.  N = 384 at BN = 256 leaves the odd CTA's half of B out of range in the last column tile; N = 128 runs BN = 128."""
    k, L = _k()
    K = 200
    a, af = _operand(M, K, a_mn, 1.0, seed=100 + M)
    b, bf = _operand(N, K, b_mn, 0.05, seed=200 + N)
    bias = _rand((N,), seed=300)
    out = k.gemm(a, b, a_layout=L.LAYOUT_MN if a_mn else L.LAYOUT_K, b_layout=L.LAYOUT_MN if b_mn else L.LAYOUT_K, bias=bias)
    _close(out, af @ bf.t() + bias.float())


def test_fewer_pair_units_than_slots():
    """4 pair tiles on a GPU with many more pair slots; the output beyond the matrix (a column slice of a wider buffer) is untouched."""
    k, L = _k()
    a, w = _rand((512, 320), seed=110), _rand((512, 320), 0.05, seed=111)
    buf = torch.zeros((512, 1024), device="cuda", dtype=torch.bfloat16)
    k.gemm(a, w, out=buf[:, 256:768])
    _close(buf[:, 256:768], a.float() @ w.float().t())
    assert buf[:, :256].abs().max().item() == 0.0 and buf[:, 768:].abs().max().item() == 0.0


@pytest.mark.parametrize("M,N,K", [(384, 264, 1000), (130, 512, 4040), (1024, 1024, 2500)])
@pytest.mark.parametrize("splits", [1, 3, 8])
def test_split_k_on_pair_units(M, N, K, splits):
    """split-K divides the k-blocks of each pair unit (K not a multiple of 64: a partial last k-block in the last split)."""
    k, L = _k()
    dy, dyf = _operand(M, K, True, 1.0, seed=120)
    x, xf = _operand(N, K, True, 1.0, seed=121)
    out = k.gemm(dy, x, a_layout=L.LAYOUT_MN, b_layout=L.LAYOUT_MN, epilogue=L.EPI_ATOMIC_F32, splits=splits)
    want = dyf @ xf.t()
    torch.testing.assert_close(out, want, rtol=1e-3, atol=1e-3 * want.abs().max().item())


@pytest.mark.parametrize("tile_n", [256, 128])
def test_every_epilogue_several_pair_tiles_per_cluster(tile_n):
    """3-4 pair tiles per cluster (sized from the device's SM count), a bias that differs per column tile, every epilogue."""
    k, L = _k()
    slots = torch.cuda.get_device_properties(0).multi_processor_count // 2
    N, K = 4 * tile_n, 192
    M = -(-(7 * slots) // 8) * 256 - 96            # 3.5 pair tiles per cluster over 4 column tiles, the last pair tile ragged
    a, w = _rand((M, K), seed=130), _rand((N, K), 0.1, seed=131)
    bias = (_rand((N,), 1.0, seed=132).float() + torch.arange(N, device="cuda").float() / N).to(torch.bfloat16)
    res = _rand((M, N), 1.0, seed=133)
    base = a.float() @ w.float().t()
    tn = 0 if tile_n == 256 else 128
    _close(k.gemm(a, w, bias=bias, tile_n=tn), base + bias.float())
    _close(k.gemm(a, w, bias=bias, aux=res, epilogue=L.EPI_BIAS_DROPOUT_RESIDUAL, dropout_p=0.0, tile_n=tn), base + bias.float() + res.float())
    g, u = k.gemm(a, w, bias=bias, epilogue=L.EPI_BIAS_GELU, tile_n=tn)
    _close(u, base + bias.float())
    _close(g, torch.nn.functional.gelu(u.float(), approximate="tanh"), rtol=1e-2, atol=1e-2)
    _close(k.gemm(a, w, aux=res, epilogue=L.EPI_ADD, tile_n=tn), base + res.float())
    cs = torch.zeros(N, device="cuda")
    out = k.gemm(a, w, aux=res, epilogue=L.EPI_DGELU, colsum_out=cs, tile_n=tn)
    rf = res.float().requires_grad_(True)
    torch.nn.functional.gelu(rf, approximate="tanh").sum().backward()
    _close(out, base * rf.grad)
    torch.testing.assert_close(cs, out.float().sum(dim=0), rtol=1e-3, atol=1e-2 * out.float().abs().sum(dim=0).max().item())
    ref = base + bias.float()
    torch.testing.assert_close(k.gemm(a, w, bias=bias, epilogue=L.EPI_F32, tile_n=tn), ref, rtol=1e-4, atol=1e-3)
    _close(k.gemm(a, w, bias=bias, epilogue=L.EPI_BIAS_TANH, tile_n=tn), torch.tanh(ref))
    acc = k.gemm(a, w, epilogue=L.EPI_ATOMIC_F32, splits=2, tile_n=tn)
    torch.testing.assert_close(acc, base, rtol=1e-3, atol=1e-3 * base.abs().max().item())


def test_dropout_mask_independent_of_tiling():
    """The dropout RNG is keyed by the global row and column, so BN = 128 and BN = 256 tilings keep the same elements; the keep rate
    is within the bound of test_gemm_gpu.py."""
    k, L = _k()
    M, N, K = 65536, 1024, 64
    a, w = _rand((M, K), seed=140), _rand((N, K), 0.1, seed=141)
    bias, res = _rand((N,), seed=142), _rand((M, N), seed=143)
    kw = dict(bias=bias, aux=res, epilogue=L.EPI_BIAS_DROPOUT_RESIDUAL, dropout_p=0.1, seed=99, dropout_stream=3)
    o256 = k.gemm(a, w, tile_n=0, **kw)
    o128 = k.gemm(a, w, tile_n=128, **kw)
    base = a.float() @ w.float().t() + bias.float()
    sure = base.abs() > 0.5                     # where a kept element cannot round back to the residual
    dropped256 = (o256 == res) & sure
    assert torch.equal(dropped256, (o128 == res) & sure)
    frac = dropped256.float().sum() / sure.float().sum()
    assert 0.08 < frac.item() < 0.12
