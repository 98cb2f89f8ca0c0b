"""Recompute-stage kernels against plain PyTorch fp32 references of the same op (called through
the C-ABI test hooks with device pointers)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _gelu(x):
    return torch.nn.functional.gelu(x)


@pytest.mark.parametrize("M", [1, 37, 128, 129, 1000, 4096 + 77, 148 * 128 * 3 + 5])
@pytest.mark.parametrize("N,K,epi", [(384, 384, 0), (1152, 384, 0), (1536, 384, 0), (384, 1536, 0),
                                     (1536, 384, 1),                  # GELU epilogue: only the FFN up-projection uses it
                                     (384, 384, 2), (384, 1536, 2)])  # residual epilogue: only the H-wide projections
def test_gemm_tcgen05_vs_torch(lib, cuda_ok, M, N, K, epi):
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N + K + epi)
    A = (torch.randn(M, K, device="cuda", generator=g) * 1.0).half()
    W = (torch.randn(N, K, device="cuda", generator=g) * 0.05).half()
    bias = torch.randn(N, device="cuda", generator=g) * 0.1
    res = torch.randn(M, N, device="cuda", generator=g).half()
    C = torch.full((M, N), float("nan"), device="cuda", dtype=torch.float16)
    rc = lib.lb2_test_gemm_f16(A.data_ptr(), W.data_ptr(), bias.data_ptr(), res.data_ptr(), C.data_ptr(), M, N, K, epi)
    assert rc == 0, lib.lb2_last_error()
    ref = A.float() @ W.float().T + bias
    if epi == 1:
        ref = _gelu(ref)
    if epi == 2:
        ref = ref + res.float()
    err = (C.float() - ref).abs()
    tol = 2e-3 + 1.5e-3 * ref.abs()  # fp16 output rounding (2^-11 relative) + accumulation-order noise
    assert torch.isfinite(C).all()
    assert (err <= tol).all(), f"max err {err.max().item()} at {torch.nonzero(err > tol)[:3].tolist()}"


@pytest.mark.parametrize("M", [5, 300, 20000])
def test_gemm_grouped_head_major_output(lib, cuda_ok, M):
    N, K, G = 1152, 384, 96
    g = torch.Generator(device="cuda").manual_seed(M)
    A = torch.randn(M, K, device="cuda", generator=g).half()
    W = (torch.randn(N, K, device="cuda", generator=g) * 0.05).half()
    bias = torch.randn(N, device="cuda", generator=g) * 0.1
    C = torch.full((N // G, M, G), float("nan"), device="cuda", dtype=torch.float16)
    assert lib.lb2_test_gemm_grouped_f16(A.data_ptr(), W.data_ptr(), bias.data_ptr(), C.data_ptr(), M, N, K, G) == 0, lib.lb2_last_error()
    ref = (A.float() @ W.float().T + bias).view(M, N // G, G).permute(1, 0, 2)
    assert torch.isfinite(C).all()
    assert ((C.float() - ref).abs() <= 2e-3 + 1.5e-3 * ref.abs()).all()


def test_gemm_rejects_unsupported_shapes(lib, cuda_ok):
    A = torch.zeros(8, 100, device="cuda", dtype=torch.float16)
    rc = lib.lb2_test_gemm_f16(A.data_ptr(), A.data_ptr(), A.data_ptr(), A.data_ptr(), A.data_ptr(), 8, 100, 100, 0)
    assert rc != 0 and b"unsupported shape" in lib.lb2_last_error()


@pytest.mark.parametrize("H", [384, 768])
@pytest.mark.parametrize("rows", [1, 7, 8, 1000])
def test_layernorm_vs_torch(lib, cuda_ok, H, rows):
    g = torch.Generator(device="cuda").manual_seed(rows + H)
    x = (torch.randn(rows, H, device="cuda", generator=g) * 3 + 0.5).half()
    gam = torch.randn(H, device="cuda", generator=g)
    bet = torch.randn(H, device="cuda", generator=g)
    out = torch.empty_like(x)
    assert lib.lb2_test_layernorm_f16(x.data_ptr(), gam.data_ptr(), bet.data_ptr(), out.data_ptr(), rows, H, 1e-12) == 0
    ref = torch.nn.functional.layer_norm(x.float(), (H,), gam, bet, 1e-12)
    assert (out.float() - ref).abs().max().item() <= 2e-3 + 1e-3 * ref.abs().max().item()


@pytest.mark.parametrize("H,heads", [(384, 12), (768, 12)])
def test_attention_vs_torch(lib, cuda_ok, H, heads):
    lens = [1, 2, 15, 16, 17, 63, 64, 65, 100, 128, 200, 255, 256]
    T = sum(lens)
    hd = H // heads
    g = torch.Generator(device="cuda").manual_seed(H)
    qkv = (torch.randn(T, 3 * H, device="cuda", generator=g) * 1.5).half()
    ctx = torch.full((T, H), float("nan"), device="cuda", dtype=torch.float16)
    dl = torch.tensor(lens, dtype=torch.int32, device="cuda")
    ds = (torch.cumsum(dl, 0) - dl).to(torch.int32)
    # the kernel reads the head-major layout the QKV GEMM writes: [heads][T][q|k|v]
    qkvh = qkv.view(T, 3, heads, hd).permute(2, 0, 1, 3).contiguous()
    rc = lib.lb2_test_attention_f16(qkvh.data_ptr(), ds.data_ptr(), dl.data_ptr(), len(lens), T, H, heads, 256, ctx.data_ptr())
    assert rc == 0, lib.lb2_last_error()
    assert torch.isfinite(ctx).all()
    off = 0
    worst = 0.0
    for L in lens:
        blk = qkv[off:off + L].float()
        q, k, v = (blk[:, i * H:(i + 1) * H].reshape(L, heads, hd).transpose(0, 1) for i in range(3))
        p = torch.softmax(q @ k.transpose(1, 2) / hd ** 0.5, dim=-1)
        ref = (p @ v).transpose(0, 1).reshape(L, H)
        worst = max(worst, (ctx[off:off + L].float() - ref).abs().max().item())
        off += L
    assert worst <= 4e-3, worst  # P is rounded to fp16 before P.V, output to fp16


@pytest.mark.parametrize("M", [1, 127, 128, 129, 1000, 148 * 128 + 77, 40000])
@pytest.mark.parametrize("K", [384, 1536])
def test_gemm_res_ln_fused_vs_torch(lib, cuda_ok, M, K):
    """Linear + residual + LayerNorm in one kernel (gemm_f16_ln_kernel) against torch fp32 of the same op, with the
    statistics real checkpoints have: LayerNorm gains up to 5, an outlier channel in the residual stream."""
    N = 384
    g = torch.Generator(device="cuda").manual_seed(M + K)
    A = torch.randn(M, K, device="cuda", generator=g).half()
    W = (torch.randn(N, K, device="cuda", generator=g) * 0.05).half()
    bias = torch.randn(N, device="cuda", generator=g) * 0.1
    res = torch.randn(M, N, device="cuda", generator=g)
    res[:, 7] *= 30.0
    res = res.half()
    gam = torch.exp(torch.randn(N, device="cuda", generator=g) * 0.5).clamp(0.3, 5.0)
    bet = torch.randn(N, device="cuda", generator=g) * 0.3
    C = torch.full((M, N), float("nan"), device="cuda", dtype=torch.float16)
    rc = lib.lb2_test_gemm_res_ln_f16(A.data_ptr(), W.data_ptr(), bias.data_ptr(), res.data_ptr(), gam.data_ptr(), bet.data_ptr(),
                                      1e-12, C.data_ptr(), M, N, K)
    assert rc == 0, lib.lb2_last_error()
    y = (A.float() @ W.float().T + bias + res.float()).half().float()  # the pipeline normalises the fp16-rounded tensor
    ref = torch.nn.functional.layer_norm(y, (N,), gam, bet, 1e-12)
    assert torch.isfinite(C).all()
    err = (C.float() - ref).abs()
    tol = 4e-3 + 2e-3 * ref.abs()  # fp16 output rounding + an fp16 ulp of the pre-norm value flipping under accumulation-order noise
    assert (err <= tol).all(), f"max err {err.max().item()} at {torch.nonzero(err > tol)[:3].tolist()}"


@pytest.mark.parametrize("M", [1, 129, 256, 257, 1000, 148 * 128 + 77, 40000])
@pytest.mark.parametrize("K", [384, 1536])
def test_gemm_res_ln_cta_pair_matches_single_cta(lib, cuda_ok, M, K):
    """The cta_group::2 kernel of the fused Linear + residual + LayerNorm (two CTAs share the W panel; taken when M spans
    more than one 128-row block) against the single-CTA kernel (taken for one row block), run on each 128-row slice of the
    same inputs: same accumulation order per row, so the results are identical."""
    N = 384
    g = torch.Generator(device="cuda").manual_seed(M + K)
    A = torch.randn(M, K, device="cuda", generator=g).half()
    W = (torch.randn(N, K, device="cuda", generator=g) * 0.05).half()
    bias = torch.randn(N, device="cuda", generator=g) * 0.1
    res = torch.randn(M, N, device="cuda", generator=g).half()
    gamma = torch.rand(N, device="cuda", generator=g) + 0.5
    beta = torch.randn(N, device="cuda", generator=g) * 0.1
    whole = torch.full((M, N), float("nan"), device="cuda", dtype=torch.float16)
    rc = lib.lb2_test_gemm_res_ln_f16(A.data_ptr(), W.data_ptr(), bias.data_ptr(), res.data_ptr(), gamma.data_ptr(),
                                      beta.data_ptr(), 1e-12, whole.data_ptr(), M, N, K)
    assert rc == 0, lib.lb2_last_error()
    sliced = torch.full((M, N), float("nan"), device="cuda", dtype=torch.float16)
    for r0 in range(0, M, 128):  # row slices of contiguous tensors: 16-byte aligned for TMA
        m = min(128, M - r0)
        rc = lib.lb2_test_gemm_res_ln_f16(A[r0:].data_ptr(), W.data_ptr(), bias.data_ptr(), res[r0:].data_ptr(),
                                          gamma.data_ptr(), beta.data_ptr(), 1e-12, sliced[r0:].data_ptr(), m, N, K)
        assert rc == 0, lib.lb2_last_error()
    torch.cuda.synchronize()
    assert torch.isfinite(whole).all()
    assert torch.equal(whole, sliced)


def test_attention_tc_rotated_tail_blocks(lib, cuda_ok):
    """Second query blocks (rows 128 .. L-1; the warps past the passage idle) of every tail length 1 .. 128, several times,
    plus short and full passages, against torch.  The only attention test with many items per CTA: it checks the multi-item
    pipeline and the drain before a long item (more than 192 keys) overwrites the O accumulators."""
    H, heads, hd = 384, 12, 32
    lens = ([L for L in range(129, 257)] * 3 + [1, 16, 100, 128, 31, 64]
            + [1, 2, 15, 17, 31, 33, 63, 65, 100, 128, 129, 160, 192, 193, 200, 255, 256] * 3)
    T = sum(lens)
    g = torch.Generator(device="cuda").manual_seed(11)
    qkv = (torch.randn(T, 3 * H, device="cuda", generator=g) * 1.5).half()
    dl = torch.tensor(lens, dtype=torch.int32, device="cuda")
    ds = (torch.cumsum(dl, 0) - dl).to(torch.int32)
    qkvh = qkv.view(T, 3, heads, hd).permute(2, 0, 1, 3).contiguous()
    ctx = torch.full((T, H), float("nan"), device="cuda", dtype=torch.float16)
    assert lib.lb2_test_attention_f16(qkvh.data_ptr(), ds.data_ptr(), dl.data_ptr(), len(lens), T, H, heads, 256, ctx.data_ptr()) == 0, lib.lb2_last_error()
    torch.cuda.synchronize()
    assert torch.isfinite(ctx).all()
    off, worst = 0, 0.0
    for L in lens:
        blk = qkv[off:off + L].float()
        q, k, v = (blk[:, i * H:(i + 1) * H].reshape(L, heads, hd).transpose(0, 1) for i in range(3))
        p = torch.softmax(q @ k.transpose(1, 2) / hd ** 0.5, dim=-1)
        ref = (p @ v).transpose(0, 1).reshape(L, H)
        worst = max(worst, (ctx[off:off + L].float() - ref).abs().max().item())
        off += L
    assert worst <= 4e-3, worst
