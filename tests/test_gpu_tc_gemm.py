"""fp16-split tcgen05 GEMM building blocks of the MLP towers vs an fp64 matmul (GPU)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _amax(t):
    return t.abs().max().reshape(1).to(torch.float32)


@pytest.mark.parametrize("M,K,mode", [(128, 32, 0), (128, 256, 0), (1000, 128, 0), (5000, 256, 0), (262144, 256, 0),
                                      (128, 256, 1), (5000, 256, 1), (70000, 256, 1)])
@pytest.mark.parametrize("grad_like", [False, True])
def test_tc_gemm_h_matches_fp64(M, K, mode, grad_like):
    """C = A . B^T (mode 0, forward layout) / A . B (mode 1, dgrad layout) through three kind::f16 MMAs per product
    (fp16 hi/lo split): error vs fp64 at the fp32-GEMM level. grad_like: operand ~1e-7 with its max published (scaled
    into fp16 range by the kernel); without scaling such an operand would flush to zero."""
    from rlinf_b200 import _lib as L

    lib = L.load()
    g = torch.Generator(device="cuda").manual_seed(M + K + mode)
    A = torch.randn(M, K, device="cuda", generator=g)
    if grad_like:
        A = A * 3e-7 * torch.exp(2 * torch.randn(M, 1, device="cuda", generator=g))
    B = torch.randn(256, K, device="cuda", generator=g) / K ** 0.5
    C = torch.empty(M, 256, device="cuda")
    work = torch.empty(512 * K, device="cuda")  # forward pack + dgrad pack of the weights
    amax = _amax(A) if grad_like else None
    L.check(lib.rb200_tc_gemm_h(L.ptr(A), L.ptr(B), L.ptr(C), M, K, mode, L.ptr(amax), L.ptr(work), L.stream_ptr()), "tc_gemm_h")
    Bd = B.double().t() if mode == 0 else B.double()
    ref = A.double() @ Bd
    scale = (A.double().abs() @ Bd.abs()).clamp_min(1e-300)
    if grad_like:
        # ONE power-of-two scale per operand (from its published max) puts max|a| at 2^13; an element keeps all 22 bits
        # of the (hi, lo) pair down to |a| = amax * 2^-16 and loses them gradually below (lo falls into fp16's
        # subnormals, quantum amax * 2^-38 = the 2^-22 relative error of an element of size amax * 2^-16).  The rows
        # of this operand spread over e^(+-7.4) ~ 2^21 (measured on B200: 2.5e-5 relative on the smallest rows, 4e-7
        # on typical ones); such rows are ~1e-6 of any sum over samples, so the bound carries the absolute floor.
        floor = (amax.double() * 2.0 ** -16) * Bd.abs().sum(dim=0, keepdim=True)
        scale = scale + floor
    err = ((C.double() - ref).abs() / scale).max().item()
    print(f"tc_gemm_h M={M} K={K} mode={mode} grad_like={grad_like}: max |err| / (|A|.|B|) = {err:.2e}")
    assert err < 2e-6, err  # fp32 SGEMM is ~1e-7..1e-6 on this measure; plain fp16/bf16 would be ~1e-3


@pytest.mark.parametrize("n,IN", [(32, 32), (1000, 128), (4096, 256), (70000, 256), (262144, 128)])
@pytest.mark.parametrize("grad_like", [False, True])
def test_tc_wgrad_h_matches_fp64(n, IN, grad_like):
    from rlinf_b200 import _lib as L

    lib = L.load()
    g = torch.Generator(device="cuda").manual_seed(n + IN)
    Z = torch.randn(n, 256, device="cuda", generator=g)
    if grad_like:
        Z = Z * 1e-8 * torch.exp(2 * torch.randn(n, 1, device="cuda", generator=g))
    H = torch.tanh(torch.randn(n, IN, device="cuda", generator=g))
    dW = torch.zeros(256, IN, device="cuda")
    amax = _amax(Z) if grad_like else None
    L.check(lib.rb200_tc_wgrad_h(L.ptr(Z), L.ptr(H), L.ptr(dW), n, IN, L.ptr(amax), L.stream_ptr()), "tc_wgrad_h")
    ref = Z.double().t() @ H.double()
    scale = (Z.double().abs().t() @ H.double().abs()).clamp_min(1e-300)
    err = ((dW.double() - ref).abs() / scale).max().item()
    print(f"tc_wgrad_h n={n} IN={IN} grad_like={grad_like}: max |err| / (|Z|^T.|H|) = {err:.2e}")
    assert err < 2e-6, err


def test_fp16_split_kernel_timing_report():
    """Not an assertion on speed: prints per-launch times of the fp16-split kernels at the headline mini-batch shape so
    that every GPU test log carries them."""
    from rlinf_b200 import _lib as L

    lib = L.load()
    n, K = 262144, 256
    A = torch.randn(n, K, device="cuda")
    B = torch.randn(256, K, device="cuda") / 16
    C = torch.empty(n, 256, device="cuda")
    work = torch.empty(512 * K, device="cuda")
    dW = torch.zeros(256, K, device="cuda")

    def timeit(fn, reps=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps * 1e3

    t = {
        "f16x2 gemm fwd": timeit(lambda: lib.rb200_tc_gemm_h(L.ptr(A), L.ptr(B), L.ptr(C), n, K, 0, None, L.ptr(work), L.stream_ptr())),
        "f16x2 gemm dgrad": timeit(lambda: lib.rb200_tc_gemm_h(L.ptr(A), L.ptr(B), L.ptr(C), n, K, 1, None, L.ptr(work), L.stream_ptr())),
        "f16x2 wgrad": timeit(lambda: lib.rb200_tc_wgrad_h(L.ptr(C), L.ptr(A), L.ptr(dW), n, K, None, L.stream_ptr())),
    }
    print("TIMING us/launch (incl. the weight-split helper kernel of the test entries):", {k: round(v, 1) for k, v in t.items()})
