"""Box-head FC layers on the 3xTF32 tensor-core kernel (ops.linear_3xtf32): accuracy against an fp64 product, tails, NaN/Inf,
and the dispatch of FastRCNNConvFCHead (native only without autograd and with matmul.allow_tf32 off)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

VGG = [(1024, 25088), (1024, 1024)]
R101 = [(2048, 50176), (2048, 2048)]


@pytest.fixture(autouse=True)
def strict_fp32():
    a = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32 = a


def _init_linear(N, K, seed):
    torch.manual_seed(seed)
    fc = torch.nn.Linear(K, N)
    torch.nn.init.kaiming_uniform_(fc.weight, a=1)   # c2_xavier_fill, as the box head
    torch.nn.init.uniform_(fc.bias, -0.1, 0.1)       # nonzero, so that the bias add is checked
    return fc


def _scaled_err(y, x, w, b, relu):
    ref = x.double() @ w.double().T + b.double()
    scale = x.double().abs() @ w.double().abs().T + b.double().abs()
    if relu:
        ref = ref.clamp_min(0)
    e = (y.double() - ref).abs() / scale.clamp_min(1e-300)
    return e.max().item(), e.mean().item()


def _pooled_features(dev, R, seed):
    from sfod_b200 import ops, synth
    feat = synth.features(synth.V, 8, seed).to(dev)
    rois = synth.random_rois(8, R, seed + 1).to(dev)
    props = [rois[rois[:, 0] == i, 1:].contiguous() for i in range(8)]
    return ops.roi_align(feat, props, (7, 7), 1.0 / 32, 0, True).flatten(1)


def test_fc1_at_the_bench_shape_no_less_accurate_than_fp32_linear(cuda_device):
    from sfod_b200 import ops
    x = _pooled_features(cuda_device, 16000, 7)
    fc = _init_linear(1024, 25088, 3).to(cuda_device)
    w, b = fc.weight.detach(), fc.bias.detach()
    got = _scaled_err(ops.linear_3xtf32(x, w, b, relu=False), x, w, b, False)
    lib = _scaled_err(F.linear(x, w, b), x, w, b, False)
    print(f"fc1 scaled |error| max/mean: 3xTF32 {got[0]:.3e} / {got[1]:.3e}, F.linear fp32 {lib[0]:.3e} / {lib[1]:.3e}")
    assert got[0] <= lib[0] and got[1] <= lib[1]


def test_split_is_applied_tf32_trap(cuda_device):
    """A trap operand of alternating sign, +(1 + u) and -(1 + 2^-10 - u) with 0 < u < 2^-11: TF32 rounds the first down to 1 and
    the second away to -(1 + 2^-10), so every rounding error has the same sign while the products cancel, and a plain TF32
    product errs by ~2e-4 of |x|.|W| (emulated below by rounding the trap operand).  The partner operand is exact in TF32.  The
    trap is put on x and then on W, so both splits are checked; 3xTF32 must stay within 1e-6."""
    from sfod_b200 import ops
    g = torch.Generator().manual_seed(5)
    R, K = 256, 4096
    u = torch.randint(1, 1 << 12, (R, K), generator=g).double() * 2.0 ** -23
    sign = torch.tensor([1.0, -1.0]).repeat(K // 2)
    trap = torch.where(sign > 0, 1 + u, -(1 + 2.0 ** -10 - u)).float()
    exact = (1 + torch.randint(0, 1 << 10, (R, K), generator=g).float() * 2.0 ** -10)     # 11 significant bits
    trap_tf32 = torch.where(sign > 0, torch.ones(()), -torch.ones(()) - 2.0 ** -10).expand(R, K)
    b = torch.zeros(R, device=cuda_device)
    for name, x, w, x_tf32, w_tf32 in (("x", trap, exact, trap_tf32, exact), ("W", exact, trap, exact, trap_tf32)):
        ref = x.double() @ w.double().T
        scale = x.double().abs() @ w.double().abs().T
        plain = ((x_tf32.double() @ w_tf32.double().T - ref).abs() / scale).max().item()
        y = ops.linear_3xtf32(x.to(cuda_device), w.to(cuda_device), b).cpu()
        got = ((y.double() - ref).abs() / scale).max().item()
        print(f"trap on {name}: 3xTF32 {got:.3e}, plain TF32 (emulated) {plain:.3e}")
        assert plain > 1e-4 and got <= 1e-6, name


@pytest.mark.parametrize("N,K", VGG + R101)
def test_shapes_and_tails(cuda_device, N, K):
    from sfod_b200 import ops
    fc = _init_linear(N, K, N + K).to(cuda_device)
    w, b = fc.weight.detach(), fc.bias.detach()
    g = torch.Generator(device=cuda_device).manual_seed(K)
    x_all = torch.randn(16000, K, device=cuda_device, generator=g)
    for M in (1, 127, 128, 129, 2000, 16000):
        x = x_all[:M]
        for relu in (False, True):
            y = ops.linear_3xtf32(x, w, b, relu=relu)
            err = _scaled_err(y, x, w, b, relu)[0]
            assert y.shape == (M, N) and err <= 1e-6, (M, relu, err)
            if relu:
                assert (y >= 0).all()


def test_nan_and_inf_propagate_as_torch(cuda_device):
    from sfod_b200 import ops
    g = torch.Generator(device=cuda_device).manual_seed(2)
    M, N, K = 300, 256, 1024
    x = torch.randn(M, K, device=cuda_device, generator=g)
    w = torch.randn(N, K, device=cuda_device, generator=g) * 0.03
    b = torch.randn(N, device=cuda_device, generator=g)
    w[:, 17] = torch.round(w[:, 17] * 256) / 256        # exactly representable in TF32: a zero low part
    x[3, 5] = float("nan")
    x[10, 17] = float("inf")
    x[11, 17] = -float("inf")
    w[40, 900] = float("inf")
    x[12, 900] = 0.0                                   # 0 * inf: NaN in row 12, column 40
    for relu in (False, True):
        ref = F.linear(x, w, b)
        if relu:
            ref = torch.relu(ref)
        y = ops.linear_3xtf32(x, w, b, relu=relu)
        assert torch.equal(torch.isnan(y), torch.isnan(ref)), relu
        assert torch.equal(torch.isposinf(y), torch.isposinf(ref)) and torch.equal(torch.isneginf(y), torch.isneginf(ref)), relu
        assert torch.isnan(y[3]).all() and torch.isnan(y[12, 40])


def test_box_head_dispatch(cuda_device):
    """Native only when no gradient is needed and matmul.allow_tf32 is off; otherwise the nn.Sequential (cuBLAS) path."""
    from sfod_b200 import ops
    from sfod_b200.modeling.roi_heads import FastRCNNConvFCHead
    from sfod_b200.structures import ShapeSpec
    head = FastRCNNConvFCHead(ShapeSpec(channels=512, height=7, width=7), fc_dims=[1024, 1024]).to(cuda_device)
    x = torch.randn(300, 512, 7, 7, device=cuda_device)

    def calls(fn):
        ops.timers.start()
        out = fn()
        return out, ops.timers.stop().get("box_head_fc", (0, 0.0))[0]

    with torch.no_grad():
        y, n = calls(lambda: head(x))
        ref = torch.relu(F.linear(torch.relu(F.linear(x.flatten(1), head.fc1.weight, head.fc1.bias)), head.fc2.weight, head.fc2.bias))
    assert n == 2 and (y - ref).abs().max().item() <= 1e-5 * ref.abs().max().item()
    y, n = calls(lambda: head(x))                          # grad enabled, parameters require grad: autograd path
    assert n == 0 and y.requires_grad
    torch.backends.cuda.matmul.allow_tf32 = True
    with torch.no_grad():
        _, n = calls(lambda: head(x))
    assert n == 0
