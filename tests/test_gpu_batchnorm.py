"""Fused BatchNorm(+residual)(+ReLU) channels_last kernels vs a plain fp32 PyTorch reference."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _reference(x, res, w, b, relu, eps=1e-5):
    xr = x.detach().float().requires_grad_()
    rr = res.detach().float().requires_grad_() if res is not None else None
    wr, br = w.detach().clone().requires_grad_(), b.detach().clone().requires_grad_()
    rm, rv = torch.zeros_like(w), torch.ones_like(w)
    y = F.batch_norm(xr, rm, rv, wr, br, True, 0.1, eps)
    if rr is not None:
        y = y + rr
    if relu:
        y = torch.relu(y)
    return xr, rr, wr, br, rm, rv, y


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(32, 64, 56, 56), (32, 2048, 7, 7), (4, 24, 5, 5), (8, 256, 14, 14), (1, 8, 1, 3)])
@pytest.mark.parametrize("relu,residual", [(False, False), (True, False), (True, True), (False, True)])
def test_fused_batchnorm_fwd_bwd(dtype, shape, relu, residual):
    from b200ddp import _ext
    from b200ddp.ops import FusedBatchNormAct2d
    C = _ext.get()
    torch.manual_seed(0)
    dev = "cuda"
    x = (torch.randn(*shape, device=dev) * 2 + 0.5).to(dtype).contiguous(memory_format=torch.channels_last).requires_grad_()
    res = torch.randn(*shape, device=dev).to(dtype).contiguous(memory_format=torch.channels_last).requires_grad_() if residual else None
    bn = FusedBatchNormAct2d(shape[1], relu=relu).to(dev)
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5)
        bn.bias.uniform_(-0.5, 0.5)
    before = C.launch_count()
    y = bn(x, residual=res) if residual else bn(x)
    assert C.launch_count() - before in (1, 2), "forward = one fused launch (or stats + apply)"
    assert y.dtype == dtype and y.is_contiguous(memory_format=torch.channels_last)
    dy = torch.randn_like(y)
    y.backward(dy)
    assert C.launch_count() - before in (2, 4)
    xr, rr, wr, br, rm, rv, yr = _reference(x, res, bn.weight, bn.bias, relu)
    yr.backward(dy.float())
    tol = 2e-4 if dtype == torch.float32 else 4e-2
    assert torch.allclose(y.float(), yr, atol=tol, rtol=tol), (y.float() - yr).abs().max()
    gscale = max(1.0, float(xr.grad.abs().max()))
    assert torch.allclose(x.grad.float(), xr.grad, atol=tol * gscale, rtol=tol), (x.grad.float() - xr.grad).abs().max()
    if residual:
        assert torch.allclose(res.grad.float(), rr.grad, atol=tol, rtol=tol)
    n = x.numel() / shape[1]
    ptol = tol * max(1.0, n ** 0.5)
    assert torch.allclose(bn.weight.grad, wr.grad, atol=ptol, rtol=tol * 4), (bn.weight.grad - wr.grad).abs().max()
    assert torch.allclose(bn.bias.grad, br.grad, atol=ptol, rtol=tol * 4)
    assert torch.allclose(bn.running_mean, rm, atol=tol, rtol=tol) and torch.allclose(bn.running_var, rv, atol=tol, rtol=tol)
    assert int(bn.num_batches_tracked) == 1
    # reproducible: no float atomics anywhere
    bn2 = FusedBatchNormAct2d(shape[1], relu=relu).to(dev)
    bn2.load_state_dict(bn.state_dict())
    y1 = bn2(x.detach(), residual=res.detach() if residual else None)
    bn2.load_state_dict(bn.state_dict())
    y2 = bn2(x.detach(), residual=res.detach() if residual else None)
    assert torch.equal(y1, y2)


def test_resnet50_fused_matches_stock_modules():
    """Whole network, fp32 channels_last: fused-BN ResNet-50 vs torchvision's (same weights) - outputs and grads agree."""
    import torchvision
    from b200ddp.models import resnet50
    torch.manual_seed(1)
    ours = resnet50().cuda().to(memory_format=torch.channels_last)
    stock = torchvision.models.resnet50().cuda().to(memory_format=torch.channels_last)
    stock.load_state_dict(ours.state_dict())
    x = torch.randn(8, 3, 96, 96, device="cuda").contiguous(memory_format=torch.channels_last)
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        a, b = ours(x), stock(x)
        a.square().mean().backward()
        b.square().mean().backward()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    assert torch.allclose(a, b, atol=2e-3, rtol=2e-3), (a - b).abs().max()
    for (n, p), q in zip(ours.named_parameters(), stock.parameters()):
        # 53 normalisation layers deep, a different (but fixed) summation order flips a few ReLU masks: compare in norm
        rel = float((p.grad - q.grad).norm() / (q.grad.norm() + 1e-12))
        assert rel < 3e-2, (n, rel)
    for (n, p), q in zip(ours.named_buffers(), stock.buffers()):
        assert torch.allclose(p.float(), q.float(), atol=1e-3, rtol=1e-3), n


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(32, 64, 112, 112), (2, 8, 7, 9), (3, 16, 6, 6), (1, 8, 1, 1)])
def test_maxpool3x3s2_matches_torch(dtype, shape):
    from b200ddp.ops import MaxPool3x3s2
    torch.manual_seed(0)
    x = torch.randn(*shape, device="cuda").to(dtype).contiguous(memory_format=torch.channels_last).requires_grad_()
    y = MaxPool3x3s2()(x)
    dy = torch.randn_like(y)
    y.backward(dy)
    xr = x.detach().clone().requires_grad_()
    yr = F.max_pool2d(xr, 3, stride=2, padding=1)
    yr.backward(dy)
    assert torch.equal(y, yr)
    assert torch.allclose(x.grad.float(), xr.grad.float(), atol=1e-2 if dtype == torch.bfloat16 else 1e-6)
