"""`cross_entropy2d` of the reference's training/loss_utils.py:4-18: per-pixel cross entropy between a logit image
[N,C,H,W] and an integer label map [N,Ht,Wt], averaged over the pixels (training/loss.py:611-616 calls it on the 512^2
semantic image and on the 128^2 raw one).

CUDA fp32 logits go through `p3d_cross_entropy2d_fwd/bwd` (include/p3d.h), which read the NCHW logits in place; everything
else (CPU tensors, other dtypes, `size_average=False` is not a mode of the reference either) evaluates the reference's
composition of torch ops.
"""
import torch
import torch.nn.functional as F

from .. import _lib

CE_WORKSPACE_DOUBLES = 2048
IGNORE_INDEX = -100      # F.cross_entropy default


def cross_entropy2d(input, target, weight=None, size_average=True):
    n, c, h, w = input.size()
    nt, ht, wt = target.size()
    if (h != ht) or (w != wt):
        # upsample the logits to the label resolution (loss_utils.py:8-10)
        input = F.interpolate(input, size=(ht, wt), mode='bilinear', align_corners=True)
    if input.device.type == 'cuda' and input.dtype == torch.float32 and target.dtype == torch.int64:
        return _CrossEntropy2d.apply(input, target, weight)
    input = input.transpose(1, 2).transpose(2, 3).contiguous().view(-1, c)
    return F.cross_entropy(input, target.reshape(-1), weight=weight, reduction='mean')


class _CrossEntropy2d(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, target, weight):
        x = logits.contiguous()
        t = target.contiguous()
        wgt = None if weight is None else weight.to(device=x.device, dtype=torch.float32).contiguous()
        n, c, h, w = x.shape
        assert t.shape == (n, h, w) and (wgt is None or wgt.shape == (c,))
        out = torch.empty(2, device=x.device, dtype=torch.float32)          # loss, sum of weights
        ws = torch.empty(CE_WORKSPACE_DOUBLES, device=x.device, dtype=torch.float64)
        _lib.call('p3d_cross_entropy2d_fwd', x, t, wgt, n, c, h * w, IGNORE_INDEX, out[0:1], out[1:2], ws, device=x.device)
        ctx.save_for_backward(x, t, wgt if wgt is not None else x.new_empty(0), out)
        ctx.has_weight = wgt is not None
        return out[0].clone()

    @staticmethod
    def backward(ctx, dloss):
        x, t, wgt, out = ctx.saved_tensors
        if not ctx.needs_input_grad[0]:
            return None, None, None
        n, c, h, w = x.shape
        g = dloss.to(torch.float32).reshape(1).contiguous()
        gx = torch.empty_like(x)
        _lib.call('p3d_cross_entropy2d_bwd', x, t, wgt if ctx.has_weight else None, g, out[1:2], n, c, h * w, IGNORE_INDEX, gx,
                  device=x.device)
        return gx, None, None
