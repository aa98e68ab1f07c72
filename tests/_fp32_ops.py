"""Test infrastructure: the two kernel-backed training ops of train_ops.py (conv2d_nhwc, bn_act) restated on fp32 PyTorch ops --
cuDNN on the CUDA cores when TF32 is off, autograd for the backward: what an fp32 user of the reference computes.  The fp32_tc
training mode is checked against it (tests/test_gpu_train_fp32.py) and timed against it (scripts/train_precision.py)."""
import torch.nn.functional as F

from rdfc_gan_b200 import _cabi as C


def fp32_torch_ops():
    """-> (conv, bn) with the signatures of train_ops.conv2d_nhwc / train_ops.bn_act, over fp32 NHWC tensors."""
    def conv(x, weight, k=3, stride=1, transposed=False):
        xn = x.permute(0, 3, 1, 2)
        y = (F.conv_transpose2d(xn, weight, stride=2, padding=1, output_padding=1) if transposed else
             F.conv2d(xn, weight, stride=stride, padding=(k - 1) // 2))
        return y.permute(0, 2, 3, 1)

    def bn(y, mod, residual=None, act=C.ACT_NONE):
        z = F.batch_norm(y.permute(0, 3, 1, 2), mod.running_mean, mod.running_var, mod.weight, mod.bias, True, mod.momentum, mod.eps)
        if mod.num_batches_tracked is not None:
            mod.num_batches_tracked.add_(1)
        z = z.permute(0, 2, 3, 1)
        if residual is not None:
            z = z + residual
        return {C.ACT_NONE: z, C.ACT_RELU: F.relu(z), C.ACT_LEAKY02: F.leaky_relu(z, 0.2)}[act]
    return conv, bn
