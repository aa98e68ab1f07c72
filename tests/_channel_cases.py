"""Test infrastructure: the channel counts the training ops accept beyond the generators' defaults, shared by the bf16 per-op tests
(tests/test_gpu_train.py) and their fp32 twins (tests/test_gpu_train_fp32.py)."""

# B, Cin, Cout, H, W, k, stride, transposed: every conv form with an output that takes a partial 32-channel block (Cout 8 / 24 / 40 /
# 48), which the forward accepts (Cout % 8 == 0); the backward zero-pads d(output) to 32-channel multiples for the data gradient
THIN_COUT_CASES = [(2, 64, 48, 20, 28, 3, 1, False), (2, 64, 24, 21, 27, 3, 2, False), (2, 96, 48, 10, 13, 3, 2, True),
                   (2, 64, 8, 12, 15, 3, 2, True), (1, 96, 8, 9, 12, 1, 1, False), (2, 64, 40, 14, 15, 1, 2, False)]

# B, H, W, C, act, residual: channel counts whose C / 8 does not divide the 256-thread block, so the BatchNorm kernels take their plain
# (unhoisted) form; 24 and 48 fill part of one 64-channel reduction block, 96 part of its second
THIN_BN_CASES = [(2, 19, 27, 24, 1, True), (3, 12, 10, 48, 2, False), (1, 30, 44, 96, 0, True), (2, 17, 23, 192, 2, True),
                 (1, 9, 14, 320, 1, False)]
