"""torch-CPU functional restatement of RDF-GAN's ESANet guidance network (TEST INFRASTRUCTURE ONLY).

Restates, over a plain ``state_dict`` (reference key names), what ``ESANetOneModality.forward_net`` computes
(F/lib/models/segmentator/esa_net/esa_net_one_modality.py:145-172, F = the RDF-GAN reference) in the configuration
rdfc_gan_b200.esanet covers: ResNet-18 / 34 BasicBlock encoder, 'SE-add' weighting, pyramid pooling context module, 'add'
encoder-decoder fusion, 'learned-3x3-zeropad' up-sampling, eval-mode BatchNorm.
  conv1 + bn1 + ReLU, SE, max pool 3x3 / 2                       esa_net_one_modality.py:148-150
  layer1..4 (BasicBlocks), SE after each, skip convs 1..3        :152-170
  PPM: adaptive average pools, 1x1 ConvBNAct, nearest up-sampling  model_utils.py:99-134
  decoder modules: ConvBNAct 3x3, NonBottleneck1D, learned up-sampling to the skip's size + skip   decoder.py:64-134
  conv_out, two learned x2 up-samplings                          decoder.py:120-134
The learned up-sampling (decoder.py:137-191) is a nearest resize to the target size followed by a depth-wise 3x3 conv with zero
padding and bias.  Pinned against tests/golden/esanet_*.npz (outputs of the reference's own Python).
"""
import torch
import torch.nn.functional as F


def _bn(sd, p, x, eps=1e-5):
    return F.batch_norm(x, sd[p + ".running_mean"], sd[p + ".running_var"], sd[p + ".weight"], sd[p + ".bias"], False, 0.0, eps)


def _conv_bn_act(sd, p, x):
    """model_utils.py:6-18: conv (no bias, padding k // 2) + BatchNorm + ReLU"""
    w = sd[p + ".conv.weight"]
    return F.relu(_bn(sd, p + ".bn", F.conv2d(x, w, None, 1, w.shape[2] // 2)))


def _se(sd, p, x):
    """model_utils.py:34-49"""
    s = F.adaptive_avg_pool2d(x, 1)
    s = F.relu(F.conv2d(s, sd[p + ".fc.0.weight"], sd[p + ".fc.0.bias"]))
    return x * torch.sigmoid(F.conv2d(s, sd[p + ".fc.2.weight"], sd[p + ".fc.2.bias"]))


def _basic_block(sd, p, x, stride):
    out = F.relu(_bn(sd, p + ".bn1", F.conv2d(x, sd[p + ".conv1.weight"], None, stride, 1)))
    out = _bn(sd, p + ".bn2", F.conv2d(out, sd[p + ".conv2.weight"], None, 1, 1))
    if (p + ".downsample.0.weight") in sd:
        x = _bn(sd, p + ".downsample.1", F.conv2d(x, sd[p + ".downsample.0.weight"], None, stride))
    return F.relu(out + x)


def _res_layer(sd, p, x, stride):
    i = 0
    while (p + f".{i}.conv1.weight") in sd:
        x = _basic_block(sd, p + f".{i}", x, stride if i == 0 else 1)
        i += 1
    return x


def _non_bottleneck_1d(sd, p, x):
    """resnet.py:75-143 (ERFNet block, dilation 1, BatchNorm eps 1e-3)"""
    out = F.relu(F.conv2d(x, sd[p + ".conv3x1_1.weight"], sd[p + ".conv3x1_1.bias"], padding=(1, 0)))
    out = F.conv2d(out, sd[p + ".conv1x3_1.weight"], sd[p + ".conv1x3_1.bias"], padding=(0, 1))
    out = F.relu(_bn(sd, p + ".bn1", out, 1e-3))
    out = F.relu(F.conv2d(out, sd[p + ".conv3x1_2.weight"], sd[p + ".conv3x1_2.bias"], padding=(1, 0)))
    out = F.conv2d(out, sd[p + ".conv1x3_2.weight"], sd[p + ".conv1x3_2.bias"], padding=(0, 1))
    return F.relu(_bn(sd, p + ".bn2", out, 1e-3) + x)


def _upsample(sd, p, x, size):
    """decoder.py:137-191, 'learned-3x3-zeropad': nearest resize to `size`, depth-wise 3x3 conv (zero padding) + bias"""
    x = F.interpolate(x, size=size, mode="nearest")
    return F.conv2d(x, sd[p + ".conv.weight"], sd[p + ".conv.bias"], padding=1, groups=x.shape[1])


def esanet_forward(sd, image):
    """``sd``: an ESANetOneModality state dict; ``image`` (B, Cin, H, W) -> fp32 logits (B, num_classes, 4 h, 4 w), where
    (h, w) is the size after the stem and the max pool."""
    sd = {k: v.detach().float().cpu() for k, v in sd.items() if torch.is_tensor(v)}
    with torch.no_grad():
        x = F.relu(_bn(sd, "encoder.bn1", F.conv2d(image.float().cpu(), sd["encoder.conv1.weight"], None, 2, 3)))
        x = _se(sd, "se_layer0", x)
        x = F.max_pool2d(x, 3, 2, 1)
        skips = []
        for i in (1, 2, 3, 4):
            x = _res_layer(sd, f"encoder.layer{i}", x, 1 if i == 1 else 2)
            x = _se(sd, f"se_layer{i}", x)
            if i < 4:
                skips.append(_conv_bn_act(sd, f"skip_layer{i}.0", x) if f"skip_layer{i}.0.conv.weight" in sd else x)
        # pyramid pooling module
        h, w = x.shape[2:]
        feats = [x]
        nbins = sum(1 for k in sd if k.startswith("context_module.features.") and k.endswith(".1.conv.weight"))
        for j, b in enumerate({2: (1, 5), 4: (1, 2, 4, 8)}[nbins]):          # context_module 'ppm' / 'ppm-1-2-4-8'
            y = _conv_bn_act(sd, f"context_module.features.{j}.1", F.adaptive_avg_pool2d(x, b))
            feats.append(F.interpolate(y, size=(h, w), mode="nearest"))
        x = _conv_bn_act(sd, "context_module.final_conv", torch.cat(feats, 1))
        # decoder
        for m, skip in zip((1, 2, 3), reversed(skips)):
            p = f"decoder.decoder_module_{m}"
            x = _conv_bn_act(sd, p + ".conv3x3", x)
            b = 0
            while f"{p}.decoder_blocks.{b}.conv3x1_1.weight" in sd:
                x = _non_bottleneck_1d(sd, f"{p}.decoder_blocks.{b}", x)
                b += 1
            x = _upsample(sd, p + ".upsample", x, skip.shape[2:]) + skip
        x = F.conv2d(x, sd["decoder.conv_out.weight"], sd["decoder.conv_out.bias"], padding=1)
        x = _upsample(sd, "decoder.upsample1", x, (2 * x.shape[2], 2 * x.shape[3]))
        return _upsample(sd, "decoder.upsample2", x, (2 * x.shape[2], 2 * x.shape[3]))
