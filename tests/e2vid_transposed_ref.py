"""CPU fp32 restatement of E2VIDRecurrent with use_upsample_conv=False, for the tests of that option.

Every layer except the decoders is the oracle's (oracle/oracle_torch.py); the decoders are the reference's
TransposedConvLayer (model/e2vid/submodules.py, class TransposedConvLayer; built by BaseUNet.build_decoders with
kernel_size=5, padding=2 when use_upsample_conv=False, model/e2vid/unet.py):
ConvTranspose2d(stride=2, padding=2, output_padding=1) -> ReLU, fed by skip_sum(x, block) as in UNetRecurrent.forward
(unet.py:167-200).  State-dict keys: ``unetrecurrent.decoders.{i}.transposed_conv2d.{weight [Cin, Cout, 5, 5], bias}``.
"""
import torch
import torch.nn.functional as F

from oracle import oracle_torch as O


def transposed_conv(sd, prefix, x, act="relu"):
    w = sd[prefix + ".transposed_conv2d.weight"]
    y = F.conv_transpose2d(x, w, sd.get(prefix + ".transposed_conv2d.bias"), stride=2, padding=w.shape[-1] // 2,
                           output_padding=1)
    return O._act(y, act)


def e2vid_transposed_forward(sd, x, prev_states, num_encoders=4, num_residual_blocks=2, prefix="unetrecurrent"):
    """One step, as O.e2vid_recurrent_forward with TransposedConvLayer decoders: (img, states)."""
    p = prefix + "." if prefix else ""
    x = O.conv_layer(sd, p + "head", x, 1, "relu")
    head = x
    if prev_states is None:
        prev_states = [None] * num_encoders
    blocks, states = [], []
    for i in range(num_encoders):
        x = O.conv_layer(sd, p + "encoders.%d.conv" % i, x, 2, "relu")
        x, st = O.recurrent_step(sd, p + "encoders.%d.recurrent_block" % i, x, prev_states[i])
        blocks.append(x)
        states.append(st)
    for r in range(num_residual_blocks):
        x = O.residual_block(sd, p + "resblocks.%d" % r, x)
    for i in range(num_encoders):
        x = transposed_conv(sd, p + "decoders.%d" % i, x + blocks[num_encoders - 1 - i], "relu")
    img = torch.sigmoid(F.conv2d(x + head, sd[p + "pred.conv2d.weight"], sd[p + "pred.conv2d.bias"]))
    return img, states
