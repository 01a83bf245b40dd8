"""ORACLE — test infrastructure only.

Plain torch-fp32 (CPU) restatement of the reference's descriptor gather and refinement
net, driven by the reference's own ``state_dict`` (identical keys), so that tests need
neither the reference nor a GPU.  Pinned to outputs of the reference modules stored in
tests/golden/ (tests/test_oracle_pin_reference.py, tests/test_oracle_golden.py).

Follows:
  READ/models/texture.py:42-70    PointTexture.forward   -> point_texture()
  READ/models/compose.py:125-181  NetAndTexture.forward  -> net_and_texture()
  READ/models/unet.py:22-53       BasicConv (gated conv) -> basic_conv()
  READ/models/unet.py:11-20,56-117 ResBlock/EBlock/DBlock/AFF/SCM/FAM
  READ/models/unet.py:202-285     UNet.forward           -> unet_forward()
"""
import torch
import torch.nn.functional as F


def point_texture(texture_, ids, activation="none"):
    """texture_ [1,C,N] f32; ids [B,1|3,h,w] float -> [B,C,h,w].  texture.py:52-70."""
    idx = ids[:, 0].long()                                   # :52  BxHxW
    B, h, w = idx.shape
    C = texture_.shape[1]
    sample = torch.index_select(texture_[0], 1, idx.reshape(-1))   # :61 (C x B*h*w); expand over B is a no-op
    sample = sample.view(C, B, h, w).permute(1, 0, 2, 3)     # :62-63
    if activation == "sigmoid":
        return torch.sigmoid(sample)
    if activation == "tanh":
        return torch.tanh(sample)
    return sample


def basic_conv(sd, prefix, x, k, stride=1, relu=True):
    """unet.py:22-53.  padding = int((k-1)/2) zeros (padding_mode arg is stored, not applied :36-38)."""
    p = int((k - 1) / 2)
    f = F.conv2d(x, sd[prefix + ".block.conv_f.weight"], sd[prefix + ".block.conv_f.bias"],
                 stride=stride, padding=p)
    if relu:
        f = F.elu(f)                                          # act_fun=nn.ELU (alpha=1)
    m = torch.sigmoid(F.conv2d(x, sd[prefix + ".block.conv_m.weight"], sd[prefix + ".block.conv_m.bias"],
                               stride=stride, padding=p))
    y = f * m
    n = prefix + ".block.norm."
    return F.batch_norm(y, sd[n + "running_mean"], sd[n + "running_var"], sd[n + "weight"], sd[n + "bias"],
                        training=False, eps=1e-5)             # eval-mode BN (eval_in_train, train.py:271-273)


def res_block(sd, prefix, x):
    y = basic_conv(sd, prefix + ".main.0", x, 3, 1, True)     # unet.py:14-17
    y = basic_conv(sd, prefix + ".main.1", y, 3, 1, False)
    return y + x                                              # :20


def block4(sd, prefix, x, num_res=4):
    for i in range(num_res):                                  # EBlock/DBlock unet.py:56-76
        x = res_block(sd, f"{prefix}.layers.{i}", x)
    return x


def scm(sd, prefix, x):
    y = basic_conv(sd, prefix + ".main.0", x, 3, 1, True)     # unet.py:95-100
    y = basic_conv(sd, prefix + ".main.1", y, 1, 1, True)
    y = basic_conv(sd, prefix + ".main.2", y, 3, 1, True)
    y = basic_conv(sd, prefix + ".main.3", y, 1, 1, True)
    y = torch.cat([x, y], dim=1)                              # :105
    return basic_conv(sd, prefix + ".conv", y, 1, 1, False)   # :102,106


def fam(sd, prefix, x1, x2):
    return x1 + basic_conv(sd, prefix + ".merge", x1 * x2, 3, 1, False)   # unet.py:114-117


def aff(sd, prefix, x1, x2, x3, x4):
    x = torch.cat([x1, x2, x3, x4], dim=1)                    # unet.py:88
    x = basic_conv(sd, prefix + ".conv.0", x, 1, 1, True)
    return basic_conv(sd, prefix + ".conv.1", x, 3, 1, False)


def up4(x):
    return F.interpolate(x, scale_factor=4, mode="bilinear", align_corners=False)   # unet.py:200


def unet_forward(sd, inputs):
    """unet.py:202-285.  inputs: list of >=4 tensors [B,8,h_l,w_l]; returns [B,3,H,W]."""
    x, x_2, x_4, x_8 = inputs[0], inputs[1], inputs[2], inputs[3]
    z2 = scm(sd, "SCM2", x_2)
    z4 = scm(sd, "SCM1", x_4)
    z8 = scm(sd, "SCM0", x_8)

    x_ = basic_conv(sd, "feat_extract.0", x, 3, 1, True)
    res1 = block4(sd, "Encoder.0", x_)

    z = basic_conv(sd, "feat_extract.1", res1, 3, 2, True)
    z = fam(sd, "FAM2", z, z2)
    res2 = block4(sd, "Encoder.1", z)

    z = basic_conv(sd, "feat_extract.2", res2, 3, 2, True)
    z = fam(sd, "FAM1", z, z4)
    res3 = block4(sd, "Encoder.2", z)

    z = basic_conv(sd, "feat_extract.6", res3, 3, 2, True)
    z = fam(sd, "FAM0", z, z8)
    z = block4(sd, "Encoder.3", z)

    z12 = F.interpolate(res1, scale_factor=0.5)
    z13 = F.interpolate(res1, scale_factor=0.25)
    z21 = F.interpolate(res2, scale_factor=2)
    z23 = F.interpolate(res2, scale_factor=0.5)
    z32 = F.interpolate(res3, scale_factor=2)
    z31 = F.interpolate(res3, scale_factor=4)
    z43 = F.interpolate(z, scale_factor=2)
    z42 = F.interpolate(z43, scale_factor=2)
    z41 = F.interpolate(z42, scale_factor=2)

    res1 = aff(sd, "AFFs.0", res1, z21, z31, z41)
    res2 = aff(sd, "AFFs.1", z12, res2, z32, z42)
    res3 = aff(sd, "AFFs.2", z13, z23, res3, z43)

    z = block4(sd, "Decoder.0", z)
    z = basic_conv(sd, "feat_extract.7", z, 4, 2, True)
    z = up4(z)
    z = torch.cat([z, res3], dim=1)
    z = basic_conv(sd, "Convs.0", z, 1, 1, True)
    z = block4(sd, "Decoder.1", z)

    z = basic_conv(sd, "feat_extract.3", z, 4, 2, True)
    z = up4(z)
    z = torch.cat([z, res2], dim=1)
    z = basic_conv(sd, "Convs.1", z, 1, 1, True)
    z = block4(sd, "Decoder.2", z)

    z = basic_conv(sd, "feat_extract.4", z, 4, 2, True)
    z = up4(z)
    z = torch.cat([z, res1], dim=1)
    z = basic_conv(sd, "Convs.2", z, 1, 1, True)
    z = block4(sd, "Decoder.3", z)
    return basic_conv(sd, "feat_extract.5", z, 3, 1, False)


def net_and_texture(sd, texture_, index_maps, activation="none"):
    """compose.py:125-181 for the TexturePipeline case (every input key is 'uv*', ss=1, no
    temporal average): per batch item, gather every level then run the net with batch 1."""
    B = index_maps[0].shape[0]
    outs = []
    for i in range(B):
        feats = [point_texture(texture_, m[i][None], activation) for m in index_maps]
        outs.append(unet_forward(sd, feats))
    return torch.cat(outs, 0)


# ---- deterministic synthetic weights (SURVEY.md §8d): identical keys/shapes to UNet.state_dict() ----

def _bc_shapes(cin, cout, k):
    return {
        "block.conv_f.weight": (cout, cin, k, k), "block.conv_f.bias": (cout,),
        "block.conv_m.weight": (cout, cin, k, k), "block.conv_m.bias": (cout,),
        "block.norm.weight": (cout,), "block.norm.bias": (cout,),
        "block.norm.running_mean": (cout,), "block.norm.running_var": (cout,),
        "block.norm.num_batches_tracked": (),
    }


def unet_layer_table(base=32, num_res=4):
    """(prefix, cin, cout, k) for every BasicConv of UNet.__init__ (unet.py:130-200), incl. unused ConvsOut."""
    c = base
    t = []
    for e, ch in enumerate([c, 2 * c, 4 * c, 8 * c]):
        for r in range(num_res):
            t += [(f"Encoder.{e}.layers.{r}.main.0", ch, ch, 3), (f"Encoder.{e}.layers.{r}.main.1", ch, ch, 3)]
    t += [("feat_extract.0", 8, c, 3), ("feat_extract.1", c, 2 * c, 3), ("feat_extract.2", 2 * c, 4 * c, 3),
          ("feat_extract.3", 4 * c, 2 * c, 4), ("feat_extract.4", 2 * c, c, 4), ("feat_extract.5", c, 3, 3),
          ("feat_extract.6", 4 * c, 8 * c, 3), ("feat_extract.7", 8 * c, 4 * c, 4)]
    for d, ch in enumerate([8 * c, 4 * c, 2 * c, c]):
        for r in range(num_res):
            t += [(f"Decoder.{d}.layers.{r}.main.0", ch, ch, 3), (f"Decoder.{d}.layers.{r}.main.1", ch, ch, 3)]
    t += [("Convs.0", 8 * c, 4 * c, 1), ("Convs.1", 4 * c, 2 * c, 1), ("Convs.2", 2 * c, c, 1)]
    t += [("ConvsOut.0", 4 * c, 3, 3), ("ConvsOut.1", 2 * c, 3, 3)]
    for a, ch in enumerate([c, 2 * c, 4 * c]):
        t += [(f"AFFs.{a}.conv.0", 15 * c, ch, 1), (f"AFFs.{a}.conv.1", ch, ch, 3)]
    for name, ch in [("FAM1", 4 * c), ("SCM1", 4 * c), ("FAM2", 2 * c), ("SCM2", 2 * c), ("FAM0", 8 * c), ("SCM0", 8 * c)]:
        if name.startswith("FAM"):
            t += [(f"{name}.merge", ch, ch, 3)]
        else:
            t += [(f"{name}.main.0", 8, ch // 4, 3), (f"{name}.main.1", ch // 4, ch // 2, 1),
                  (f"{name}.main.2", ch // 2, ch // 2, 3), (f"{name}.main.3", ch // 2, ch - 8, 1),
                  (f"{name}.conv", ch, ch, 1)]
    return t
