"""The model families of the hot path, built from an `nn` namespace (b200gan.nn by default).

These restate the architectures of the reference scripts so that bench.py / smoke() can run on a
box where /root/reference does not exist; with the launcher (launch.py) the reference's own
classes are used unmodified instead.  Citations: implementations/<name>/...
"""
import types

import torch.nn as tnn

from . import nn as bnn


def namespace(stock=False):
    """An object exposing Conv2d, BatchNorm2d, ... : b200gan drop-ins, or stock torch.nn."""
    ns = types.SimpleNamespace()
    for name in dir(tnn):
        setattr(ns, name, getattr(tnn, name))
    if not stock:
        for name, cls in bnn.REPLACEMENTS.items():
            setattr(ns, name, cls)
    return ns


def weights_init_normal(m):
    """dcgan.py:36-42 / pix2pix/models.py:6-12: dispatch on the class *name*."""
    import torch
    classname = m.__class__.__name__
    if classname.find("Conv") != -1:
        torch.nn.init.normal_(m.weight.data, 0.0, 0.02)
    elif classname.find("BatchNorm2d") != -1:
        torch.nn.init.normal_(m.weight.data, 1.0, 0.02)
        torch.nn.init.constant_(m.bias.data, 0.0)


class DCGANGenerator(tnn.Module):
    """dcgan/dcgan.py:45-70."""

    def __init__(self, img_size=64, latent_dim=100, channels=1, nn=None):
        super().__init__()
        nn = nn or namespace()
        self.init_size = img_size // 4
        self.l1 = nn.Sequential(nn.Linear(latent_dim, 128 * self.init_size ** 2))
        self.conv_blocks = nn.Sequential(
            nn.BatchNorm2d(128),
            nn.Upsample(scale_factor=2),
            nn.Conv2d(128, 128, 3, stride=1, padding=1),
            nn.BatchNorm2d(128, 0.8),
            nn.LeakyReLU(0.2, inplace=True),
            nn.Upsample(scale_factor=2),
            nn.Conv2d(128, 64, 3, stride=1, padding=1),
            nn.BatchNorm2d(64, 0.8),
            nn.LeakyReLU(0.2, inplace=True),
            nn.Conv2d(64, channels, 3, stride=1, padding=1),
            nn.Tanh(),
        )

    def forward(self, z):
        out = self.l1(z)
        out = out.view(out.shape[0], 128, self.init_size, self.init_size)
        return self.conv_blocks(out)


class DCGANDiscriminator(tnn.Module):
    """dcgan/dcgan.py:73-99."""

    # forward = conv blocks -> view -> Linear + Sigmoid, nothing batch-dependent outside `model`: train.dcgan_step may run
    # the real and the fake pass of the D step as one grouped pass (ops.bn_groups)
    _b200_batchable_passes = True

    def __init__(self, img_size=64, channels=1, nn=None):
        super().__init__()
        nn = nn or namespace()

        def block(cin, cout, bn=True):
            layers = [nn.Conv2d(cin, cout, 3, 2, 1), nn.LeakyReLU(0.2, inplace=True), nn.Dropout2d(0.25)]
            if bn:
                layers.append(nn.BatchNorm2d(cout, 0.8))
            return layers

        self.model = nn.Sequential(*block(channels, 16, bn=False), *block(16, 32), *block(32, 64), *block(64, 128))
        ds_size = img_size // 2 ** 4
        self.adv_layer = nn.Sequential(nn.Linear(128 * ds_size ** 2, 1), nn.Sigmoid())

    def forward(self, img):
        out = self.model(img)
        out = out.view(out.shape[0], -1)
        return self.adv_layer(out)


class WGANGPGenerator(tnn.Module):
    """wgan_gp/wgan_gp.py:42-65 (MLP; BatchNorm1d(out, 0.8): second positional argument is eps)."""

    def __init__(self, img_shape=(1, 32, 32), latent_dim=100, nn=None):
        super().__init__()
        nn = nn or namespace()
        self.img_shape = tuple(img_shape)

        def block(i, o, normalize=True):
            layers = [nn.Linear(i, o)]
            if normalize:
                layers.append(nn.BatchNorm1d(o, 0.8))
            layers.append(nn.LeakyReLU(0.2, inplace=True))
            return layers

        n_out = 1
        for v in self.img_shape:
            n_out *= v
        self.model = nn.Sequential(*block(latent_dim, 128, normalize=False), *block(128, 256), *block(256, 512),
                                   *block(512, 1024), nn.Linear(1024, n_out), nn.Tanh())

    def forward(self, z):
        img = self.model(z)
        return img.view(img.shape[0], *self.img_shape)


class WGANGPDiscriminator(tnn.Module):
    """wgan_gp/wgan_gp.py:68-83."""

    def __init__(self, img_shape=(1, 32, 32), nn=None):
        super().__init__()
        nn = nn or namespace()
        n_in = 1
        for v in img_shape:
            n_in *= v
        self.model = nn.Sequential(nn.Linear(n_in, 512), nn.LeakyReLU(0.2, inplace=True), nn.Linear(512, 256),
                                   nn.LeakyReLU(0.2, inplace=True), nn.Linear(256, 1))

    def forward(self, img):
        return self.model(img.view(img.shape[0], -1))


class DualGANDiscriminator(tnn.Module):
    """dualgan/models.py:102-123: a WGAN-GP critic with BatchNorm2d(out, 0.8) + LeakyReLU(0.2) blocks and a patch head
    (ZeroPad2d((1, 0, 1, 0)) -> Conv2d(256, 1, 4)); its gradient penalty (dualgan.py:116-135) differentiates through the
    BatchNorm backward."""

    def __init__(self, in_channels=3, nn=None):
        super().__init__()
        nn = nn or namespace()

        def block(i, o, normalize=True):
            layers = [nn.Conv2d(i, o, 4, stride=2, padding=1)]
            if normalize:
                layers.append(nn.BatchNorm2d(o, 0.8))
            layers.append(nn.LeakyReLU(0.2, inplace=True))
            return layers

        self.model = nn.Sequential(*block(in_channels, 64, normalize=False), *block(64, 128), *block(128, 256),
                                   nn.ZeroPad2d((1, 0, 1, 0)), nn.Conv2d(256, 1, kernel_size=4))

    def forward(self, img):
        return self.model(img)


# ------------------------------------------------------------------------------------------------
# Pix2Pix (BASELINE config 3): pix2pix/models.py:20-133
# ------------------------------------------------------------------------------------------------
def weights_init_normal_cyclegan(m):
    """cyclegan/models.py:6-14: as above, plus conv biases set to 0."""
    import torch
    classname = m.__class__.__name__
    if classname.find("Conv") != -1:
        torch.nn.init.normal_(m.weight.data, 0.0, 0.02)
        if hasattr(m, "bias") and m.bias is not None:
            torch.nn.init.constant_(m.bias.data, 0.0)
    elif classname.find("BatchNorm2d") != -1:
        torch.nn.init.normal_(m.weight.data, 1.0, 0.02)
        torch.nn.init.constant_(m.bias.data, 0.0)


class UNetDown(tnn.Module):
    """pix2pix/models.py:20-32."""

    def __init__(self, in_size, out_size, normalize=True, dropout=0.0, nn=None):
        super().__init__()
        nn = nn or namespace()
        layers = [nn.Conv2d(in_size, out_size, 4, 2, 1, bias=False)]
        if normalize:
            layers.append(nn.InstanceNorm2d(out_size))
        layers.append(nn.LeakyReLU(0.2))
        if dropout:
            layers.append(nn.Dropout(dropout))
        self.model = nn.Sequential(*layers)

    def forward(self, x):
        return self.model(x)


class UNetUp(tnn.Module):
    """pix2pix/models.py:35-52."""

    def __init__(self, in_size, out_size, dropout=0.0, nn=None):
        super().__init__()
        nn = nn or namespace()
        layers = [nn.ConvTranspose2d(in_size, out_size, 4, 2, 1, bias=False), nn.InstanceNorm2d(out_size),
                  nn.ReLU(inplace=True)]
        if dropout:
            layers.append(nn.Dropout(dropout))
        self.model = nn.Sequential(*layers)

    def forward(self, x, skip_input):
        import torch
        return torch.cat((self.model(x), skip_input), 1)


class GeneratorUNet(tnn.Module):
    """pix2pix/models.py:55-101."""

    def __init__(self, in_channels=3, out_channels=3, nn=None):
        super().__init__()
        nn = nn or namespace()
        self.down1 = UNetDown(in_channels, 64, normalize=False, nn=nn)
        self.down2 = UNetDown(64, 128, nn=nn)
        self.down3 = UNetDown(128, 256, nn=nn)
        self.down4 = UNetDown(256, 512, dropout=0.5, nn=nn)
        self.down5 = UNetDown(512, 512, dropout=0.5, nn=nn)
        self.down6 = UNetDown(512, 512, dropout=0.5, nn=nn)
        self.down7 = UNetDown(512, 512, dropout=0.5, nn=nn)
        self.down8 = UNetDown(512, 512, normalize=False, dropout=0.5, nn=nn)
        self.up1 = UNetUp(512, 512, dropout=0.5, nn=nn)
        self.up2 = UNetUp(1024, 512, dropout=0.5, nn=nn)
        self.up3 = UNetUp(1024, 512, dropout=0.5, nn=nn)
        self.up4 = UNetUp(1024, 512, dropout=0.5, nn=nn)
        self.up5 = UNetUp(1024, 256, nn=nn)
        self.up6 = UNetUp(512, 128, nn=nn)
        self.up7 = UNetUp(256, 64, nn=nn)
        self.final = nn.Sequential(nn.Upsample(scale_factor=2), nn.ZeroPad2d((1, 0, 1, 0)),
                                   nn.Conv2d(128, out_channels, 4, padding=1), nn.Tanh())

    def forward(self, x):
        d1 = self.down1(x)
        d2 = self.down2(d1)
        d3 = self.down3(d2)
        d4 = self.down4(d3)
        d5 = self.down5(d4)
        d6 = self.down6(d5)
        d7 = self.down7(d6)
        d8 = self.down8(d7)
        u1 = self.up1(d8, d7)
        u2 = self.up2(u1, d6)
        u3 = self.up3(u2, d5)
        u4 = self.up4(u3, d4)
        u5 = self.up5(u4, d3)
        u6 = self.up6(u5, d2)
        u7 = self.up7(u6, d1)
        return self.final(u7)


class Pix2PixDiscriminator(tnn.Module):
    """pix2pix/models.py:109-133 (PatchGAN on cat(A, B))."""

    def __init__(self, in_channels=3, nn=None):
        super().__init__()
        nn = nn or namespace()

        def block(i, o, normalization=True):
            layers = [nn.Conv2d(i, o, 4, stride=2, padding=1)]
            if normalization:
                layers.append(nn.InstanceNorm2d(o))
            layers.append(nn.LeakyReLU(0.2, inplace=True))
            return layers

        self.model = nn.Sequential(*block(in_channels * 2, 64, normalization=False), *block(64, 128), *block(128, 256),
                                   *block(256, 512), nn.ZeroPad2d((1, 0, 1, 0)),
                                   nn.Conv2d(512, 1, 4, padding=1, bias=False))

    def forward(self, img_A, img_B):
        import torch
        return self.model(torch.cat((img_A, img_B), 1))


# ------------------------------------------------------------------------------------------------
# CycleGAN (BASELINE config 4): cyclegan/models.py:22-122
# ------------------------------------------------------------------------------------------------
class ResidualBlock(tnn.Module):
    """cyclegan/models.py:22-37."""

    def __init__(self, in_features, nn=None):
        super().__init__()
        nn = nn or namespace()
        self.block = nn.Sequential(nn.ReflectionPad2d(1), nn.Conv2d(in_features, in_features, 3),
                                   nn.InstanceNorm2d(in_features), nn.ReLU(inplace=True), nn.ReflectionPad2d(1),
                                   nn.Conv2d(in_features, in_features, 3), nn.InstanceNorm2d(in_features))

    def forward(self, x):
        return x + self.block(x)


class GeneratorResNet(tnn.Module):
    """cyclegan/models.py:40-87 (note: the first/last ReflectionPad2d take `channels` as pad, :49,:81)."""

    def __init__(self, input_shape, num_residual_blocks, nn=None):
        super().__init__()
        nn = nn or namespace()
        channels = input_shape[0]
        out_features = 64
        model = [nn.ReflectionPad2d(channels), nn.Conv2d(channels, out_features, 7), nn.InstanceNorm2d(out_features),
                 nn.ReLU(inplace=True)]
        in_features = out_features
        for _ in range(2):
            out_features *= 2
            model += [nn.Conv2d(in_features, out_features, 3, stride=2, padding=1), nn.InstanceNorm2d(out_features),
                      nn.ReLU(inplace=True)]
            in_features = out_features
        for _ in range(num_residual_blocks):
            model += [ResidualBlock(out_features, nn=nn)]
        for _ in range(2):
            out_features //= 2
            model += [nn.Upsample(scale_factor=2), nn.Conv2d(in_features, out_features, 3, stride=1, padding=1),
                      nn.InstanceNorm2d(out_features), nn.ReLU(inplace=True)]
            in_features = out_features
        model += [nn.ReflectionPad2d(channels), nn.Conv2d(out_features, channels, 7), nn.Tanh()]
        self.model = nn.Sequential(*model)

    def forward(self, x):
        return self.model(x)


class CycleGANDiscriminator(tnn.Module):
    """cyclegan/models.py:95-122."""

    def __init__(self, input_shape, nn=None):
        super().__init__()
        nn = nn or namespace()
        channels, height, width = input_shape
        self.output_shape = (1, height // 2 ** 4, width // 2 ** 4)

        def block(i, o, normalize=True):
            layers = [nn.Conv2d(i, o, 4, stride=2, padding=1)]
            if normalize:
                layers.append(nn.InstanceNorm2d(o))
            layers.append(nn.LeakyReLU(0.2, inplace=True))
            return layers

        self.model = nn.Sequential(*block(channels, 64, normalize=False), *block(64, 128), *block(128, 256),
                                   *block(256, 512), nn.ZeroPad2d((1, 0, 1, 0)), nn.Conv2d(512, 1, 4, padding=1))

    def forward(self, img):
        return self.model(img)
