"""A small stand-alone MLP GAN training script on the CPU, written in the API idiom of the reference's fully connected
scripts -- torch.nn classes looked up by attribute on `nn` at model-construction time, `nn.Sequential(*layers)`,
`BatchNorm1d(n, 0.8)`, `torch.FloatTensor(numpy_array)`, `Variable`, `.type(Tensor)`, torchvision's MNIST loader -- so that
the launcher (b200gan/launch.py) can be exercised end to end on BASELINE config 0 (MLP on the host) by the test suite
alone.  It is not a copy of any reference script: its own layer widths, latent size and option names."""
import argparse

import numpy as np
import torch
import torch.nn as nn
import torchvision.transforms as transforms
from torch.autograd import Variable
from torch.utils.data import DataLoader
from torchvision import datasets

ap = argparse.ArgumentParser()
ap.add_argument("--epochs", type=int, default=1)
ap.add_argument("--batch_size", type=int, default=32)
ap.add_argument("--zdim", type=int, default=32)
cfg = ap.parse_args()
Tensor = torch.FloatTensor
pixels = 28 * 28


def dense(cin, cout, norm=True):
    layers = [nn.Linear(cin, cout)]
    if norm:
        layers.append(nn.BatchNorm1d(cout, 0.8))
    layers.append(nn.LeakyReLU(0.2, inplace=True))
    return layers


class Gen(nn.Module):
    def __init__(self):
        super().__init__()
        self.model = nn.Sequential(*dense(cfg.zdim, 64, norm=False), *dense(64, 128), *dense(128, 256),
                                   nn.Linear(256, pixels), nn.Tanh())

    def forward(self, z):
        return self.model(z).view(z.shape[0], 1, 28, 28)


class Disc(nn.Module):
    def __init__(self):
        super().__init__()
        self.model = nn.Sequential(nn.Linear(pixels, 192), nn.LeakyReLU(0.2, inplace=True), nn.Linear(192, 1),
                                   nn.Sigmoid())

    def forward(self, img):
        return self.model(img.view(img.shape[0], -1))


bce = torch.nn.BCELoss()
generator, discriminator = Gen(), Disc()
data = DataLoader(datasets.MNIST("../../data/mnist", train=True, download=True,
                                 transform=transforms.Compose([transforms.ToTensor(), transforms.Normalize([0.5], [0.5])])),
                  batch_size=cfg.batch_size, shuffle=True)
opt_g = torch.optim.Adam(generator.parameters(), lr=2e-4, betas=(0.5, 0.999))
opt_d = torch.optim.Adam(discriminator.parameters(), lr=2e-4, betas=(0.5, 0.999))
for epoch in range(cfg.epochs):
    for it, (imgs, _) in enumerate(data):
        ones = Variable(Tensor(imgs.size(0), 1).fill_(1.0), requires_grad=False)
        zeros = Variable(Tensor(imgs.size(0), 1).fill_(0.0), requires_grad=False)
        real = Variable(imgs.type(Tensor))
        opt_g.zero_grad()
        z = Variable(Tensor(np.random.normal(0, 1, (imgs.shape[0], cfg.zdim))))
        fakes = generator(z)
        loss_g = bce(discriminator(fakes), ones)
        loss_g.backward()
        opt_g.step()
        opt_d.zero_grad()
        loss_d = (bce(discriminator(real), ones) + bce(discriminator(fakes.detach()), zeros)) / 2
        loss_d.backward()
        opt_d.step()
        print("[epoch %d] [it %d/%d] [D loss: %f] [G loss: %f]" % (epoch, it, len(data), loss_d.item(), loss_g.item()))
