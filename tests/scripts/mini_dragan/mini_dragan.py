"""A small DRAGAN training script in the API idiom of the reference's scripts (see tests/scripts/mini_convgan), so that
the launcher (b200gan/launch.py) can run the DRAGAN step end to end on a GPU box, where /root/reference does not exist.
Its own generator; the discriminator is the DCGAN one that DRAGAN uses unchanged.  The D step follows dragan.py:144-167,
199-217 literally -- including that d_loss is only printed and gradient_penalty.backward() alone fills the gradients --
with one deviation: the perturbation noise is drawn on the device (the reference mixes a CPU torch.rand into CUDA math,
dragan.py:149, which fails on a GPU)."""
import argparse

import numpy as np
import torch
import torch.autograd as autograd
import torch.nn as nn
import torchvision.transforms as transforms
from torch.autograd import Variable
from torch.utils.data import DataLoader
from torchvision import datasets

ap = argparse.ArgumentParser()
ap.add_argument("--n_epochs", type=int, default=1)
ap.add_argument("--batch_size", type=int, default=64)
ap.add_argument("--lr", type=float, default=0.0002)
ap.add_argument("--b1", type=float, default=0.5)
ap.add_argument("--b2", type=float, default=0.999)
ap.add_argument("--latent_dim", type=int, default=32)
ap.add_argument("--img_size", type=int, default=32)
ap.add_argument("--channels", type=int, default=1)
opt = ap.parse_args()
cuda = torch.cuda.is_available()
Tensor = torch.cuda.FloatTensor if cuda else torch.FloatTensor
lambda_gp = 10


def weights_init_normal(m):
    classname = m.__class__.__name__
    if classname.find("Conv") != -1:
        torch.nn.init.normal_(m.weight.data, 0.0, 0.02)
    elif classname.find("BatchNorm2d") != -1:
        torch.nn.init.normal_(m.weight.data, 1.0, 0.02)
        torch.nn.init.constant_(m.bias.data, 0.0)


class Generator(nn.Module):
    def __init__(self):
        super().__init__()
        self.s0 = opt.img_size // 4
        self.fc = nn.Sequential(nn.Linear(opt.latent_dim, 64 * self.s0 ** 2))
        self.body = nn.Sequential(
            nn.BatchNorm2d(64),
            nn.Upsample(scale_factor=2), nn.Conv2d(64, 64, 3, stride=1, padding=1), nn.BatchNorm2d(64, 0.8),
            nn.LeakyReLU(0.2, inplace=True),
            nn.Upsample(scale_factor=2), nn.Conv2d(64, 32, 3, stride=1, padding=1), nn.BatchNorm2d(32, 0.8),
            nn.LeakyReLU(0.2, inplace=True),
            nn.Conv2d(32, opt.channels, 3, stride=1, padding=1), nn.Tanh(),
        )

    def forward(self, z):
        h = self.fc(z)
        return self.body(h.view(h.shape[0], 64, self.s0, self.s0))


class Discriminator(nn.Module):
    def __init__(self):
        super().__init__()

        def block(cin, cout, bn=True):
            layers = [nn.Conv2d(cin, cout, 3, 2, 1), nn.LeakyReLU(0.2, inplace=True), nn.Dropout2d(0.25)]
            if bn:
                layers.append(nn.BatchNorm2d(cout, 0.8))
            return layers

        self.model = nn.Sequential(*block(opt.channels, 16, bn=False), *block(16, 32), *block(32, 64), *block(64, 128))
        self.adv_layer = nn.Sequential(nn.Linear(128 * (opt.img_size // 16) ** 2, 1), nn.Sigmoid())

    def forward(self, img):
        out = self.model(img)
        return self.adv_layer(out.view(out.shape[0], -1))


def compute_gradient_penalty(D, X):
    alpha = Tensor(np.random.random(size=X.shape))
    noise = torch.rand(X.size(), device=X.device)
    interpolates = alpha * X + ((1 - alpha) * (X + 0.5 * X.std() * noise))
    interpolates = Variable(interpolates, requires_grad=True)
    d_interpolates = D(interpolates)
    ones = Variable(Tensor(X.shape[0], 1).fill_(1.0), requires_grad=False)
    gradients = autograd.grad(outputs=d_interpolates, inputs=interpolates, grad_outputs=ones, create_graph=True,
                              retain_graph=True, only_inputs=True)[0]
    return lambda_gp * ((gradients.norm(2, dim=1) - 1) ** 2).mean()


adversarial_loss = torch.nn.BCELoss()
generator, discriminator = Generator(), Discriminator()
if cuda:
    generator.cuda(); discriminator.cuda(); adversarial_loss.cuda()
generator.apply(weights_init_normal)
discriminator.apply(weights_init_normal)
loader = DataLoader(datasets.MNIST("../../data/mnist", train=True, download=True,
                                   transform=transforms.Compose([transforms.Resize(opt.img_size), transforms.ToTensor(),
                                                                 transforms.Normalize([0.5], [0.5])])),
                    batch_size=opt.batch_size, shuffle=False)
optimizer_G = torch.optim.Adam(generator.parameters(), lr=opt.lr, betas=(opt.b1, opt.b2))
optimizer_D = torch.optim.Adam(discriminator.parameters(), lr=opt.lr, betas=(opt.b1, opt.b2))
history = []
for epoch in range(opt.n_epochs):
    for i, (imgs, _) in enumerate(loader):
        valid = Variable(Tensor(imgs.shape[0], 1).fill_(1.0), requires_grad=False)
        fake = Variable(Tensor(imgs.shape[0], 1).fill_(0.0), requires_grad=False)
        real_imgs = Variable(imgs.type(Tensor))

        optimizer_G.zero_grad()
        z = Variable(Tensor(np.random.normal(0, 1, (imgs.shape[0], opt.latent_dim))))
        gen_imgs = generator(z)
        g_loss = adversarial_loss(discriminator(gen_imgs), valid)
        g_loss.backward()
        optimizer_G.step()

        optimizer_D.zero_grad()
        real_loss = adversarial_loss(discriminator(real_imgs), valid)
        fake_loss = adversarial_loss(discriminator(gen_imgs.detach()), fake)
        d_loss = (real_loss + fake_loss) / 2
        gradient_penalty = compute_gradient_penalty(discriminator, real_imgs.data)
        gradient_penalty.backward()
        optimizer_D.step()

        history.append((d_loss.item(), g_loss.item(), gradient_penalty.item()))
        print("[Epoch %d/%d] [Batch %d/%d] [D loss: %f] [G loss: %f] [GP: %f]"
              % (epoch, opt.n_epochs, i, len(loader), d_loss.item(), g_loss.item(), gradient_penalty.item()))
