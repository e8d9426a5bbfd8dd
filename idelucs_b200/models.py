"""Trainer with the reference's interface (idelucs/models.py:46-195).  The arithmetic that is on
the hot path — pair featurisation and the IIC loss — runs in the sm_100a kernels; the MLP,
InfoNCE, optimiser stay PyTorch (scope contract).  Differences that are deliberate:
batches never leave the GPU (no DataLoader workers / H2D copies), and ``predict`` featurises
from the packed device-resident sequences instead of re-parsing the FASTA file."""
import random
import sys

import numpy as np
import torch
import torch.optim as optim

from .LossFunctions import IID_loss, info_nce_loss
from .PytorchUtils import NetLinear, myNet
from .utils import SequenceDataset, create_dataloader

# idelucs/models.py:18-21 seeds the global generators at import; kept for drop-in behaviour
torch.manual_seed(0)
np.random.seed(0)
random.seed(0)

device = "cuda"


def weights_init(m):
    """Kaiming-normal weights, zero bias (idelucs/models.py:36-44)."""
    if isinstance(m, torch.nn.Linear):
        torch.nn.init.kaiming_normal_(m.weight)
        torch.nn.init.zeros_(m.bias)


class IID_model(object):
    def __init__(self, args: dict):
        self.sequence_file = args["sequence_file"]
        self.GT_file = args["GT_file"]
        self.n_clusters = args["n_clusters"]
        self.k = args["k"]
        if args["model_size"] == "linear":
            self.n_features = 4 ** self.k
            self.reduce = False
            self.net = NetLinear(self.n_features, args["n_clusters"])
        elif args["model_size"] == "small":   # canonical (reverse-complement folded) k-mers, idelucs/models.py:60-66
            self.n_features = (4 ** self.k + 4 ** (self.k // 2)) // 2 if self.k % 2 == 0 else (4 ** self.k) // 2
            self.reduce = True
            self.net = myNet(self.n_features, args["n_clusters"])
        elif args["model_size"] == "full":
            raise ValueError("model_size='full' (ResNet18 on FCGR images, idelucs/models.py:68-69) is outside the featurisation hot path; "
                             "use 'linear' or 'small'")
        else:
            raise ValueError("Invalid Model Type")
        self.net.apply(weights_init)
        self.net.to(device)
        self.epoch = 0
        self.EPS = sys.float_info.epsilon
        self.n_mimics = args["n_mimics"]
        self.batch_sz = args["batch_sz"]
        self.l = args["lambda"]
        self.lr = args["lr"]
        self.weight = args["weight"]
        self.schedule = args["scheduler"]
        opt = args["optimizer"]
        if opt == "RMSprop":
            self.optimizer = optim.RMSprop(self.net.parameters(), lr=self.lr, weight_decay=0.01)
        elif opt == "SGD":
            self.optimizer = optim.SGD(self.net.parameters(), lr=self.lr, weight_decay=0.01, momentum=0.9)
        elif opt == "Adam":
            self.optimizer = optim.Adam(self.net.parameters(), lr=self.lr)
        else:
            raise ValueError("Optimizer not supported")
        if self.schedule == "Plateau":
            self.scheduler = optim.lr_scheduler.ReduceLROnPlateau(self.optimizer, "min")
        elif self.schedule == "Triangle":
            self.scheduler = optim.lr_scheduler.CyclicLR(self.optimizer, base_lr=0.001, max_lr=0.1, step_size_up=5, mode="triangular2")
        self._test = None

    def build_dataloader(self):
        self.dataloader = create_dataloader(self.sequence_file, self.n_mimics, k=self.k, batch_size=self.batch_sz,
                                            GT_file=self.GT_file, reduce=self.reduce)

    def training_step(self, sample, modified):
        self.optimizer.zero_grad(set_to_none=True)
        z1, h1 = self.net(sample)
        z2, h2 = self.net(modified)
        loss = (1 - self.weight) * info_nce_loss(h1, h2, 0.85) + self.weight * IID_loss(z1, z2, lamb=self.l)
        loss.backward()
        self.optimizer.step()
        return loss.detach()

    def contrastive_training_epoch(self):
        """idelucs/models.py:113-143 (including ``running_loss /= i_batch``, the index of the last
        batch — a single-batch epoch therefore divides by zero exactly like the reference)."""
        self.net.train()
        running = torch.zeros((), device=device)
        i_batch = 0
        for i_batch, batch in enumerate(self.dataloader):
            running += self.training_step(batch["true"], batch["modified"])
        running = running / i_batch if i_batch else running / torch.zeros((), device=device)
        if self.schedule == "Plateau":
            self.scheduler.step(running)
        elif self.schedule == "Triangle":
            self.scheduler.step()
        self.epoch += 1
        return running.item()

    def _test_set(self):
        if self._test is None:
            self._test = SequenceDataset(self.sequence_file, k=self.k, transform=None, GT_file=self.GT_file, reduce=self.reduce)
        return self._test

    def predict(self, data=None, device_latent=False):
        """idelucs/models.py:145-172 -> (y_pred int[N], probabilities float[N], latent float[N,64]); with device_latent the
        latent stays on the device as the float32 tensor the network produced (what hdbscan_device takes)"""
        x = self._test_set().kmers32
        y_pred, probs, latent = [], [], []
        with torch.no_grad():
            self.net.eval()
            for b in range(0, x.shape[0], self.batch_sz):
                out, lat = self.net(x[b:b + self.batch_sz])
                p, pred = torch.max(out, 1)
                y_pred.append(pred)
                probs.append(p)
                latent.append(lat)
        latent = torch.cat(latent)
        return (torch.cat(y_pred).cpu().numpy(), torch.cat(probs).cpu().numpy().astype(np.float64),
                latent if device_latent else latent.cpu().numpy().astype(np.float64))

    def calculate_probs(self, data=None):
        """idelucs/models.py:175-195 -> float[N, n_clusters]"""
        x = self._test_set().kmers32
        outs = []
        with torch.no_grad():
            self.net.eval()
            for b in range(0, x.shape[0], self.batch_sz):
                outs.append(self.net(x[b:b + self.batch_sz])[0])
        return torch.cat(outs).cpu().numpy().astype(np.float64)
