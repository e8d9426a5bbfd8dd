"""Loss functions with the reference's names and signatures (idelucs/LossFunctions.py).

``IID_loss`` / ``compute_joint`` run the fused sm_100a kernel K5 (forward + backward in one launch) through the C ABI.
``info_nce_loss`` (SURVEY §8f rank 2) runs the fused InfoNCE kernels (idl_nce_*: normalise, masked log-softmax +
cross-entropy + gradient weights, normalisation backward) around two strict-fp32 cuBLAS GEMMs on CUDA tensors."""
import ctypes
import sys

import torch
import torch.nn.functional as F

from . import _lib


def _ws(device, C):
    from .featurise import _workspace
    return _workspace(device, _lib.load().idl_iid_loss_workspace_bytes(C), "loss%d" % C)


_IID_GEMM_MIN_C = 17   # above the single-CTA kernels' range: contractions as library GEMMs + idl_iid_joint_algebra


def _iid_device(z1, z2, lamb, EPS, want_grad=True, want_joint=False, grad_scale=1.0, loss_weight=1.0, add=None, add_weight=0.0,
                dz1=None, dz2=None):
    """IIC loss of float32 contiguous CUDA [B, C] tensors (may be the two halves of one stacked tensor): (loss, joint, dz1, dz2).
    C <= 16: one launch (idl_iid_loss_scaled: register-resident / single-CTA kernels).  Larger C (the 200 output units of the
    embedding path): S = z1^T z2, dz1 = z2 dS, dz2 = z1 dS as three small strict-fp32 GEMMs around idl_iid_joint_algebra (the C
    ABI's idl_iid_loss runs the same algebra between two contraction kernels of its own)."""
    lib = _lib.load()
    B, C = z1.shape
    dev = z1.device
    loss = torch.empty((), dtype=torch.float32, device=dev)
    joint = torch.empty((C, C), dtype=torch.float32, device=dev) if want_joint else None
    if want_grad:
        dz1 = torch.empty_like(z1) if dz1 is None else dz1
        dz2 = torch.empty_like(z2) if dz2 is None else dz2
    else:
        dz1 = dz2 = None
    with torch.cuda.device(dev):
        if C < _IID_GEMM_MIN_C:
            ws = _ws(dev, C)
            _lib.check(lib.idl_iid_loss_scaled(_lib.ptr(z1), _lib.ptr(z2), B, C, float(lamb), float(EPS), float(grad_scale), float(loss_weight),
                                               _lib.ptr(add), float(add_weight), _lib.ptr(loss), _lib.ptr(joint), _lib.ptr(dz1), _lib.ptr(dz2),
                                               _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
        else:
            S = torch.mm(z1.t(), z2)
            S = S + S.t()          # the algebra kernel reads the symmetrised joint row by row
            dS = torch.empty_like(S) if want_grad else None
            scratch = torch.empty(6 * C, dtype=torch.float32, device=dev)
            _lib.check(lib.idl_iid_joint_algebra(_lib.ptr(S), C, float(lamb), float(EPS), float(grad_scale), float(loss_weight), _lib.ptr(add),
                                                 float(add_weight), _lib.ptr(loss), _lib.ptr(joint), _lib.ptr(dS), _lib.ptr(scratch),
                                                 _lib.stream_ptr()))
            if want_grad:
                torch.mm(z2, dS, out=dz1)
                torch.mm(z1, dS, out=dz2)
    return loss, joint, dz1, dz2


class _IIDLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x_out, x_tf_out, lamb, EPS):
        if not x_out.is_cuda:
            raise _lib.IdelucsB200Error("IID_loss: tensors must be on a CUDA device (no CPU fallback)")
        z1 = x_out.detach().contiguous().float()
        z2 = x_tf_out.detach().contiguous().float()
        assert z2.shape == z1.shape
        need_grad = x_out.requires_grad or x_tf_out.requires_grad
        loss, _, dz1, dz2 = _iid_device(z1, z2, lamb, EPS, want_grad=need_grad)
        if need_grad:
            ctx.save_for_backward(dz1, dz2)
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        dz1, dz2 = ctx.saved_tensors
        return grad_out * dz1, grad_out * dz2, None, None


def IID_loss(x_out, x_tf_out, lamb=1.0, EPS=sys.float_info.epsilon):
    """idelucs/LossFunctions.py:20-46 — same arguments, returns a 0-d tensor with autograd."""
    return _IIDLoss.apply(x_out, x_tf_out, lamb, EPS)


def compute_joint(x_out, x_tf_out):
    """idelucs/LossFunctions.py:49-62 — symmetrised, normalised joint [C, C] (no autograd)."""
    z1 = x_out.detach().contiguous().float()
    z2 = x_tf_out.detach().contiguous().float()
    return _iid_device(z1, z2, 1.0, sys.float_info.epsilon, want_grad=False, want_joint=True)[1]


_targets = {}
_NCE_SPLIT = 8   # inner-dimension split of the W fn contraction (tools/mlp_probe.py)


def _info_nce_device(x, temperature, grad_scale=1.0):
    """(loss 0-d tensor, grad_scale * dh [n2, D]) of the stacked latent x (float32, contiguous, CUDA): idl_nce_normalize -> S = fn fn^T
    (cuBLAS, strict fp32) -> idl_nce_softmax_xent_scaled (loss; S becomes grad_scale * W in place) -> dfn = W fn (cuBLAS) ->
    idl_nce_normalize_backward"""
    lib = _lib.load()
    n2, D = x.shape
    dev = x.device
    fn = torch.empty_like(x)
    scratch = torch.empty(3 * n2, dtype=torch.float32, device=dev)     # inv_norm | lse | rowloss
    loss = torch.empty((), dtype=torch.float32, device=dev)
    dh = torch.empty_like(x)
    with torch.cuda.device(dev):
        st = _lib.stream_ptr()
        _lib.check(lib.idl_nce_normalize(_lib.ptr(x), n2, D, _lib.ptr(fn), _lib.ptr(scratch), st))
        sim = torch.mm(fn, fn.t())
        _lib.check(lib.idl_nce_softmax_xent_scaled(_lib.ptr(sim), n2, float(temperature), float(grad_scale),
                                                   ctypes.c_void_p(scratch.data_ptr() + 4 * n2), ctypes.c_void_p(scratch.data_ptr() + 8 * n2),
                                                   _lib.ptr(loss), st))
        # dfn = W fn: [n2, n2] x [n2, D] has n2 * D / tile outputs only — split over the inner dimension into ONE batched GEMM
        # (18 -> 6 us at n2 = 1024, D = 64); the normalisation's backward adds the parts
        ns = _NCE_SPLIT if n2 % _NCE_SPLIT == 0 and n2 >= 256 else 1
        if ns > 1:
            dfn = torch.bmm(sim.view(n2, ns, n2 // ns).transpose(0, 1), fn.view(ns, n2 // ns, D))
        else:
            dfn = torch.mm(sim, fn)
        _lib.check(lib.idl_nce_normalize_backward_parts(_lib.ptr(dfn), ns, _lib.ptr(fn), _lib.ptr(scratch), n2, D, _lib.ptr(dh), st))
    return loss, dh


def train_losses_and_grads(z, h, lamb, weight, temperature=0.85, EPS=sys.float_info.epsilon):
    """(1 - w) info_nce_loss + w IID_loss of one stacked forward (idelucs/models.py:128) WITH its gradients, no autograd node:
    returns (loss, dLoss/dz, dLoss/dh).  The weights ride inside the kernels (idl_nce_softmax_xent_scaled, idl_iid_loss_scaled, the
    latter also combines the two loss values), so between the MLP's forward and its backward there are our four kernels, the IIC
    kernel and two GEMMs — no framework kernel.  A trainer seeds the backward pass with
    ``torch.autograd.backward((z, h), (dz, dh))``."""
    lib = _lib.load()
    zz = z.detach().contiguous().float()
    n2, C = zz.shape
    B = n2 // 2
    nce, dh = _info_nce_device(h.detach().contiguous().float(), temperature, grad_scale=1.0 - weight)
    dz = torch.empty_like(zz)
    loss, _, _, _ = _iid_device(zz[:B], zz[B:], lamb, EPS, grad_scale=weight, loss_weight=weight, add=nce, add_weight=1.0 - weight,
                                dz1=dz[:B], dz2=dz[B:])
    return loss, dz, dh


class GlobalBatchLoss(object):
    """train_losses_and_grads of the GLOBAL batch for one rank of a data-parallel step: W ranks of b pairs each, the loss of the
    B = W b pairs together (idelucs/models.py:128 on the batch one GPU would train on), the gradients of this rank's rows.

    Global row order: [true rows of rank 0 .. W-1 ; modified rows of rank 0 .. W-1].  Two buffers per rank are read by the others:
      send1 = [S2_r = z1_r^T z2_r + its transpose (C x C, padded to 4) | fn_r, the normalised latent [2b, D]]
      send2 = [G_r^T fn_r [2B, D] | the 2b row losses of InfoNCE (padded to 4)]
    ``set_peers`` gives the device addresses of every rank's send1 / send2 (symmetric memory, or the slots of all-gathered copies).
    A step is ``stage1(z, h)`` (writes send1), exchange, ``stage2()`` (writes send2), exchange, ``stage3()`` -> (loss, dz, dh).
    The loss is the same on every rank; dz and dh are multiplied by W, because the optimiser averages the ranks' gradients and the
    update must be that of the gradient of the global loss.  All cross-rank sums run in rank order (no float atomics)."""

    def __init__(self, rank, world, b, C, D, device, lamb, weight, temperature=0.85, EPS=sys.float_info.epsilon, send=None):
        self.rank, self.world, self.b, self.C, self.D = rank, world, b, C, D
        self.lamb, self.weight, self.temperature, self.EPS = lamb, weight, temperature, EPS
        B = world * b
        self.n_s2 = C * C + (-C * C) % 4
        self.len1, self.len2 = self.buffer_sizes(world, b, C, D)
        f32 = dict(dtype=torch.float32, device=device)
        self.send1, self.send2 = send if send is not None else (torch.zeros(self.len1, **f32), torch.zeros(self.len2, **f32))
        assert self.send1.numel() >= self.len1 and self.send2.numel() >= self.len2
        self.s2 = self.send1[:C * C]
        self.fn = self.send1[self.n_s2:self.n_s2 + 2 * b * D].view(2 * b, D)
        self.prod = self.send2[:2 * B * D].view(2 * B, D)
        self.rowloss = self.send2[2 * B * D:2 * B * D + 2 * b]
        self.inv_norm = torch.empty(2 * b, **f32)
        self.fn_all = torch.empty((2 * B, D), **f32)
        self.ws = torch.empty(_lib.load().idl_iid_loss_workspace_bytes(C), dtype=torch.uint8, device=device)

    @staticmethod
    def buffer_sizes(world, b, C, D):
        """floats of send1 and send2 (each a multiple of 4, so that slots of an all-gathered copy stay 16-byte aligned)"""
        return C * C + (-C * C) % 4 + 2 * b * D + (-2 * b * D) % 4, 2 * world * b * D + 2 * b + (-2 * b) % 4

    def set_peers(self, addr1, addr2):
        """device addresses (ints, rank order) at which this process reads every rank's send1 / send2"""
        W = self.world
        self._p_s2 = (ctypes.c_uint64 * W)(*addr1)
        self._p_fn = (ctypes.c_uint64 * W)(*[a + 4 * self.n_s2 for a in addr1])
        self._p_prod = (ctypes.c_uint64 * W)(*addr2)

    def stage1(self, z, h):
        """this rank's partial joint and normalised latent into send1"""
        lib = _lib.load()
        b, C = self.b, self.C
        self._z = z.detach().contiguous().float()
        hh = h.detach().contiguous().float()
        with torch.cuda.device(hh.device):
            st = _lib.stream_ptr()
            _lib.check(lib.idl_iid_partial_s2(_lib.ptr(self._z[:b]), _lib.ptr(self._z[b:]), b, C, _lib.ptr(self.s2), st))
            _lib.check(lib.idl_nce_normalize(_lib.ptr(hh), 2 * b, self.D, _lib.ptr(self.fn), _lib.ptr(self.inv_norm), st))

    def stage2(self):
        """(every rank's send1 readable) fn_all, this rank's row block of the similarity -> (1 - w) W G_r, its local term
        G_r fn_all, and G_r^T fn_r with the row losses into send2"""
        lib = _lib.load()
        b, D, W = self.b, self.D, self.world
        with torch.cuda.device(self.fn.device):
            st = _lib.stream_ptr()
            _lib.check(lib.idl_nce_gather_rows(self._p_fn, W, b, D, _lib.ptr(self.fn_all), st))
            sim = torch.mm(self.fn, self.fn_all.t())   # [2b, 2B]: this rank's rows only
            _lib.check(lib.idl_nce_softmax_xent_rows(_lib.ptr(sim), b, self.rank, W, float(self.temperature), float((1.0 - self.weight) * W),
                                                     _lib.ptr(self.rowloss), st))
            self._local = torch.mm(sim, self.fn_all)
            torch.mm(sim.t(), self.fn, out=self.prod)

    def stage3(self):
        """(every rank's send2 readable) (loss, dz, dh) of this rank's rows"""
        lib = _lib.load()
        b, C, D, W = self.b, self.C, self.D, self.world
        dev = self.fn.device
        nce = torch.empty((), dtype=torch.float32, device=dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        dh = torch.empty((2 * b, D), dtype=torch.float32, device=dev)
        dz = torch.empty_like(self._z)
        with torch.cuda.device(dev):
            st = _lib.stream_ptr()
            _lib.check(lib.idl_nce_normalize_backward_global(_lib.ptr(self._local), 1, self._p_prod, W, _lib.ptr(self.fn), _lib.ptr(self.inv_norm),
                                                             b, D, self.rank, _lib.ptr(dh), _lib.ptr(nce), st))
            _lib.check(lib.idl_iid_global_finish(self._p_s2, W, _lib.ptr(self._z[:b]), _lib.ptr(self._z[b:]), b, C, float(self.lamb), float(self.EPS),
                                                 float(self.weight * W), float(self.weight), _lib.ptr(nce), float(1.0 - self.weight), _lib.ptr(loss),
                                                 _lib.ptr(dz[:b]), _lib.ptr(dz[b:]), _lib.ptr(self.ws), self.ws.numel(), st))
        return loss, dz, dh


class _InfoNCE(torch.autograd.Function):
    """fused CUDA form: value and gradient with respect to the stacked latent, computed together in the forward"""

    @staticmethod
    def forward(ctx, h, temperature):
        loss, dh = _info_nce_device(h.detach().contiguous().float(), temperature)
        ctx.save_for_backward(dh)
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        (dh,) = ctx.saved_tensors
        return grad_out * dh, None


class _TrainLosses(torch.autograd.Function):
    """(1 - w) info_nce_loss + w IID_loss of one stacked forward (idelucs/models.py:128) as ONE autograd node: the two fused
    loss paths run back to back on the stacked outputs (no slicing copies, no per-loss autograd bookkeeping) and leave the
    gradients with respect to z and h ready."""

    @staticmethod
    def forward(ctx, z, h, lamb, weight, temperature, EPS):
        loss, dz, dh = train_losses_and_grads(z, h, lamb, weight, temperature, EPS)
        ctx.save_for_backward(dz, dh)
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        dz, dh = ctx.saved_tensors
        return grad_out * dz, grad_out * dh, None, None, None, None


def train_losses(z, h, lamb, weight, temperature=0.85, EPS=sys.float_info.epsilon):
    """the training loss of idelucs/models.py:128 for one stacked forward: z [2B, C] cluster probabilities, h [2B, D] latent
    (rows 0..B-1 = 'true' view)"""
    return _TrainLosses.apply(z, h, lamb, weight, temperature, EPS)


def _info_nce_torch(h, temperature):
    """mask-gather-free PyTorch formulation (any device / width): cross-entropy of the self-masked similarity rows against
    the index of the other view == the reference's [positive, negatives] gather with label 0"""
    n2 = h.shape[0]
    feats = F.normalize(h.float(), dim=1)
    logits = (feats @ feats.T) / temperature
    logits.fill_diagonal_(float("-inf"))      # in place: the division's backward does not need its output
    key = (n2, logits.device)
    if key not in _targets:
        idx = torch.arange(n2, device=logits.device)
        _targets[key] = (idx + n2 // 2) % n2
    return F.cross_entropy(logits, _targets[key])


def info_nce_loss_stacked(h, temperature):
    """info_nce_loss on the two views already stacked as one [2n, d] tensor (rows 0..n-1 = first view).  CUDA tensors take the
    fused kernels around two cuBLAS GEMMs; CPU tensors the PyTorch form (host-side tests only)."""
    if h.is_cuda and h.dim() == 2 and h.shape[0] % 2 == 0 and h.shape[0] >= 2:
        return _InfoNCE.apply(h, temperature)
    return _info_nce_torch(h, temperature)


def info_nce_loss(z1, z2, temperature):
    """SimCLR NT-Xent (idelucs/LossFunctions.py:65-98).  The reference gathers [positive, negatives] per row with boolean
    masks and takes cross-entropy against label 0; that equals the cross-entropy of the self-masked similarity row against
    the index of the other view, which needs no mask gathers (and no host synchronisation)."""
    return info_nce_loss_stacked(torch.cat((z1, z2), 0), temperature)
