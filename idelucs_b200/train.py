"""Sharded training loop on top of the hot path (BASELINE.json configs[3]: synthetic 1 M x 2 kb,
k=6, n_mimics=50, batch_sz=512, sharded over 1/2/4/8 B200).

Each rank owns a contiguous shard of the packed sequences, regenerates its pair batches on the fly with the mimic kernel (selection
mode — the 1.6 TB x_train of the reference never exists) and runs the reference's training step (idelucs/models.py:113-143: two
forwards, (1-w) InfoNCE + w IIC loss, backward, RMSprop or the SGD / Adam of `optimizer=`) as ONE CUDA graph on two streams:

  * every dense contraction of the encoder stays a PyTorch / cuBLAS GEMM in strict fp32, issued in the shape that fills the GPU for
    this batch (_FirstLinear / _FlatLinear: inner-dimension splits as batched GEMMs, gradients written straight into a flat buffer);
  * everything between the GEMMs is a hand-written kernel behind the C ABI: ReLU - Dropout fused with the tail of the GEMM before it,
    the two losses with their weights and gradients (LossFunctions.train_losses_and_grads seeds the backward pass), the optimiser;
  * parameters, gradients and the RMSprop state live in flat buffers; with several ranks ONE kernel averages the gradient slices over
    NVLink (8.5 MB at k=6), applies RMSprop and broadcasts the new parameters (idl_rmsprop_allreduce_step);
  * the next pair batch is regenerated on the side stream under the middle of the step.

batch_sz is PER RANK (weak scaling in the batch, strong in the data set)."""
import torch
import torch.distributed as dist

from . import featurise as ft
from .LossFunctions import GlobalBatchLoss, train_losses_and_grads
from .PytorchUtils import NetLinear
from .models import weights_init

OPTIMIZERS = {"RMSprop": 1, "SGD": 1, "Adam": 2}   # the optimisers of idelucs/models.py:86-99 -> state buffers per parameter
SGD_MOMENTUM = 0.9
ADAM_BETAS = (0.9, 0.999)


def _relu_dropout_fwd(parts, n_parts, bias, M, N, drop):
    """idl_relu_dropout_forward on [n_parts, M, N] partial products (+ bias): the post-dropout activations [M, N]"""
    from . import _lib
    lib = _lib.load()
    p, seed, step, tag = drop
    out = torch.empty((M, N), dtype=torch.float32, device=parts.device)
    with torch.cuda.device(parts.device):
        _lib.check(lib.idl_relu_dropout_forward(_lib.ptr(parts), n_parts, _lib.ptr(bias), M, N, float(p), int(seed) & (2 ** 64 - 1), _lib.ptr(step),
                                                int(tag), _lib.ptr(out), _lib.stream_ptr()))
    return out


def _relu_dropout_bwd(out, dy, p):
    from . import _lib
    lib = _lib.load()
    dy = dy.contiguous()
    dx = torch.empty_like(out)
    with torch.cuda.device(out.device):
        _lib.check(lib.idl_relu_dropout_backward(_lib.ptr(out), _lib.ptr(dy), out.numel(), float(p), _lib.ptr(dx), _lib.stream_ptr()))
    return dx


class _ReluDropout(torch.autograd.Function):
    """ReLU - Dropout(p) (idelucs/PytorchUtils.py:40-44) as one kernel each way; the backward needs no stored mask (the output is
    positive exactly where the unit was active and kept)."""

    @staticmethod
    def forward(ctx, x, drop):
        x = x.contiguous()
        out = _relu_dropout_fwd(x, 1, None, x.shape[0], x.shape[1], drop)
        ctx.save_for_backward(out)
        ctx.p = drop[0]
        return out

    @staticmethod
    def backward(ctx, dy):
        (out,) = ctx.saved_tensors
        return _relu_dropout_bwd(out, dy, ctx.p), None


class _FirstLinear(torch.autograd.Function):
    """The encoder's first Linear (4^k -> 512: 97 % of the MLP's flops) as PyTorch / cuBLAS calls shaped for this batch: the forward
    contraction [2B, 4^k] x [4^k, 512] is split over its inner dimension into ONE batched GEMM (more output tiles than SMs: 110 ->
    84 us at 2B = 1024 in strict fp32); the backward writes the weight gradient straight into its slice of the flat gradient buffer
    (no zero-fill and no accumulate pass over 8.4 MB) and needs no input gradient.  With ``drop`` = (p, seed, step tensor, tag) the
    ReLU - Dropout behind the layer is part of it: the parts of the split GEMM, the bias, the activation and the dropout are ONE
    kernel (idl_relu_dropout_forward) instead of a reduction and three elementwise launches, and the output is the activation."""

    @staticmethod
    def forward(ctx, x, weight, bias, gw_out, gb_out, n_split, side=None, drop=None):
        M, K = x.shape
        N = weight.shape[0]
        if n_split > 1 and K % n_split == 0:
            parts = torch.bmm(x.view(M, n_split, K // n_split).transpose(0, 1), weight.view(N, n_split, K // n_split).permute(1, 2, 0))
        else:
            n_split = 1
            parts = torch.mm(x, weight.t())
        if drop is not None:
            out = _relu_dropout_fwd(parts, n_split, bias, M, N, drop)
            ctx.save_for_backward(x, out)
        else:
            out = parts.sum(0) if n_split > 1 else parts
            out += bias
            ctx.save_for_backward(x)
        ctx.gw_out, ctx.gb_out, ctx.side, ctx.drop = gw_out, gb_out, side, drop
        return out

    @staticmethod
    def backward(ctx, dy):
        if ctx.drop is not None:
            x, out = ctx.saved_tensors
            dy = _relu_dropout_bwd(out, dy, ctx.drop[0])
        else:
            (x,) = ctx.saved_tensors
        if ctx.side is not None:   # the bias gradient (a column sum) runs beside the weight-gradient GEMM; the caller joins the streams
            main = torch.cuda.current_stream(dy.device)
            ctx.side.wait_stream(main)
            with torch.cuda.stream(ctx.side):
                torch.sum(dy, 0, out=ctx.gb_out)
            torch.mm(dy.t(), x, out=ctx.gw_out)
        else:
            torch.mm(dy.t(), x, out=ctx.gw_out)
            torch.sum(dy, 0, out=ctx.gb_out)
        return None, None, None, None, None, None, None, None


def _split_mm(a, b, ns):
    """a [M, K] @ b [K, N] as ONE batched GEMM over ns slices of K -> partial products [ns, M, N] (a GEMM with few output tiles
    leaves most SMs idle: [1024, 512] x [512, 64] takes 11 us as one GEMM, 4.6 us split 8-fold — tools/mlp_probe.py)"""
    M, K = a.shape
    N = b.shape[1]
    aa = a.reshape(M, ns, K // ns).transpose(0, 1) if a.is_contiguous() else a.t().reshape(ns, K // ns, M).transpose(1, 2)
    bb = b.reshape(ns, K // ns, N) if b.is_contiguous() else b.t().reshape(N, ns, K // ns).permute(1, 2, 0)
    return torch.bmm(aa, bb)


class _FlatLinear(torch.autograd.Function):
    """A later Linear of the encoder: its weight and bias gradients go straight into their slices of the flat gradient buffer (no
    zero-fill, no accumulate pass per parameter), the bias gradient of a wide layer as a [1, M] x [M, N] product (the framework's
    column reduction of a [1024, 64] matrix takes 10 us).  ``split`` = (forward, weight-gradient) inner-dimension splits of the two
    contractions with few output tiles; the parts are added by idl_sum_parts_bias / one reduction into the flat buffer."""

    @staticmethod
    def forward(ctx, x, weight, bias, gw_out, gb_out, ones, split=(1, 1)):
        ctx.save_for_backward(x, weight)
        ctx.gw_out, ctx.gb_out, ctx.ones, ctx.wsplit = gw_out, gb_out, ones, split[1]
        M, K = x.shape
        N = weight.shape[0]
        if split[0] > 1 and K % split[0] == 0 and N % 4 == 0 and x.is_contiguous():
            from . import _lib
            lib = _lib.load()
            parts = _split_mm(x, weight.t(), split[0])
            out = torch.empty((M, N), dtype=torch.float32, device=x.device)
            with torch.cuda.device(x.device):
                _lib.check(lib.idl_sum_parts_bias(_lib.ptr(parts), split[0], _lib.ptr(bias), M, N, _lib.ptr(out), _lib.stream_ptr()))
            return out
        return torch.addmm(bias, x, weight.t())

    @staticmethod
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        M, N = dy.shape
        dy = dy.contiguous()
        if ctx.wsplit > 1 and M % ctx.wsplit == 0:
            torch.sum(_split_mm(dy.t(), x, ctx.wsplit), 0, out=ctx.gw_out)
        else:
            torch.mm(dy.t(), x, out=ctx.gw_out)
        if N >= 32 and ctx.ones.shape[1] >= M:
            torch.mm(ctx.ones[:, :M], dy, out=ctx.gb_out.view(1, N))
        else:
            torch.sum(dy, 0, out=ctx.gb_out)
        return torch.mm(dy, weight), None, None, None, None, None, None


class ShardedTrainer(object):
    """Data-parallel replica of the reference's training step (idelucs/models.py:113-143) fed by the mimic kernel.

    Step layout (captured in ONE CUDA graph, two streams; kernel timeline: profiles/train_timeline_r2.txt):
      main stream  first Linear's forward (batched split GEMM) + its ReLU - Dropout kernel -> second / third Linear -> fused InfoNCE +
                   IIC losses, whose gradients seed the backward -> backward, every gradient written into ONE flat buffer -> optimiser:
                   idl_rmsprop_step at N = 1; with several ranks idl_rmsprop_allreduce_step (gradient mean + RMSprop + parameter
                   broadcast as one kernel over NVLink peer memory: symmetric buffers, NVLS multimem when available; NCCL
                   all-reduce + idl_rmsprop_step when symmetric memory cannot be set up);
      side stream  pair batch t+1 regenerated from the packed sequences (selection mode of idl_profiles, one CTA per SM) under the
                   small kernels of the middle of the step, the first layer's bias gradient beside its weight-gradient GEMM, the
                   hand-over of the batch beside the optimiser.
    The parameters of the network are views into one flat buffer, so the optimiser and the collectives see one tensor.
    With several ranks and global_batch_loss=True the losses are those of all ranks' pairs together (_global_losses); by default,
    and always at one rank, each rank's losses are those of its own batch_sz pairs."""

    def __init__(self, seqset, k=6, n_clusters=5, n_mimics=50, batch_sz=512, lamb=2.8, weight=0.25, lr=1e-3, seed=0,
                 seq_id0=0, world=1, materialize_bytes=0, alpha=0.99, eps=1e-8, weight_decay=None, use_symmetric_memory=True,
                 overlap_featurise_with="forward", optimizer="RMSprop", global_batch_loss=False):
        from .utils import PairBatchLoader
        if optimizer not in OPTIMIZERS:
            raise ValueError("optimizer must be one of %s, got %r" % (", ".join(OPTIMIZERS), optimizer))
        if weight_decay is None:   # idelucs/models.py:86-99: RMSprop and SGD with weight_decay=0.01, Adam without
            weight_decay = 0.0 if optimizer == "Adam" else 0.01
        self.dev = seqset.device
        self.world = world
        self.rank = dist.get_rank() if world > 1 else 0
        group = dist.group.WORLD if world > 1 else None
        self.loader = PairBatchLoader(seqset, n_mimics, k=k, batch_size=batch_sz, seed=seed, group=group, seq_id0=seq_id0,
                                      materialize_bytes=materialize_bytes, drop_last=True)
        torch.manual_seed(seed)  # identical initial replicas on every rank
        net = NetLinear(4 ** k, n_clusters)
        net.apply(weights_init)
        net.to(self.dev)
        self.net = net
        # ---- flat parameter / gradient / second-moment buffers (padded to a multiple of 4 * world elements).  With several
        # ranks the two big buffers are SYMMETRIC memory (every rank maps every rank's copy, plus an NVLS multicast address when
        # the fabric has one): the optimiser step is then ONE kernel that reduces, updates and broadcasts over NVLink ----
        params = [p for p in net.parameters() if p.requires_grad]
        n = sum(p.numel() for p in params)
        self._n = n
        pad = (-n) % (4 * world)
        self._mode = "single"
        self._flat_param = self._flat_grad = None
        # global_batch_loss (several ranks): the step's losses are those of the world * batch_sz pairs together, exchanged between
        # the ranks (LossFunctions.GlobalBatchLoss); at one rank the local batch already is the global one
        self._gsizes = GlobalBatchLoss.buffer_sizes(world, batch_sz, n_clusters, net.layers[3].out_features) if world > 1 and global_batch_loss else None
        self._gloss = None
        if world > 1 and use_symmetric_memory:
            try:
                self._setup_symmetric(n + pad)
                self._mode = "symm"
            except Exception as e:  # noqa: BLE001 — symmetric memory not available on this fabric / build: NCCL all-reduce instead
                self._symm_error = repr(e)
        if world > 1:   # every rank must take the same path
            okf = torch.tensor([1.0 if self._mode == "symm" else 0.0], device=self.dev)
            dist.all_reduce(okf, op=dist.ReduceOp.MIN)
            self._mode = "symm" if float(okf.item()) == 1.0 else "nccl"
        if self._mode != "symm":
            self._flat_param = torch.zeros(n + pad, dtype=torch.float32, device=self.dev)
            self._flat_grad = torch.zeros(n + pad, dtype=torch.float32, device=self.dev)
        if self._gsizes is not None:
            self._setup_global_loss(batch_sz, n_clusters, net.layers[3].out_features, lamb, weight)
        o = 0
        for p in params:
            self._flat_param[o:o + p.numel()].copy_(p.data.reshape(-1))
            p.data = self._flat_param[o:o + p.numel()].view_as(p)
            p.grad = self._flat_grad[o:o + p.numel()].view_as(p)
            o += p.numel()
        self.first_layer_split = 4
        self.small_gemm_split = (8, 16)   # forward / weight-gradient splits of the later Linears' contractions
        self._ones = torch.ones((1, 2 * batch_sz), dtype=torch.float32, device=self.dev)
        self._step_no = torch.zeros((), dtype=torch.int64, device=self.dev)
        self._drop_seed = (seed * 1000003 + 7919 * self.rank + 12345) & (2 ** 63 - 1)   # dropout masks differ between the replicas
        if world > 1:   # replicas must start identical whatever the RNG state of the rank was
            dist.broadcast(self._flat_param, src=0)
        self._shard = (n + pad) // world if self._mode == "symm" else n + pad
        # optimiser state of this rank's slice: RMSprop's square average (_sq), SGD's momentum buffer, Adam's two moments
        self.optimizer = optimizer
        self._state = [torch.zeros(self._shard, dtype=torch.float32, device=self.dev) for _ in range(OPTIMIZERS[optimizer])]
        self._sq = self._state[0] if optimizer == "RMSprop" else None
        self._loss_sum = torch.zeros((), dtype=torch.float32, device=self.dev)   # sum of the step losses since epoch_loss()
        self.lr, self.alpha, self.eps, self.weight_decay = lr, alpha, eps, weight_decay
        self.overlap_featurise_with = overlap_featurise_with
        self.lamb, self.weight, self.batch_sz = lamb, weight, batch_sz
        self.gen = torch.Generator(device=self.dev).manual_seed(seed * 1000003 + seq_id0 + 1)
        self._graph = None
        self._ids = torch.zeros(batch_sz, dtype=torch.int64, device=self.dev)       # pair ids of the NEXT batch (graph input)
        self._perm, self._cursor, self.epoch = None, 0, 0
        self._side = torch.cuda.Stream(device=self.dev)
        self._batch = None       # the batch the next step consumes (featurised by the previous step; static buffer once created)

    def _setup_symmetric(self, n_total):
        import ctypes
        import torch.distributed._symmetric_memory as symm
        grp = dist.group.WORLD
        g = symm.empty(n_total, dtype=torch.float32, device=self.dev)
        p = symm.empty(n_total, dtype=torch.float32, device=self.dev)
        self._hg, self._hp = symm.rendezvous(g, grp), symm.rendezvous(p, grp)
        g.zero_(); p.zero_()
        self._flat_grad, self._flat_param = g, p
        self._gp = (ctypes.c_uint64 * self.world)(*[int(x) for x in self._hg.buffer_ptrs])
        self._pp = (ctypes.c_uint64 * self.world)(*[int(x) for x in self._hp.buffer_ptrs])
        mc_g = int(getattr(self._hg, "multicast_ptr", 0) or 0)
        mc_p = int(getattr(self._hp, "multicast_ptr", 0) or 0)
        self._mc = (mc_g, mc_p) if (mc_g and mc_p) else (0, 0)
        if self._gsizes is not None:   # the two buffers of the global-batch loss every rank reads
            self._gsend = [symm.empty(n, dtype=torch.float32, device=self.dev) for n in self._gsizes]
            self._gh = [symm.rendezvous(t, grp) for t in self._gsend]
            for t in self._gsend:
                t.zero_()

    def _setup_global_loss(self, b, C, D, lamb, weight):
        """GlobalBatchLoss of this rank: its send buffers are symmetric memory (peers read them in place after a barrier) or, with
        NCCL, local tensors all-gathered into one copy per rank"""
        if self._mode == "symm":
            gl = GlobalBatchLoss(self.rank, self.world, b, C, D, self.dev, lamb, weight, send=self._gsend)
            gl.set_peers(*[[int(a) for a in h.buffer_ptrs] for h in self._gh])
        else:
            gl = GlobalBatchLoss(self.rank, self.world, b, C, D, self.dev, lamb, weight)
            self._gathered = [torch.zeros(self.world * n, dtype=torch.float32, device=self.dev) for n in self._gsizes]
            gl.set_peers(*[[g.data_ptr() + 4 * n * r for r in range(self.world)] for g, n in zip(self._gathered, self._gsizes)])
        self._gloss = gl

    def _global_losses(self, z, h):
        """LossFunctions.GlobalBatchLoss's three stages with the exchanges between them: (loss, dz, dh) of this rank's rows.
        Symmetric memory: one barrier after each rank wrote send1 (partial joint, normalised latent) and one after send2
        (G_r^T fn_r, row losses); peers then read both in place.  No barrier is needed before a rank overwrites them in the next
        step: every peer's last read (stage 3) precedes, in its stream order, its arrival at the optimiser's first barrier, and
        this rank writes again only after passing that barrier.  NCCL: each buffer is all-gathered instead."""
        gl = self._gloss
        gl.stage1(z, h)
        for k, send in enumerate((gl.send1, gl.send2)):
            if self._mode == "symm":
                self._gh[k].barrier(channel=0)
            else:
                dist.all_gather_into_tensor(self._gathered[k], send)
            if k == 0:
                gl.stage2()
        return gl.stage3()

    # ---- optimiser: torch.optim.RMSprop's / SGD's / Adam's arithmetic on flat buffers ----
    def _optimizer_step(self):
        from . import _lib
        lib = _lib.load()
        st = [_lib.ptr(t) for t in self._state]
        step = _lib.ptr(self._step_no)   # (SGD's first step and Adam's bias corrections: the counter the step incremented)
        with torch.cuda.device(self.dev):
            if self._mode == "symm":
                # ONE kernel: mean of every rank's gradient slice (NVLS multimem.ld_reduce, or peer loads) -> the update of this rank's
                # slice -> new parameters stored into every rank's buffer; symmetric-memory barriers (5 us each) on both sides
                peers = (self._gp, self._pp, self._mc[0], self._mc[1])
                n, r, w = self._flat_grad.numel(), self.rank, self.world
                self._hg.barrier(channel=0)
                if self.optimizer == "RMSprop":
                    rc = lib.idl_rmsprop_allreduce_step(*peers, *st, n, r, w, self.lr, self.alpha, self.eps, self.weight_decay, _lib.stream_ptr())
                elif self.optimizer == "SGD":
                    rc = lib.idl_sgd_allreduce_step(*peers, *st, n, r, w, self.lr, SGD_MOMENTUM, self.weight_decay, step, _lib.stream_ptr())
                else:
                    rc = lib.idl_adam_allreduce_step(*peers, *st, n, r, w, self.lr, *ADAM_BETAS, self.eps, self.weight_decay, step,
                                                     _lib.stream_ptr())
                _lib.check(rc)
                self._hp.barrier(channel=0)
                return
            if self._mode == "nccl":
                dist.all_reduce(self._flat_grad, op=dist.ReduceOp.AVG)
            p, g = _lib.ptr(self._flat_param), _lib.ptr(self._flat_grad)
            if self.optimizer == "RMSprop":
                rc = lib.idl_rmsprop_step(p, g, *st, self._shard, self.lr, self.alpha, self.eps, self.weight_decay, 1.0, _lib.stream_ptr())
            elif self.optimizer == "SGD":
                rc = lib.idl_sgd_step(p, g, *st, self._shard, self.lr, SGD_MOMENTUM, self.weight_decay, step, 1.0, _lib.stream_ptr())
            else:
                rc = lib.idl_adam_step(p, g, *st, self._shard, self.lr, *ADAM_BETAS, self.eps, self.weight_decay, step, 1.0, _lib.stream_ptr())
            _lib.check(rc)

    def reinit(self, seed):
        """A fresh voter (idelucs/__main__.py:106-109): new Kaiming-normal weights and zero biases (models.weights_init, drawn on
        rank 0 from `seed` and broadcast).  The optimiser state and the step counter are kept, as the reference keeps its
        optimiser between voters; every buffer stays in place, so a captured CUDA graph stays valid."""
        if self.rank == 0:
            with torch.random.fork_rng(devices=[self.dev]):
                torch.manual_seed(seed)
                self.net.apply(weights_init)   # (in place: the parameters are views into the flat buffer)
        if self.world > 1:
            dist.broadcast(self._flat_param, src=0)

    def reset_optimizer(self):
        """zero the optimiser state and the step counter: the state of a fresh torch optimiser (after the warm-up steps of
        enable_cuda_graph, before the first voter)"""
        for t in self._state:
            t.zero_()
        self._step_no.zero_()
        self._loss_sum.zero_()

    def epoch_loss(self, n_steps):
        """the mean loss of the n_steps steps since the last call, as contrastive_training_epoch divides it (idelucs/models.py:
        137-143: the sum over the epoch over the index of its last batch, n_steps - 1), averaged over the ranks; read once per
        epoch (one synchronisation), then the accumulator restarts"""
        s = self._loss_sum.clone()
        self._loss_sum.zero_()
        if self.world > 1:
            dist.all_reduce(s, op=dist.ReduceOp.AVG)
        return float((s / float(n_steps - 1)).item()) if n_steps > 1 else float((s / torch.zeros_like(s)).item())

    def enable_cuda_graph(self, warmup=11):
        """Capture the whole step (both streams) in ONE CUDA graph: the step is launch-bound, so replaying a graph removes the
        host from the loop.  The pair ids of the next batch are the only input (static buffer filled before every replay).
        Returns False (and stays eager) if capture is not possible."""
        try:
            s = torch.cuda.Stream(device=self.dev)
            s.wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(s):
                for _ in range(warmup):
                    self._ids.copy_(self._next_ids())
                    self._step_from_ids()
            torch.cuda.current_stream(self.dev).wait_stream(s)
            g = torch.cuda.CUDAGraph()
            if self.world > 1:
                # the NCCL watchdog thread polls events while this thread captures: only this thread's calls may
                # invalidate the capture
                torch.cuda.synchronize(self.dev)
                with torch.cuda.graph(g, stream=s, capture_error_mode="thread_local"):
                    self._loss = self._step_from_ids()
            else:
                with torch.cuda.graph(g, stream=s):
                    self._loss = self._step_from_ids()
            self._graph = g
        except Exception as e:  # noqa: BLE001 — eager fallback of an optimisation, not of the CUDA path
            self._graph = None
            self._graph_error = repr(e)
            torch.cuda.synchronize(self.dev)
        if self.world > 1:   # all ranks replay the graph or none does (a rank that fell back must not face captured collectives alone)
            okf = torch.tensor([1.0 if self._graph is not None else 0.0], device=self.dev)
            dist.all_reduce(okf, op=dist.ReduceOp.MIN)
            if float(okf.item()) < 1.0:
                self._graph = None
        return self._graph is not None

    def _next_ids(self):
        """the next batch of a shuffled epoch over this rank's pairs: every pair once per epoch, a fresh permutation per
        epoch, the ragged tail dropped (DataLoader(shuffle=True) of idelucs/utils.py:427; the per-rank batch is fixed-size
        because it feeds a captured CUDA graph)"""
        n = self.loader.n_pairs
        if n < self.batch_sz:   # degenerate shard: sample with replacement
            return torch.randint(0, max(n, 1), (self.batch_sz,), device=self.dev, generator=self.gen)
        if self._perm is None or self._cursor + self.batch_sz > n:
            self._perm = torch.randperm(n, device=self.dev, generator=self.gen)
            self._cursor = 0
            self.epoch += 1
        ids = self._perm[self._cursor:self._cursor + self.batch_sz]
        self._cursor += self.batch_sz
        return ids

    def _featurise(self, ids, cta_cap=0):
        """pair batch as one stacked [2B, F] tensor (rows 0..B-1 = 'true' side)"""
        batch = self.loader.batch(ids, cta_cap=cta_cap)
        if "both" in batch:
            return batch["both"]
        return torch.cat((batch["true"], batch["modified"]), 0)

    def step(self):
        """one training step on the next batch of this rank's shuffled pairs; returns the loss tensor"""
        if self._batch is None:   # the very first batch has no previous step to featurise it
            self._batch = self._featurise(self._next_ids()).clone()
        self._ids.copy_(self._next_ids())
        if self._graph is not None:
            self._graph.replay()
            return self._loss
        return self._step_from_ids()

    def _drop(self, tag):
        """dropout descriptor of the fused ReLU - Dropout kernels: (p, seed, step counter on the device, layer tag); p = 0 in eval mode"""
        return (0.5 if self.net.training else 0.0, self._drop_seed, self._step_no, tag)

    def _tail(self, d1):
        """NetLinear.forward behind the first Linear - ReLU - Dropout block (PytorchUtils.py: Linear -> latent; ReLU - Dropout -
        Linear - Softmax -> cluster probabilities), the two Linears through _FlatLinear: (cluster probabilities, latent)"""
        lin2, lin3 = self.net.layers[3], self.net.classifier[2]
        h = _FlatLinear.apply(d1, lin2.weight, lin2.bias, lin2.weight.grad, lin2.bias.grad, self._ones, self.small_gemm_split)
        z = torch.softmax(_FlatLinear.apply(_ReluDropout.apply(h, self._drop(2)), lin3.weight, lin3.bias, lin3.weight.grad, lin3.bias.grad,
                                            self._ones, (1, self.small_gemm_split[1])), 1)
        return z, h

    def _forward(self, x, side=None):
        """NetLinear.forward with the Linears issued by _FirstLinear / _FlatLinear and ReLU - Dropout by the fused kernels: (cluster
        probabilities, latent) of the stacked batch"""
        lin1 = self.net.layers[0]
        d1 = _FirstLinear.apply(x, lin1.weight, lin1.bias, lin1.weight.grad, lin1.bias.grad, self.first_layer_split, side, self._drop(1))
        return self._tail(d1)

    def _step_from_ids(self):
        if self._batch is None:
            self._batch = self._featurise(self._ids).clone()
        main = torch.cuda.current_stream(self.dev)
        # ---- side stream: batch t+1 (ids in self._ids) into a fresh buffer.  One rank: under the MIDDLE of the step — the two big
        # GEMMs of the first layer (forward at the start, weight gradient at the end) fill every SM's register file, and a
        # featurisation kernel launched beside them only delays them (measured: 28 us of idle main stream); between them sit ~160 us
        # of small GEMMs, losses and elementwise kernels that leave the SMs mostly empty.  The kernel is capped at one CTA per SM so
        # that those small kernels still find room.  Several ranks: under the optimiser step, whose kernel waits on NVLink, not on SMs ----
        late = self.world > 1 and self.overlap_featurise_with == "optimizer"
        nxt = None
        # ---- main stream: step t on self._batch ----
        x = self._batch
        # (every parameter's gradient is WRITTEN by _FirstLinear / _FlatLinear into its slice of the flat buffer: nothing to zero)
        # one pass over the stacked [2B, F] batch: same per-row math as the reference's two forwards
        lin1 = self.net.layers[0]
        self._step_no.add_(1)   # (the fused dropout kernels read it on the device: a graph replay draws fresh masks)
        d1 = _FirstLinear.apply(x, lin1.weight, lin1.bias, lin1.weight.grad, lin1.bias.grad, self.first_layer_split, self._side, self._drop(1))
        if not late:
            self._side.wait_stream(main)          # (after the first layer's forward GEMM)
            with torch.cuda.stream(self._side):
                nxt = self._featurise(self._ids, cta_cap=1)
        z, h = self._tail(d1)
        # (1 - w) InfoNCE + w IIC (models.py:128) and its gradients with respect to z and h straight from the fused kernels (the
        # weights ride inside them); the MLP's backward pass is seeded with those — no framework kernel between forward and backward
        if self._gloss is not None:
            loss, dz, dh = self._global_losses(z, h)
        else:
            loss, dz, dh = train_losses_and_grads(z, h, self.lamb, self.weight, 0.85)
        self._side.wait_stream(main)          # (the epoch's loss sum: a one-element add beside the backward pass, off the main stream)
        with torch.cuda.stream(self._side):
            self._loss_sum.add_(loss)
        torch.autograd.backward((z, h), (dz, dh))
        if late:
            self._side.wait_stream(main)
            with torch.cuda.stream(self._side):
                nxt = self._featurise(self._ids)
        if late:
            self._optimizer_step()
            main.wait_stream(self._side)
            self._batch.copy_(nxt)   # (static buffer: the graph's next replay reads it)
            return loss
        # the hand-over of batch t+1 into the static buffer (16 MB) rides on the side stream beside the optimiser step: x's last
        # reader (the first layer's weight-gradient GEMM) is done, the featurisation and the bias gradient are earlier on that stream
        main.wait_event(self._side.record_event())   # the bias gradient of the first layer, before the optimiser reads it
        self._side.wait_stream(main)
        with torch.cuda.stream(self._side):
            self._batch.copy_(nxt)
        self._optimizer_step()
        main.wait_stream(self._side)
        return loss

    @torch.no_grad()
    def predict(self, seqset, k=6, batch=4096):
        """idelucs/models.py:145-172 over the sharded sequences: (y_pred int64[N], probabilities float32[N], latent
        float32[N, 64]) of ALL sequences on every rank — each rank featurises and scores its own shard (clean float64
        profiles, one StandardScaler over all shards), then the three row blocks are all-gathered in rank order."""
        from . import parallel
        f64 = ft.profiles(seqset, k, [ft.VariantSpec(ft.KIND_CLEAN)], out_kind=ft.OUT_FREQ_F64)[0]
        sc = ft.Scaler.fit(f64, group=dist.group.WORLD if self.world > 1 else None)
        x = sc.transform64(f64, want32=True)
        net = self.net
        net.eval()
        preds, probs, lats = [], [], []
        for b in range(0, x.shape[0], batch):
            out, lat = net(x[b:b + batch])
            pr, pd = torch.max(out, 1)
            preds.append(pd); probs.append(pr); lats.append(lat)
        net.train()
        C = lats[0].shape[1] if lats else 64
        preds = torch.cat(preds) if preds else torch.zeros(0, dtype=torch.int64, device=self.dev)
        probs = torch.cat(probs) if probs else torch.zeros(0, dtype=torch.float32, device=self.dev)
        lats = torch.cat(lats) if lats else torch.zeros((0, C), dtype=torch.float32, device=self.dev)
        if self.world > 1:
            preds, probs, lats = parallel.all_gather_ragged([preds, probs, lats])
        return preds, probs, lats
