"""Value-network trainer: mirror of crowd_nav/utils/trainer.py:19-82 (MSE, SGD momentum 0.9, batch 100).

Batches are drawn directly from the device-resident replay tensors instead of a DataLoader over Python tuples.
Three execution forms of the same optimisation step (MSE -> backward -> [gradient all-reduce] -> SGD momentum):

* ``fused``  (CUDA; SARL and OM-SARL with or without the global state, CADRL, LSTM-RL ValueNetwork1 / 2 with or without
  occupancy maps): the hand-written forward / backward kernel + SGD kernel of the C ABI (``cn_trainer_*``,
  csrc/trainer.cu, csrc/trainer_nets.cu) working on ONE flat fp32 parameter block that the torch model's parameters are
  views of; the gradient all-reduce (NCCL, one bucket: 386 kB for SARL) sits between the two kernels.
* ``graph``  (CUDA, any network): torch autograd captured once per batch shape into a CUDA graph and replayed.
* ``eager``  (CPU / gloo tests, odd batch sizes): plain torch autograd.

No form synchronises with the host per batch: the loss is accumulated on the device and read once per
``optimize_*`` call (the reference's ``loss.data.item()`` per batch, trainer.py:54,76, is a host sync per step).

Data parallel (SURVEY §8(e)): replay buffers stay rank-local, gradients are averaged over ranks, so every rank must
run the SAME number of steps per call: the step count comes from the LARGEST ``len(memory)`` over the ranks and short
ranks wrap around their own buffer.
"""
import logging

import torch
import torch.nn as nn
import torch.optim as optim


def sample_batches(n, b, num_batches, device):
    """(num_batches, b) indices into a memory of n items; every row is a uniform sample WITHOUT replacement in random order
    -- the head of a fresh shuffle, what next(iter(DataLoader(shuffle=True))) yields (trainer.py:68).  Drawn with replacement
    and repaired: rows of b << n items rarely collide (b^2 / 2n), so a few re-draws of the colliding entries converge; the
    exact fallback (b largest of n uniform keys per row) only runs if collisions survive, e.g. for n close to b."""
    if b >= n:
        return torch.stack([torch.randperm(n, device=device)[:b] for _ in range(num_batches)])
    idx = torch.randint(n, (num_batches, b), device=device)
    for _ in range(6):
        srt, order = torch.sort(idx, dim=1)
        dup_sorted = torch.zeros_like(srt, dtype=torch.bool)
        dup_sorted[:, 1:] = srt[:, 1:] == srt[:, :-1]
        dup = torch.zeros_like(dup_sorted).scatter_(1, order, dup_sorted)
        if not bool(dup.any()):                   # one small host sync per round; almost always the first or second
            return idx
        idx = torch.where(dup, torch.randint(n, idx.shape, device=device), idx)
    rows = max(1, min(num_batches, (1 << 25) // n))
    return torch.cat([torch.rand((min(rows, num_batches - i), n), device=device).topk(b, dim=1).indices
                      for i in range(0, num_batches, rows)])


class Trainer(object):
    def __init__(self, model, memory, device, batch_size, dist_group=None, policy=None, mode=None):
        self.model = model
        self.device = device
        self.criterion = nn.MSELoss().to(device)
        self.memory = memory
        self.data_loader = None          # kept for interface parity; batches come from the replay tensors
        self.batch_size = batch_size
        self.optimizer = None
        self.dist_group = dist_group
        self.policy = policy             # SARL façade whose GPU lookahead weights are refreshed after training
        self.lr = None
        self.momentum = 0.9
        is_cuda = torch.device(device).type == "cuda"
        self.mode = mode or ("graph" if is_cuda else "eager")
        assert self.mode in ("eager", "graph", "fused")
        if self.mode != "eager" and not is_cuda:
            raise ValueError("Trainer mode %r needs a CUDA device" % self.mode)
        self._graphs = {}                # (B, state shape) -> (CUDAGraph, x, y, loss)
        self._fused = None
        self._loss_sum = None

    def set_learning_rate(self, learning_rate):
        logging.info("Current learning rate: %f", learning_rate)
        self.lr = float(learning_rate)
        if self.mode == "fused":
            from .fused_trainer import FusedTrainer
            if self._fused is None:
                self._fused = FusedTrainer(self.model, self.device, momentum=self.momentum)
            self._fused.lr = self.lr
            self.optimizer = self._fused          # "Learning rate is not set!" check below
            return
        self.optimizer = optim.SGD(self.model.parameters(), lr=learning_rate, momentum=self.momentum)
        self._graphs.clear()                      # captured graphs hold the old optimiser's buffers

    # -- data-parallel plumbing ---------------------------------------------------------------------
    def _world(self):
        if self.dist_group is None:
            return 1
        import torch.distributed as dist
        return dist.get_world_size(self.dist_group)

    def _common_len(self):
        """len(memory) every rank iterates over: the maximum over the ranks (one tiny all-reduce per optimize_* call)."""
        n = len(self.memory)
        if self.dist_group is None:
            return n
        import torch.distributed as dist
        dev = self.device if dist.get_backend(self.dist_group) == "nccl" else "cpu"
        t = torch.tensor([n], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.dist_group)
        return int(t.item())

    def _sync_gradients(self):
        """Average the gradients over the ranks as ONE flat bucket (96,502 fp32 = 386 kB: latency bound)."""
        if self.dist_group is None:
            return
        import torch.distributed as dist
        params = [p for p in self.model.parameters() if p.grad is not None]
        flat = torch.cat([p.grad.reshape(-1) for p in params])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.dist_group)
        flat /= dist.get_world_size(self.dist_group)
        off = 0
        for p in params:
            n = p.grad.numel()
            p.grad.copy_(flat[off:off + n].view_as(p.grad))
            off += n

    def broadcast_weights(self, src=0):
        """Make every rank start from rank `src`'s weights (after load_state_dict / random init)."""
        if self.dist_group is None:
            return
        import torch.distributed as dist
        for p in self.model.parameters():
            dist.broadcast(p.data, src=src, group=self.dist_group)

    # -- one optimisation step ------------------------------------------------------------------------
    def _eager_step(self, inputs, values):
        self.optimizer.zero_grad()
        outputs = self.model(inputs)
        loss = self.criterion(outputs, values)
        loss.backward()
        self._sync_gradients()
        self.optimizer.step()
        return loss.detach()

    def _graph_step(self, inputs, values):
        key = (tuple(inputs.shape), tuple(values.shape))
        g = self._graphs.get(key)
        if g is None:
            x, y = inputs.clone(), values.clone()
            # warm-up on a side stream (allocates the gradients and the momentum buffers), restoring the weights after
            saved = [p.detach().clone() for p in self.model.parameters()]
            saved_mom = {id(p): st["momentum_buffer"].detach().clone() for p, st in self.optimizer.state.items()
                         if st.get("momentum_buffer") is not None}
            s = torch.cuda.Stream(device=self.device)
            s.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(s):
                for _ in range(2):
                    self.optimizer.zero_grad(set_to_none=False)
                    loss = self.criterion(self.model(x), y)
                    loss.backward()
                    self.optimizer.step()
            torch.cuda.current_stream(self.device).wait_stream(s)
            with torch.no_grad():
                for p, q in zip(self.model.parameters(), saved):
                    p.copy_(q)
                for p, st in self.optimizer.state.items():
                    if st.get("momentum_buffer") is not None:       # a fresh optimiser starts from zero momentum
                        if id(p) in saved_mom:
                            st["momentum_buffer"].copy_(saved_mom[id(p)])
                        else:
                            st["momentum_buffer"].zero_()
            params = [p for p in self.model.parameters()]
            graph = torch.cuda.CUDAGraph()
            graph2, flat = None, None
            if self.dist_group is None:
                with torch.cuda.graph(graph):
                    self.optimizer.zero_grad(set_to_none=False)
                    loss = self.criterion(self.model(x), y)
                    loss.backward()
                    self.optimizer.step()
            else:
                # data parallel: the NCCL all-reduce stays OUTSIDE the captured work (the process group's watchdog thread
                # polls CUDA events, which is not allowed while a capture is open): graph 1 = forward + backward + gradient
                # bucket, eager all-reduce of the one 386 kB bucket, graph 2 = un-bucket + SGD step
                with torch.cuda.graph(graph):
                    self.optimizer.zero_grad(set_to_none=False)
                    loss = self.criterion(self.model(x), y)
                    loss.backward()
                    flat = torch.cat([p.grad.reshape(-1) for p in params])
                graph2 = torch.cuda.CUDAGraph()
                scale = 1.0 / self._world()
                with torch.cuda.graph(graph2, pool=graph.pool()):
                    off = 0
                    for p in params:
                        n = p.grad.numel()
                        p.grad.copy_(flat[off:off + n].view_as(p.grad) * scale)
                        off += n
                    self.optimizer.step()
            # SGD's first step copies the gradient into the momentum buffer (buf = grad) and later ones do
            # buf = mu * buf + grad; with the buffers zeroed above the captured "later" form covers both.
            g = self._graphs[key] = (graph, x, y, loss, graph2, flat)
        graph, x, y, loss, graph2, flat = g
        x.copy_(inputs); y.copy_(values)
        graph.replay()
        if graph2 is not None:
            import torch.distributed as dist
            dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.dist_group)
            graph2.replay()
        return loss

    def _step_tensors(self, inputs, values):
        if self.mode == "fused":
            return self._fused.step(inputs, values, self.dist_group)
        if self.mode == "graph" and inputs.shape[0] == self.batch_size:
            return self._graph_step(inputs, values)
        return self._eager_step(inputs, values)

    def _step(self, idx):
        """One SGD step on memory[idx]; returns the loss as a 0-d device tensor (no host sync)."""
        inputs = self.memory.states[idx].to(self.device)
        values = self.memory.values[idx].to(self.device)
        return self._step_tensors(inputs, values)

    def _fused_indexed_ok(self):
        m = self.memory
        if self.mode != "fused" or getattr(m, "states", None) is None:
            return False
        # (capacity, H, D) replay tensors; CADRL's single-human states are (capacity, D)
        shape_ok = m.states.dim() == 2 if self._fused.single_human else (
            m.states.dim() == 3 and m.states.shape[1] <= self._fused.max_humans)
        return (shape_ok and m.states.is_cuda and m.states.dtype == torch.float32 and m.values.dtype == torch.float32
                and m.states.is_contiguous() and m.values.is_contiguous())

    def _after(self):
        if self._fused is not None:
            self._fused.flush_to_model()
        if self.policy is not None:
            self.policy.sync_weights()

    # -- the reference entry points ---------------------------------------------------------------------
    def optimize_epoch(self, num_epochs):
        """trainer.py:36-59: num_epochs passes over a shuffled memory."""
        if self.optimizer is None:
            raise ValueError("Learning rate is not set!")
        n_local = len(self.memory)
        n = self._common_len()
        if n_local == 0:
            raise ValueError("optimize_epoch on an empty replay memory")
        mdev = self.memory.states.device
        average_epoch_loss = 0
        for _ in range(num_epochs):
            epoch_loss = torch.zeros((), dtype=torch.float32, device=self.device)
            perm = torch.randperm(n, device=mdev)
            if n != n_local:
                perm = perm % n_local            # short ranks wrap around: same number of steps (and collectives) everywhere
            if self._fused_indexed_ok():
                for s in range(0, n, self.batch_size):
                    self._fused.step_indexed(self.memory.states, self.memory.values, perm[s:s + self.batch_size].contiguous(),
                                             epoch_loss, self.dist_group)
            else:
                for s in range(0, n, self.batch_size):
                    epoch_loss += self._step(perm[s:s + self.batch_size]).to(self.device)
            average_epoch_loss = float(epoch_loss.item()) / n
            logging.debug("Average loss in epoch : %.2E", average_epoch_loss)
        self._after()
        return average_epoch_loss

    def optimize_batch(self, num_batches):
        """trainer.py:61-82: each batch is the head of a fresh shuffle (next(iter(DataLoader(shuffle=True))))."""
        if self.optimizer is None:
            raise ValueError("Learning rate is not set!")
        n = len(self.memory)
        if n == 0:
            raise ValueError("optimize_batch on an empty replay memory")
        mdev = self.memory.states.device
        losses = torch.zeros((), dtype=torch.float32, device=self.device)
        b = min(self.batch_size, n)
        idx = sample_batches(n, b, num_batches, mdev)
        if self._fused_indexed_ok():
            # the fused step gathers memory[idx] inside its kernel and accumulates the loss on the device: one C call per batch
            for i in range(num_batches):
                self._fused.step_indexed(self.memory.states, self.memory.values, idx[i], losses, self.dist_group)
        else:
            for i in range(num_batches):
                losses += self._step(idx[i]).to(self.device)
        average_loss = float(losses.item()) / num_batches
        logging.debug("Average loss : %.2E", average_loss)
        self._after()
        return average_loss
