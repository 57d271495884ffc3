"""Data-parallel plumbing: one process per GPU, envs sharded across ranks (SURVEY section 8e).

Exchange steps of the hot path and who performs them:

* per minibatch step -- the gradient of each net: summed INSIDE ``spo_pg_update_dp``: every
  rank pushes its gradient into peer-mapped staging slots over NVLink/NVSwitch and raises
  sequence flags; receivers only touch their own memory (csrc/spo_update.cu).
  This module only allocates those buffers, exchanges their CUDA-IPC handles through
  ``torch.distributed`` and hands the kernel the device-side pointer tables.
* per pass -- the KL sum (one fp64): ``all_reduce`` between ``spo_actor_kl_accumulate`` and
  ``spo_kl_finalize`` so every rank takes the same early-stop decision.
* per epoch -- advantage statistics (4 fp64) and the mean episode cost Jc ("fast" mode of
  SURVEY 8e: sum and count of the per-episode running means are reduced, each rank keeps its
  own 50-episode deque).

``torch.distributed`` (NCCL on GPUs, gloo in the CPU tests) is the transport for everything
that is not inside a kernel.  The weights are broadcast from rank 0 once; afterwards every
rank applies bit-identical updates (the in-kernel sum runs in rank order on all ranks).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from safepo import _lib as L


class DataParallel:
    def __init__(self, group=None):
        if not dist.is_initialized():
            raise L.SpoError("DataParallel needs an initialised torch.distributed process group")
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.seq = 0                 # minibatch steps completed by every rank on this communicator
        self._peer = None

    # ---- reductions outside kernels ------------------------------------------------------
    def all_reduce_sum(self, t):
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return t

    def all_reduce_mean(self, t):
        """In-place mean over the ranks (equal shard sizes: the mean of the per-rank means is the global mean).
        Every rank receives bit-identical values, so replicated follow-up arithmetic stays in lock-step."""
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        t.div_(self.world)
        return t

    def broadcast(self, t, src=0):
        dist.broadcast(t, src=src, group=self.group)
        return t

    def mean_episode_cost(self, logger, key="Metrics/EpCost", device=None):
        """Jc for the Lagrange update with the logger's 0.0 / NaN semantics kept
        (logger.py:369-373): global mean of the values stored on all ranks this epoch."""
        vals = logger.epoch_dict.get(key, [])
        seen = 1.0 if key in logger.log_headers else 0.0
        t = torch.tensor([float(np.sum(vals)) if len(vals) else 0.0, float(len(vals)), seen], dtype=torch.float64,
                         device=device)
        self.all_reduce_sum(t)
        s, n, seen_any = (float(x) for x in t.cpu())
        if seen_any == 0.0:
            return 0.0
        return s / n if n > 0 else float("nan")

    # ---- peer-mapped staging for the in-kernel gradient sum --------------------------------
    def setup_peer_buffers(self, dims, device):
        slot = C.c_int()
        L.call("spo_comm_slot_floats", C.byref(dims), C.byref(slot))
        nbytes_grad = 2 * self.world * 3 * slot.value * 4      # [parity][source rank][net][slot] 8-byte {value, sequence} words
        own = []
        for nbytes in (nbytes_grad, max(256, 4 * 3 * self.world)):
            ptr = C.c_void_p()
            L.call("spo_comm_alloc", nbytes, C.byref(ptr))
            own.append(ptr.value)
        handles = []
        for ptr in own:
            buf = C.create_string_buffer(64)
            L.call("spo_comm_export", ptr, buf)
            handles.append(buf.raw)
        gathered = [None] * self.world
        dist.all_gather_object(gathered, handles, group=self.group)
        grads, flags = [], []
        for r, (hg, hf) in enumerate(gathered):
            if r == self.rank:
                grads.append(own[0]); flags.append(own[1])
                continue
            pg, pf = C.c_void_p(), C.c_void_p()
            L.call("spo_comm_import", hg, C.byref(pg))
            L.call("spo_comm_import", hf, C.byref(pf))
            grads.append(pg.value); flags.append(pf.value)
        self._peer = {
            "own": own, "grads": grads, "flags": flags,
            "grad_table": torch.tensor(grads, dtype=torch.int64, device=device),
            "flag_table": torch.tensor(flags, dtype=torch.int64, device=device),
        }
        dist.barrier(group=self.group)
        return self._peer

    def comm_struct(self, spin_limit=0):
        p = self._peer
        return L.Comm(self.world, self.rank, p["grad_table"].data_ptr(), p["flag_table"].data_ptr(), self.seq, spin_limit)

    def advance(self, n_steps):
        self.seq += int(n_steps)

    def close(self):
        if self._peer is None:
            return
        lib = L.lib()
        dist.barrier(group=self.group)
        for r in range(self.world):
            if r != self.rank:
                lib.spo_comm_close(self._peer["grads"][r])
                lib.spo_comm_close(self._peer["flags"][r])
        dist.barrier(group=self.group)
        for ptr in self._peer["own"]:
            lib.spo_comm_free(ptr)
        self._peer = None
