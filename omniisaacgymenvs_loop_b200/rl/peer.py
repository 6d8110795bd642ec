"""PeerAllReduce: the PPO gradient all-reduce over NVLink peer memory (include/usv_b200.h: ppo_peer_*).

Replaces `dist.all_reduce(grads)` [ref: RLG/common/a2c_common.py:308-323] by one kernel that never leaves the stream, so the update
phase can be captured in a CUDA graph on every rank.  torch.distributed is used once, at construction, to exchange the 64-byte
CUDA-IPC handles of the per-rank windows (one process per GPU, same node)."""
from __future__ import annotations

import ctypes

import torch
import torch.distributed as dist

from .. import _lib


class PeerAllReduce:
    def __init__(self, count: int, device, rank: int = 0, world_size: int = 1, group=None):
        self.lib = _lib.lib()
        self.device = torch.device(device)
        self.rank, self.world, self.cap = int(rank), int(world_size), (int(count) + 3) // 4 * 4
        if self.world > 16:
            raise ValueError("PeerAllReduce supports up to 16 ranks on one node")
        with torch.cuda.device(self.device):
            win = ctypes.c_void_p()
            handle = (ctypes.c_ubyte * 64)()
            _lib.check(self.lib.ppo_peer_window_alloc(ctypes.c_int64(self.cap), ctypes.byref(win), handle), "ppo_peer_window_alloc")
            self._own = win
            handles = [None] * self.world
            if self.world > 1:
                dist.all_gather_object(handles, bytes(handle), group=group)
            else:
                handles[0] = bytes(handle)
            self.comm = _lib.PpoPeerComm()
            self.comm.cap, self.comm.world, self.comm.rank = self.cap, self.world, self.rank
            self._opened = []
            for r in range(self.world):
                if r == self.rank:
                    self.comm.windows[r] = win.value
                    continue
                p = ctypes.c_void_p()
                buf = (ctypes.c_ubyte * 64).from_buffer_copy(handles[r])
                _lib.check(self.lib.ppo_peer_window_open(buf, ctypes.byref(p)), f"ppo_peer_window_open(rank {r})")
                self.comm.windows[r] = p.value
                self._opened.append(p)
            self.seq = torch.zeros(1, dtype=torch.int32, device=self.device)
            self.err = torch.zeros(1, dtype=torch.int32, device=self.device)
        if self.world > 1:
            dist.barrier(group=group)          # every window is mapped everywhere before the first kernel signals

    def __call__(self, src: torch.Tensor, dst: torch.Tensor | None = None) -> torch.Tensor:
        """dst = sum over ranks of src (in place when dst is None); asynchronous on the current stream, graph-capturable."""
        dst = src if dst is None else dst
        rc = self.lib.ppo_peer_allreduce_f32(ctypes.byref(self.comm), _lib.ptr(src, torch.float32), _lib.ptr(dst, torch.float32),
                                             ctypes.c_int64(src.numel()), _lib.ptr(self.seq), _lib.ptr(self.err), _lib.stream())
        _lib.check(rc, "ppo_peer_allreduce_f32")
        return dst

    def check(self) -> None:
        """Raises if a peer failed to arrive within the kernel's spin bound (one host sync; call once per epoch at most)."""
        if int(self.err.item()) != 0:
            raise RuntimeError("PeerAllReduce: a peer rank did not reach the all-reduce (spin bound expired)")

    def clear_error(self) -> None:
        self.err.zero_()

    def close(self) -> None:
        for p in self._opened:
            self.lib.ppo_peer_window_close(p, ctypes.c_int32(0))
        self._opened = []
        if self._own is not None:
            self.lib.ppo_peer_window_close(self._own, ctypes.c_int32(1))
            self._own = None


class PeerStepExchange(PeerAllReduce):
    """The windows of the all-reduce that runs INSIDE the fused minibatch tail kernel (ppo_minibatch_step_peer_tc): per rank
    [2 parities][world][entries] packets of 8 bytes {value, sequence}.  Same IPC plumbing as PeerAllReduce; its own sequence counter."""

    def __init__(self, obs_dim: int, device, rank: int = 0, world_size: int = 1, group=None):
        entries = int(_lib.lib().ppo_minibatch_step_peer_entries(ctypes.c_int32(int(obs_dim))))
        if entries <= 0:
            raise ValueError(f"no tensor-core minibatch step for obs_dim {obs_dim}")
        self.entries = entries
        super().__init__(int(world_size) * entries * 2, device, rank, world_size, group)


class PeerLoopzExchange(PeerAllReduce):
    """The windows of the loopz learner's two exchanges (ppo_loopz_returns_peer_f32: advantage moments once per update,
    ppo_loopz_grad_exchange_f32: the gradient once per minibatch): per rank [2 parities][world][entries] packets of 8 bytes
    {value, sequence}, one sequence counter {sequence, arrival counter} shared by both."""

    def __init__(self, net, device, rank: int = 0, world_size: int = 1, group=None):
        entries = int(_lib.lib().ppo_loopz_peer_entries(ctypes.byref(net)))
        if entries <= 0:
            raise ValueError("unsupported loopz network shape")
        self.entries = entries
        super().__init__(int(world_size) * entries * 2, device, rank, world_size, group)
        self.seq = torch.zeros(2, dtype=torch.int32, device=self.device)


class InProcessStepExchange:
    """`world` ranks of the fused exchange living in ONE process on ONE device (each rank drives its own stream): the windows are plain
    device allocations instead of IPC mappings, the kernel and its packet protocol are the same.  Used to exercise the multi-rank
    data path where only one GPU is visible (tests/test_gpu_ppo.py); `ranks[r]` quacks like a PeerStepExchange."""

    class _Rank:
        pass

    def __init__(self, obs_dim: int, device, world_size: int):
        self._build(int(_lib.lib().ppo_minibatch_step_peer_entries(ctypes.c_int32(int(obs_dim)))), device, world_size, 1)

    def _build(self, entries: int, device, world_size: int, seq_words: int):
        cap = int(world_size) * entries * 2
        self.windows = [torch.zeros(2 * cap + 64, dtype=torch.float32, device=device) for _ in range(world_size)]
        self.ranks = []
        for r in range(world_size):
            k = self._Rank()
            k.world, k.rank = int(world_size), r
            k.comm = _lib.PpoPeerComm()
            k.comm.cap, k.comm.world, k.comm.rank = cap, int(world_size), r
            for q in range(world_size):
                k.comm.windows[q] = self.windows[q].data_ptr()
            k.seq = torch.zeros(seq_words, dtype=torch.int32, device=device)
            k.err = torch.zeros(1, dtype=torch.int32, device=device)
            k.check = PeerAllReduce.check.__get__(k)
            self.ranks.append(k)


class InProcessLoopzExchange(InProcessStepExchange):
    """In-process ranks of PeerLoopzExchange (tests/test_gpu_loopz_peer.py): `ranks[r]` goes to PPO(..., peer=...)."""

    def __init__(self, net, device, world_size: int):
        self._build(int(_lib.lib().ppo_loopz_peer_entries(ctypes.byref(net))), device, world_size, 2)
