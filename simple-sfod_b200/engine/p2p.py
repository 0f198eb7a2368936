"""NVLink peer-memory exchange of the AdaBN statistics (SURVEY.md 8e, collective (2)).

``PeerStatExchange`` owns one inbox per rank (``sfod_p2p_alloc``), ships its CUDA IPC handle to the other processes of the
node through ``torch.distributed`` (host plumbing only) and maps theirs; ``ops.bn_train_forward(group=<PeerStatExchange>)``
then runs ``sfod_bn_finalize_apply`` with the exchange's comm: the all-reduce of the (sum x, sum x^2, count) payload happens INSIDE the
finalize kernel with P2P stores and flags (csrc/bn.cu), instead of one NCCL all-reduce launch per BN layer
(``engine/adabn_dist.py``, the baseline it is measured against in ``bench.py``'s ``adabn`` record).

Reference: the train-mode forwards of daod/engine/trainers/base.py:270-337 (AdaBN) and
daod/engine/trainers/source_free_adaptive_teacher.py:385-390 (teacher) executed data-parallel.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Tuple

import torch

from .. import _lib


class PeerStatExchange:
    """One rank's endpoint of the exchange.  Build it with ``PeerStatExchange.from_process_group()`` (one process per GPU) or
    ``PeerStatExchange.local_ring()`` (several ranks inside one process, e.g. on separate streams of one GPU: tests)."""

    def __init__(self, rank: int, world: int, inboxes: List[int], device: torch.device, owned: Optional[int], opened: List[int]):
        if not (1 <= world <= _lib.P2P_MAX_RANKS and 0 <= rank < world and len(inboxes) == world):
            raise ValueError("PeerStatExchange: 1 <= world <= 8 ranks, one inbox pointer per rank")
        self.rank, self.world, self.device = rank, world, device
        self.comm = _lib.P2PComm()
        self.comm.rank, self.comm.world = rank, world
        for r, p in enumerate(inboxes):
            self.comm.inbox[r] = p
        self._owned, self._opened = owned, list(opened)
        self.max_channels = int(_lib.lib().sfod_p2p_max_channels())

    # ------------------------------------------------------------------------------------------------ construction
    @staticmethod
    def _alloc(device: torch.device, want_handle: bool) -> Tuple[int, bytes]:
        L = _lib.lib()
        ptr = C.c_void_p()
        handle = (C.c_ubyte * _lib.P2P_HANDLE_BYTES)()
        with torch.cuda.device(device):
            _lib.check(L.sfod_p2p_alloc(C.byref(ptr), handle if want_handle else None), "sfod_p2p_alloc")
        return int(ptr.value), bytes(handle)

    @classmethod
    def from_process_group(cls, group=None, device: Optional[torch.device] = None, probe: bool = True) -> "PeerStatExchange":
        """Collective over ``group`` (default group when None): every rank allocates its inbox, the IPC handles travel through
        ``all_gather_object`` and every rank maps its peers' inboxes.  All ranks must live on GPUs of one node with peer access;
        ``probe`` verifies that with one exchange of a known payload and raises on every rank if it does not come through."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("PeerStatExchange.from_process_group needs an initialised torch.distributed process group")
        device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        if world > _lib.P2P_MAX_RANKS:
            raise ValueError(f"PeerStatExchange supports up to {_lib.P2P_MAX_RANKS} ranks (one NVSwitch node)")
        # Every step that can fail locally is followed by a collective agreement, so that either ALL ranks obtain an endpoint or
        # ALL ranks raise -- a rank that bailed out alone would leave its peers polling for a payload that never comes.
        L = _lib.lib()
        own, handle, err = None, None, None
        try:
            own, handle = cls._alloc(device, True)
        except Exception as e:   # noqa: BLE001 - reported to every rank below
            err = f"rank {rank}: {type(e).__name__}: {e}"
        gathered: List[Optional[tuple]] = [None] * world
        dist.all_gather_object(gathered, (handle, err), group=group)
        errors = [g[1] for g in gathered if g[1] is not None]
        inboxes, opened = [], []
        if not errors:
            try:
                with torch.cuda.device(device):
                    for r in range(world):
                        if r == rank:
                            inboxes.append(own)
                            continue
                        buf = (C.c_ubyte * _lib.P2P_HANDLE_BYTES).from_buffer_copy(gathered[r][0])
                        p = C.c_void_p()
                        _lib.check(L.sfod_p2p_open(buf, C.byref(p)), f"sfod_p2p_open(rank {r})")
                        inboxes.append(int(p.value))
                        opened.append(int(p.value))
            except Exception as e:   # noqa: BLE001
                err = f"rank {rank}: {type(e).__name__}: {e}"
            gathered2: List[Optional[str]] = [None] * world
            dist.all_gather_object(gathered2, err, group=group)   # also the barrier: nobody exchanges before every mapping exists
            errors = [g for g in gathered2 if g is not None]
        if errors:
            if opened or own is not None:
                with torch.cuda.device(device):
                    for p in opened:
                        L.sfod_p2p_close(p)
                    if own is not None:
                        L.sfod_p2p_free(own)
            raise RuntimeError("PeerStatExchange: peer memory is not usable on this node: " + "; ".join(errors)[:500])
        self = cls(rank, world, inboxes, device, own, opened)
        if probe:
            self._probe(group)
        return self

    def _probe(self, group) -> None:
        """One exchange of a known payload: every rank must see the sum over all ranks and no timeout, otherwise ALL ranks raise
        (a node whose peer stores do not arrive would otherwise cost ~3 s per BN layer before anybody noticed)."""
        import torch.distributed as dist
        from .. import ops
        x = torch.full((1, 4, 2, 2), float(self.rank + 1), device=self.device)
        rm, rv = torch.zeros(4, device=self.device), torch.ones(4, device=self.device)
        ops.bn_train_forward(x, None, None, rm, rv, None, momentum=1.0, group=self, compute_output=False)
        _, timeouts = self.status()
        want = (self.world + 1) / 2.0                                   # mean of 1..world
        ok = timeouts == 0 and bool(torch.allclose(rm.cpu(), torch.full((4,), want), rtol=1e-6))
        flag = torch.tensor([1 if ok else 0], device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        if int(flag.item()) == 0:
            self.close()
            raise RuntimeError(f"PeerStatExchange: probe exchange failed on some rank (this rank: timeouts={timeouts}, "
                               f"running_mean={rm.tolist()}, expected {want}); peer access between the GPUs of this node is not usable")

    @classmethod
    def local_ring(cls, world: int, device: Optional[torch.device] = None) -> List["PeerStatExchange"]:
        """``world`` endpoints inside this process whose inboxes are plain allocations on ``device``: each endpoint must be
        driven from its own stream (the exchange kernels of all ranks have to be resident at the same time)."""
        device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        ptrs = [cls._alloc(device, False)[0] for _ in range(world)]
        return [cls(r, world, ptrs, device, ptrs[r], []) for r in range(world)]

    # ------------------------------------------------------------------------------------------------ use
    def status(self) -> Tuple[int, int]:
        """(exchanges completed, exchanges abandoned on a timeout) -- synchronises the device."""
        ex, to = C.c_uint64(0), C.c_uint32(0)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().sfod_p2p_status(C.byref(self.comm), C.byref(ex), C.byref(to)), "sfod_p2p_status")
        return int(ex.value), int(to.value)

    def close(self) -> None:
        L = _lib.lib()
        with torch.cuda.device(self.device):
            for p in self._opened:
                L.sfod_p2p_close(p)
            self._opened = []
            if self._owned is not None:
                L.sfod_p2p_free(self._owned)
                self._owned = None
