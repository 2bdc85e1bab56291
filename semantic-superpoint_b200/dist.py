"""Multi-GPU plumbing (SURVEY 8e): one process per GPU, torch.distributed for rendezvous.

The loss step shards by batch; its only exchange is the global-batch normalisers (both reference losses divide by
whole-batch quantities: Train_model_heatmap_all.py:178, utils/utils.py:886-887).  That exchange is ONE kernel over
peer memory (csrc/exchange.cu: P2P stores over NVLink + release flags, sums in rank order, the fix-ups of all
losses in place) -- no NCCL call inside the step.  `SSP_EXCHANGE=allreduce` (and any CPU / gloo group) selects the
torch.distributed fallback of the same arithmetic: one all-reduce of the packed payload.
Homography adaptation shards by source image with no data-path collective.
"""
import ctypes
import os

import torch
import torch.distributed as tdist


def init_from_env(backend=None):
    """Initialise the default process group from torchrun's environment.  Returns (rank, world, local_rank)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not tdist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
        tdist.init_process_group(backend=backend, rank=rank, world_size=world)
    return rank, world, local


def _group(group):
    return None if group is True else group


def shard_range(n_items, rank, world):
    """Contiguous shard [lo, hi) of n_items for `rank`; sizes differ by at most one."""
    base, rem = divmod(n_items, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


# ------------------------------------------------------------------------------------------------
# the exchange
# ------------------------------------------------------------------------------------------------
# payload slots (csrc/exchange.cu): all are summed over the ranks
_NV = 16


class LossExchange(object):
    """Global-batch fix-up of the loss scalars of one process group.

    run(det0=, det1=, desc8=, sem0=, sem1=, B_local=, Hc=, Wc=) rewrites the given tensors IN PLACE, stream ordered:
      det*  = out3 of a detector loss   {loss, numerator, sum(mask) + 1e-5}
      desc8 = out8 of the descriptor loss {loss, pos, neg, norm, num_loss, num_pos, num_neg, sum(mask_valid)}
      sem*  = out3 of a semantic loss   {loss, sum, count}
    B_local, Hc, Wc: the descriptor loss's shard size and cell grid; its global normaliser is
      B_global * (sum_global(mask_valid) + 1) * Hc * Wc  (utils/utils.py:886-887), B_global the SUM of the ranks' B_local
      (shards may differ by one pair).
    backend "p2p": the peer-memory kernel (CUDA tensors, ranks on one node); "allreduce": one torch all-reduce.
    """

    def __init__(self, group=True, backend=None, timeout_s=30.0):
        self.group = group
        self.rank = tdist.get_rank(_group(group))
        self.world = tdist.get_world_size(_group(group))
        if backend is None:
            backend = os.environ.get("SSP_EXCHANGE") or ("p2p" if torch.cuda.is_available() else "allreduce")
        if backend not in ("p2p", "allreduce"):
            raise ValueError("exchange backend must be 'p2p' or 'allreduce', got %r" % (backend,))
        self.backend = backend
        self.timeout_s = float(timeout_s)
        self.local = None
        self.peers = []
        self.table = None
        if backend == "p2p":
            self._open()

    # -- peer-memory backend ----------------------------------------------------------------------
    def _open(self):
        from . import _lib
        lib = _lib.load()
        if self.world > lib.ssp_xchg_max_ranks():
            raise RuntimeError("loss exchange: %d ranks exceed the %d slots of the exchange buffer" % (self.world, lib.ssp_xchg_max_ranks()))
        handle = ctypes.create_string_buffer(64)
        buf = ctypes.c_void_p()
        _lib.check(lib.ssp_xchg_alloc(ctypes.byref(buf), handle), "ssp_xchg_alloc")
        self.local = buf.value
        mine = (os.uname().nodename, os.getpid(), bytes(handle.raw))
        everyone = [None] * self.world
        tdist.all_gather_object(everyone, mine, group=_group(self.group))
        if any(e[0] != mine[0] for e in everyone):
            raise RuntimeError("loss exchange: the p2p backend needs all ranks on one node (set SSP_EXCHANGE=allreduce)")
        table = (ctypes.c_void_p * self.world)()
        for r, (_node, pid, h) in enumerate(everyone):
            if r == self.rank:
                table[r] = self.local
                continue
            peer = ctypes.c_void_p()
            _lib.check(lib.ssp_xchg_open(ctypes.create_string_buffer(h, 64), ctypes.byref(peer)), "ssp_xchg_open (rank %d)" % r)
            self.peers.append(peer.value)
            table[r] = peer.value
        self.table = table
        tdist.barrier(group=_group(self.group))  # every buffer is zeroed and mapped before anybody pushes into it

    def close(self):
        """Unmap the peers' buffers and free the local one (after a barrier: nobody may still push into it)."""
        if self.backend != "p2p" or self.local is None:
            return
        from . import _lib
        lib = _lib.load()
        torch.cuda.synchronize()
        tdist.barrier(group=_group(self.group))
        for p in self.peers:
            lib.ssp_xchg_close(ctypes.c_void_p(p))
        lib.ssp_xchg_free(ctypes.c_void_p(self.local))
        self.local, self.peers, self.table = None, [], None

    def check(self):
        """Raises if an exchange timed out waiting for a peer (synchronises the current stream)."""
        if self.backend == "p2p" and self.local is not None:
            from . import _lib
            _lib.check(_lib.load().ssp_xchg_status(ctypes.c_void_p(self.local), _lib.stream_of(torch.empty(0, device="cuda"))),
                       "loss exchange")

    # -- the one entry point ----------------------------------------------------------------------
    def run(self, det0=None, det1=None, desc8=None, sem0=None, sem1=None, B_local=0, Hc=1, Wc=1, lambda_loss=1.0, total=None):
        ts = [t for t in (det0, det1, desc8, sem0, sem1) if t is not None]
        if not ts:
            return
        if self.backend == "p2p":
            from . import _lib
            for t in ts:
                if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
                    raise RuntimeError("loss exchange (p2p): the scalars must be contiguous fp32 CUDA tensors")
            _lib.call("ssp_loss_exchange", self.table, self.rank, self.world, _lib.ptr(det0), _lib.ptr(det1), _lib.ptr(desc8),
                      _lib.ptr(sem0), _lib.ptr(sem1), int(B_local), int(Hc), int(Wc), float(lambda_loss), _lib.ptr(total),
                      self.timeout_s, _lib.stream_of(ts[0]))
            return
        # torch.distributed fallback: same payload, same fix-ups, one all-reduce
        with torch.no_grad():
            pay = torch.zeros((_NV,), dtype=torch.float32, device=ts[0].device)
            if det0 is not None:
                pay[0], pay[1] = det0[1], det0[2] - 1e-5
            if det1 is not None:
                pay[2], pay[3] = det1[1], det1[2] - 1e-5
            if desc8 is not None:
                pay[4:8] = desc8[4:8]
            pay[8:9].fill_(float(B_local))  # a fill kernel, not a host-to-device copy: legal inside CUDA graph capture
            if sem0 is not None:
                pay[9:11] = sem0[1:3]
            if sem1 is not None:
                pay[11:13] = sem1[1:3]
            tdist.all_reduce(pay, op=tdist.ReduceOp.SUM, group=_group(self.group))
            for d, i in ((det0, 0), (det1, 2)):
                if d is not None:
                    d[1] = pay[i]
                    d[2] = pay[i + 1] + 1e-5
                    d[0] = d[1] / d[2]
            if desc8 is not None:
                norm = pay[8] * (pay[7] + 1.0) * float(Hc) * float(Wc)
                desc8[3] = norm
                desc8[0:3] = pay[4:7] / norm
                desc8[4:8] = pay[4:8]
            for d, i in ((sem0, 9), (sem1, 11)):
                if d is not None:
                    d[1:3] = pay[i:i + 2]
                    d[0] = pay[i] / pay[i + 1]
            if total is not None:
                total.copy_(((det0[0] + det1[0]) + float(lambda_loss) * desc8[0]).reshape(total.shape))


_exchanges = {}


def get_exchange(group=True):
    """The LossExchange of a process group (created on first use: collective, every rank must call it)."""
    if isinstance(group, LossExchange):
        return group
    key = id(group) if group is not True else None
    ex = _exchanges.get(key)
    if ex is None:
        ex = _exchanges[key] = LossExchange(group)
    return ex


def close_exchanges():
    for ex in list(_exchanges.values()):
        ex.close()
    _exchanges.clear()


def max_over_ranks(value, device):
    """Max of a python float over all ranks (timing is reported as the slowest rank)."""
    if not tdist.is_initialized():
        return value
    t = torch.tensor([value], dtype=torch.float64, device=device)
    tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
    return float(t.item())


# ------------------------------------------------------------------------------------------------
# host placement: bind the process to the CPUs next to its GPU (pinned staging buffers are then allocated on that node)
# ------------------------------------------------------------------------------------------------
def _parse_cpulist(text):
    cpus = []
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.extend(range(int(a), int(b or a) + 1))
    return cpus


def bind_to_gpu_numa_node(device_index):
    """sched_setaffinity to the CPUs of the NUMA node the GPU hangs off (sysfs); returns a dict describing what was done.
    Host->device staging then comes from node-local pinned memory instead of crossing the socket interconnect."""
    info = {"numa_node": None, "cpus": None, "bound": False}
    try:
        props = torch.cuda.get_device_properties(device_index)
        bdf = "%04x:%02x:%02x.0" % (getattr(props, "pci_domain_id", 0), props.pci_bus_id, props.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        info["numa_node"] = node
        if node < 0:
            return info
        cpus = _parse_cpulist(open("/sys/devices/system/node/node%d/cpulist" % node).read())
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
            info.update(cpus=len(allowed), bound=True)
    except Exception as e:  # noqa: BLE001 -- placement is an optimisation, never a reason to fail
        info["error"] = repr(e)
    return info
