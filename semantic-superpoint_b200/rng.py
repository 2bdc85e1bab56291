"""Seed and launch-counter state shared by the device samplers (sparse.DeviceSampler, homography.HomographySampler)."""
import torch


class DeviceRng(object):
    """Philox4x32-10 state in a device int64 tensor [4]: {seed, launch counter, blocks done (0 between launches), a count the
    sampler may keep}, as uint64 bits.  Every launch reads the counter and advances it on the device, so eager calls and CUDA
    graph replays draw fresh numbers with no host involvement, and get_state() / set_state() reproduce a sequence bit for bit.
    Launches that share one state buffer must be ordered on one stream."""

    def __init__(self, seed=0, device="cuda"):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("%s samples on a CUDA device, got %s" % (type(self).__name__, self.device))
        seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        seed = seed - (1 << 64) if seed >= (1 << 63) else seed
        self.state = torch.tensor([seed, 0, 0, 0], dtype=torch.int64).to(self.device)

    def get_state(self):
        """{seed, launch counter} as a device int64 tensor [2] (a copy)."""
        return self.state[:2].clone()

    def set_state(self, state):
        self.state[:2].copy_(torch.as_tensor(state, dtype=torch.int64))
