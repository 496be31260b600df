"""Host-facing front end of the stage: pinned host buffers in, poses on the host out.

`HostStagePipeline.run(batches)` is the end-to-end call a `demo.py`/`test.py`-style
loop makes once the backbone features and depth maps live in host memory: every
batch is copied host->device on a side stream (double-buffered, so the copy of
batch i+1 overlaps the kernels of batch i), lifted with
`VoxelNetwork_depth.lift`, and its (B,15,3) poses are copied back into pinned buffers that are
reused by later `run` calls (copy the result out if it must outlive the next call).
The FIRST batch of a call has nothing to hide its copy behind (604 MB = 11 ms at PCIe speed for 64 frames), so
it is ramped: copied and lifted as a quarter, a quarter and a half, each part's kernels overlapping the next
part's copy -- only the first quarter's copy stays exposed.
With several ranks (`gather_fn`), every batch's LOCAL poses go to the host as they finish and the poses of all
batches of the call are all-gathered ONCE at the end (frames are independent: there is no per-batch exchange step, and
a per-batch collective would make every step run at the pace of the slowest GPU).
"""
from typing import Iterable, List, Tuple

import torch


class HostStagePipeline:
    def __init__(self, net, gather_fn=None):
        self.net = net
        self.device = torch.device(net.device)
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.slots = [None, None]
        self.ready = [torch.cuda.Event(), torch.cuda.Event()]
        self.done = [torch.cuda.Event(), torch.cuda.Event()]
        self.gather_fn = gather_fn
        self.h2d_bytes = 0
        self.d2h_bytes = 0
        self._host_gathered = None
        self._host_out = []          # pinned result buffers, reused across run() calls (cudaHostAlloc is slow)
        self.ramp_min_batch = 32     # ramp the first batch of a call when it has at least this many frames

    def _stage(self, slot: int, feat: torch.Tensor, depth: torch.Tensor) -> None:
        if not (feat.is_pinned() and depth.is_pinned()):
            raise ValueError("HostStagePipeline needs pinned host tensors")
        if self.slots[slot] is None or self.slots[slot][0].shape != feat.shape or self.slots[slot][1].shape != depth.shape:
            self.slots[slot] = (torch.empty(feat.shape, dtype=torch.float32, device=self.device),
                                torch.empty(depth.shape, dtype=torch.float32, device=self.device))
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.done[slot])          # slot's previous consumer finished
            self.slots[slot][0].copy_(feat, non_blocking=True)
            self.slots[slot][1].copy_(depth, non_blocking=True)
            self.ready[slot].record(self.copy_stream)
        self.h2d_bytes += feat.numel() * 4 + depth.numel() * 4

    def _ramp_parts(self, b: int):
        q = b // 4
        return [(0, q), (q, 2 * q), (2 * q, b)]

    def _stage_ramped(self, slot: int, feat: torch.Tensor, depth: torch.Tensor):
        """Copy the batch in parts; returns [(start, stop, ready_event)]."""
        if not (feat.is_pinned() and depth.is_pinned()):
            raise ValueError("HostStagePipeline needs pinned host tensors")
        if self.slots[slot] is None or self.slots[slot][0].shape != feat.shape or self.slots[slot][1].shape != depth.shape:
            self.slots[slot] = (torch.empty(feat.shape, dtype=torch.float32, device=self.device),
                                torch.empty(depth.shape, dtype=torch.float32, device=self.device))
        parts = []
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.done[slot])
            for s0, s1 in self._ramp_parts(feat.shape[0]):
                self.slots[slot][0][s0:s1].copy_(feat[s0:s1], non_blocking=True)
                self.slots[slot][1][s0:s1].copy_(depth[s0:s1], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self.copy_stream)
                parts.append((s0, s1, ev))
            self.ready[slot].record(self.copy_stream)
        self.h2d_bytes += feat.numel() * 4 + depth.numel() * 4
        return parts

    def run(self, batches: Iterable[Tuple]) -> List[torch.Tensor]:
        """batches: (feat, depth) pinned host tensors, or (feat, depth, camera_ids) with the host-side camera ids
        `lift` takes (a camera per frame)."""
        batches = list(batches)
        cam_ids = [b[2] if len(b) > 2 else None for b in batches]
        batches = [b[:2] for b in batches]
        out = []
        main = torch.cuda.current_stream(self.device)
        # pinned result buffers for every batch of this call BEFORE any GPU work is queued: cudaHostAlloc
        # synchronises the device, so allocating them one by one inside the loop drained the pipeline at every
        # new batch index (a 20-batch call after a 2-batch warm-up ran at a third of the speed)
        kp_shape = (batches[0][0].shape[0], self.net.num_joints, 3) if batches else None
        while kp_shape is not None and len(self._host_out) < len(batches):
            self._host_out.append(torch.empty(kp_shape, dtype=torch.float32, pin_memory=True))
        ramp = None
        local_kps = []
        if batches:
            if batches[0][0].shape[0] >= self.ramp_min_batch:
                ramp = self._stage_ramped(0, *batches[0])
            else:
                self._stage(0, *batches[0])
        for i in range(len(batches)):
            slot = i & 1
            if i + 1 < len(batches):
                self._stage(slot ^ 1, *batches[i + 1])
            feat, depth = self.slots[slot]
            with torch.no_grad():
                if i == 0 and ramp is not None:
                    kps = []
                    for s0, s1, ev in ramp:
                        main.wait_event(ev)
                        ids = None if cam_ids[0] is None else cam_ids[0][s0:s1]
                        kps.append(self.net.lift(feat[s0:s1], self.net.grid_coord_proj_batch, self.net.coord_volumes,
                                                 depth_map_batch=depth[s0:s1], camera_ids=ids)[0])
                    kp = torch.cat(kps)
                else:
                    main.wait_event(self.ready[slot])
                    kp = self.net.lift(feat, self.net.grid_coord_proj_batch, self.net.coord_volumes,
                                       depth_map_batch=depth, camera_ids=cam_ids[i])[0]
            self.done[slot].record(main)
            if self.gather_fn is not None:
                local_kps.append(kp)
            if i >= len(self._host_out) or self._host_out[i].shape != kp.shape:
                buf = torch.empty(kp.shape, dtype=kp.dtype, pin_memory=True)
                if i < len(self._host_out):
                    self._host_out[i] = buf
                else:
                    self._host_out.append(buf)
            host = self._host_out[i]
            host.copy_(kp, non_blocking=True)
            self.d2h_bytes += kp.numel() * 4
            out.append(host)
        if self.gather_fn is not None and local_kps:
            # ONE collective per call: (B_local, n_batches, J, 3) -> (B_total, n_batches, J, 3) in frame order
            if len({tuple(k.shape) for k in local_kps}) != 1:
                raise ValueError("HostStagePipeline with gather_fn needs equally sized batches")
            allkp = self.gather_fn(torch.stack(local_kps, dim=1).contiguous())
            if self._host_gathered is None or self._host_gathered.shape != allkp.shape:
                self._host_gathered = torch.empty(allkp.shape, dtype=allkp.dtype, pin_memory=True)
            self._host_gathered.copy_(allkp, non_blocking=True)
            self.d2h_bytes += allkp.numel() * 4
            main.synchronize()
            return [self._host_gathered[:, i] for i in range(len(batches))]
        main.synchronize()
        return out
