"""Inference engine: the public call a user makes to get depth maps out of host images.

``DepthEngine`` owns static device buffers for one input shape, captures the whole
``PatchmatchNet.forward`` (cuDNN feature pyramid, the native PatchMatch kernels, refinement) into ONE
CUDA graph per slot -- the cascade is ~120 short kernels, so at 640x512 launch latency, not bandwidth,
is the enemy (SURVEY.md 7.3-1) -- runs independent requests concurrently on per-slot streams (most
kernels of one request launch fewer CTAs than the 148 SMs hold) and moves data with pinned-memory
async copies on a copy stream so uploads overlap compute.

    eng = DepthEngine(net, batch=1, n_views=5, height=512, width=640, device="cuda:0")
    depth, confidence = eng.infer(images, intrinsics, extrinsics, depth_min, depth_max)   # host in, host out

There is no CPU path: construction fails without CUDA.
"""
from __future__ import annotations

from typing import Dict, List, Sequence, Tuple

import torch

Tensor = torch.Tensor


class DepthEngine:
    def __init__(
        self,
        net: torch.nn.Module,
        batch: int,
        n_views: int,
        height: int,
        width: int,
        device: str = "cuda:0",
        use_graph: bool = True,
        warmup: int = 3,
        n_slots: int = 3,
    ) -> None:
        if not torch.cuda.is_available():
            raise RuntimeError("DepthEngine needs a CUDA device (B200); there is no CPU fallback")
        self.device = torch.device(device)
        self.net = net.eval().to(self.device)
        self.shape = (batch, n_views, height, width)
        B, N, H, W = self.shape
        dev = self.device
        # One slot = static device inputs + its own compute stream + its own captured graph + pinned host outputs.
        # Several slots let independent requests overlap on the GPU: most kernels of a 640x512 forward launch far
        # fewer CTAs than 148 SMs hold, so one request alone cannot fill the machine.
        self.n_slots = max(1, int(n_slots))
        self._slots = []
        for _ in range(self.n_slots):
            slot = self._input_block(dev)
            slot.update(
                stream=torch.cuda.Stream(device=dev),
                host_depth=torch.empty(B, 1, H, W).pin_memory(),
                host_conf=torch.empty(B, H, W).pin_memory(),
                graph=None,
                outs=None,
            )
            self._slots.append(slot)
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.compute_stream = self._slots[0]["stream"]
        self.use_graph = use_graph
        self._warmup = warmup
        self._ready = False

    def _input_block(self, dev, pinned_pack: bool = False) -> Dict[str, Tensor]:
        """Device tensors for one request's inputs.  The cameras and the depth range live in ONE flat `params` buffer (the
        named entries are views into it): a request's small inputs then move with one copy instead of four -- the serving
        loop is a few dozen driver calls per request, and at > 1000 requests/s those calls, not the bytes, are the budget."""
        B, N, H, W = self.shape
        n_i, n_e = B * N * 9, B * N * 16
        params = torch.zeros(n_i + n_e + 2 * B, device=dev)
        params[n_i + n_e:n_i + n_e + B] = 1.0
        params[n_i + n_e + B:] = 2.0
        blk = dict(
            images=torch.zeros(N, B, 3, H, W, device=dev),
            params=params,
            intrinsics=params[:n_i].view(B, N, 3, 3),
            extrinsics=params[n_i:n_i + n_e].view(B, N, 4, 4),
            depth_min=params[n_i + n_e:n_i + n_e + B],
            depth_max=params[n_i + n_e + B:],
        )
        if pinned_pack:
            blk["host_params"] = torch.zeros(params.numel()).pin_memory()
        return blk

    def _pack_params(self, host_pack: Tensor, req: Dict[str, object]) -> int:
        """Write a request's cameras and depth range into the pinned pack (plain host copies); returns the bytes."""
        B, N, _, _ = self.shape
        n_i, n_e = B * N * 9, B * N * 16
        host_pack[:n_i].copy_(req["intrinsics"].reshape(-1))
        host_pack[n_i:n_i + n_e].copy_(req["extrinsics"].reshape(-1))
        host_pack[n_i + n_e:n_i + n_e + B].copy_(req["depth_min"].reshape(-1))
        host_pack[n_i + n_e + B:].copy_(req["depth_max"].reshape(-1))
        return 4 * host_pack.numel()

    # ------------------------------------------------------------------
    def _forward(self, slot: Dict[str, Tensor]) -> Tuple[Tensor, Tensor]:
        imgs = [slot["images"][i] for i in range(self.shape[1])]
        depth, conf, _ = self.net(imgs, slot["intrinsics"].clone(), slot["extrinsics"], slot["depth_min"], slot["depth_max"])
        return depth, conf

    def set_device_inputs(self, slot_idx: int, images, intrinsics, extrinsics, depth_min, depth_max) -> None:
        """Fill a slot from tensors that already live on the device (kernel-only timing path)."""
        s = self._slots[slot_idx]
        for i, im in enumerate(images):
            s["images"][i].copy_(im)
        s["intrinsics"].copy_(intrinsics)
        s["extrinsics"].copy_(extrinsics)
        s["depth_min"].copy_(depth_min.reshape(-1))
        s["depth_max"].copy_(depth_max.reshape(-1))

    def prepare(self) -> None:
        """Warm up (cuDNN autotune, allocator, BatchNorm/head folding) and capture one graph per slot.
        Slots must hold valid cameras."""
        with torch.no_grad(), torch.cuda.device(self.device):
            for slot in self._slots:
                with torch.cuda.stream(slot["stream"]):
                    for _ in range(self._warmup):
                        self._forward(slot)
                slot["stream"].synchronize()
            if self.use_graph:
                for slot in self._slots:
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=slot["stream"]):
                        slot["outs"] = self._forward(slot)
                    slot["graph"] = g
        torch.cuda.synchronize(self.device)
        self._ready = True

    def run_slot(self, slot_idx: int) -> Tuple[Tensor, Tensor]:
        """One forward on the inputs currently in the slot, enqueued on the CURRENT stream."""
        if not self._ready:
            self.prepare()
        slot = self._slots[slot_idx]
        if self.use_graph:
            slot["graph"].replay()
            return slot["outs"]
        with torch.no_grad():
            return self._forward(slot)

    def run_round(self, n: int, start: torch.cuda.Event, done: torch.cuda.Event) -> List[Tuple[Tensor, Tensor]]:
        """`n` (<= n_slots) forwards concurrently, one per slot stream, fenced by `start` (already recorded on the
        current stream) and `done` (recorded on the current stream once every slot has finished).  Returns each
        forward's (depth, confidence), valid once `done` has completed."""
        cur = torch.cuda.current_stream(self.device)
        outs = []
        for i in range(n):
            st = self._slots[i]["stream"]
            st.wait_event(start)
            with torch.cuda.stream(st):
                outs.append(self.run_slot(i))
            cur.wait_stream(st)
        done.record(cur)
        return outs

    # ------------------------------------------------------------------
    def upload(self, slot_idx: int, host: Dict[str, object], stream: torch.cuda.Stream) -> int:
        """Async pinned-host -> device copy of one request; returns the bytes moved."""
        s = self._slots[slot_idx]
        n = 0
        with torch.cuda.stream(stream):
            for i, im in enumerate(host["images"]):
                s["images"][i].copy_(im, non_blocking=True)
                n += im.numel() * im.element_size()
            for k in ("intrinsics", "extrinsics", "depth_min", "depth_max"):
                src = host[k]
                s[k].copy_(src.reshape(s[k].shape), non_blocking=True)
                n += src.numel() * src.element_size()
        return n

    def _first_use(self, host: Dict[str, object]) -> None:
        for i in range(self.n_slots):
            self.upload(i, host, self._slots[i]["stream"])
            self._slots[i]["stream"].synchronize()
        self.prepare()

    def infer(self, images: Sequence[Tensor], intrinsics: Tensor, extrinsics: Tensor, depth_min: Tensor, depth_max: Tensor):
        """Host tensors in, host (pinned) tensors out; one request, synchronous."""
        host = dict(images=list(images), intrinsics=intrinsics, extrinsics=extrinsics,
                    depth_min=depth_min.float(), depth_max=depth_max.float())
        if not self._ready:
            self._first_use(host)
        slot = self._slots[0]
        with torch.cuda.device(self.device), torch.cuda.stream(slot["stream"]):
            self.upload(0, host, slot["stream"])
            depth, conf = self.run_slot(0)
            slot["host_depth"].copy_(depth, non_blocking=True)
            slot["host_conf"].copy_(conf, non_blocking=True)
        slot["stream"].synchronize()
        return slot["host_depth"], slot["host_conf"]

    def _staging(self):
        """Device staging buffers for uploads (2 per slot): the PCIe copy of a request overlaps the compute of the
        slot's previous request, then a device-to-device copy (20 MB at HBM speed) moves it into the slot's
        graph-captured input buffers.  Each carries a pinned host pack for the request's small inputs and the events
        the loop re-records (no per-request event construction)."""
        if getattr(self, "_stage", None) is None:
            self._stage = []
            for _ in range(2 * self.n_slots):
                blk = self._input_block(self.device, pinned_pack=True)
                blk["uploaded"] = torch.cuda.Event()
                blk["free"] = torch.cuda.Event()
                blk["used"] = False
                self._stage.append(blk)
            for slot in self._slots:
                slot["drained"] = torch.cuda.Event()
        return self._stage

    def infer_stream(self, requests: Sequence[Dict[str, object]], on_result=None) -> Tuple[int, int]:
        """Pipelined serving loop over pinned-host requests.  Request i is uploaded (copy stream) into a staging
        buffer while earlier requests compute, then slot i % n_slots copies it into its static inputs, replays its
        CUDA graph on its own stream and reads the results back to the slot's pinned host buffers.  Every request
        pays its host->device and device->host copies.  Returns (h2d_bytes, d2h_bytes) per request.
        Driver calls per request: one image upload when the request's views are adjacent slices of one pinned buffer (else one
        per view), one upload of the packed cameras + depth range, two device-to-device copies, the graph launch, two result
        downloads, three event records."""
        from .net import _adjacent_views

        if not self._ready:
            self._first_use(requests[0])
        S = self.n_slots
        stage = self._staging()
        NS = len(stage)
        h2d = d2h = 0
        used = [False] * S  # slot has a result in flight from this call
        for buf in stage:
            buf["used"] = False
        with torch.cuda.device(self.device):
            for i, req in enumerate(requests):
                k, j = i % S, i % NS
                slot, buf = self._slots[k], stage[j]
                if buf["used"]:
                    self.copy_stream.wait_event(buf["free"])  # the slot that consumed this staging buffer has copied it out
                    buf["uploaded"].synchronize()             # ... and its pinned pack has long been read by the copy engine
                h2d = self._pack_params(buf["host_params"], req)
                images = req["images"]
                with torch.cuda.stream(self.copy_stream):
                    first = images[0]
                    if len(images) == buf["images"].shape[0] and _adjacent_views(images):
                        stacked = torch.as_strided(first, (len(images),) + tuple(first.shape), (first.numel(),) + tuple(first.stride()))
                        buf["images"].copy_(stacked, non_blocking=True)
                        h2d += stacked.numel() * stacked.element_size()
                    else:
                        for v, im in enumerate(images):
                            buf["images"][v].copy_(im, non_blocking=True)
                            h2d += im.numel() * im.element_size()
                    buf["params"].copy_(buf["host_params"], non_blocking=True)
                    buf["uploaded"].record(self.copy_stream)
                buf["used"] = True
                if on_result is not None and used[k]:
                    slot["drained"].synchronize()  # hand the slot's previous result to the caller before it is overwritten
                    on_result(i - S, slot["host_depth"], slot["host_conf"])
                st = slot["stream"]
                with torch.cuda.stream(st):
                    st.wait_event(buf["uploaded"])
                    slot["images"].copy_(buf["images"], non_blocking=True)
                    slot["params"].copy_(buf["params"], non_blocking=True)
                    buf["free"].record(st)
                    depth, conf = self.run_slot(k)
                    slot["host_depth"].copy_(depth, non_blocking=True)
                    slot["host_conf"].copy_(conf, non_blocking=True)
                    d2h = depth.numel() * 4 + conf.numel() * 4
                    slot["drained"].record(st)
                    used[k] = True
            for k in range(S):
                self._slots[k]["stream"].synchronize()
            if on_result is not None:
                for i in range(max(0, len(requests) - S), len(requests)):
                    k = i % S
                    on_result(i, self._slots[k]["host_depth"], self._slots[k]["host_conf"])
        return h2d, d2h
