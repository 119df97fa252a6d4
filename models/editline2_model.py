"""EditLine2Model, inference subset (reference models/editline2_model.py:49-147, 184-242, 338-370).

``forward(data, mode)`` with mode 'inference' returns ``(composed_image, mask)`` exactly like the
reference: netM predicts the edit mask from (image, sketch), the mask is binarised at 0.5, netG inpaints,
and the result is blended with the SOFT mask. All of it is one C-ABI call (``se_forward_inference``) on the
B200 kernels. Mode 'inpaint' takes the region to edit from ``data['region']`` instead of netM and returns
``(composed_image, region)`` (one ``se_forward_inpaint`` call). In both, tensors in ``data`` may live on the CPU
(they are copied to the GPU like the reference's ``preprocess_input`` does) and the outputs are CUDA tensors. Training modes are out of scope."""
import torch

import models.networks as networks
import util.util as util


class EditLine2Model(torch.nn.Module):
    @staticmethod
    def modify_commandline_options(parser, is_train):
        networks.modify_commandline_options(parser, is_train)
        parser.add_argument("--precision", default="bf16", choices=("bf16", "fp32", "fp32_direct"),
                            help="B200 arithmetic: bf16 tensor-core path, fp32-parity arithmetic on the tensor cores (split-half fp16), "
                                 "or its fp32 CUDA-core cross-check")
        return parser

    def __init__(self, opt):
        super().__init__()
        self.opt = opt
        if getattr(opt, "isTrain", False):
            raise NotImplementedError("only the inference path is implemented on B200")
        self.precision = getattr(opt, "precision", "bf16")
        self.netM, self.netG, self.netD = self.initialize_networks(opt)
        self._engine = None
        self._engine_key = None

    def use_gpu(self):
        return len(self.opt.gpu_ids) > 0

    def initialize_networks(self, opt):
        netG = networks.define_G(opt)
        saved = opt.netG
        opt.netG = "MD"
        netM = networks.define_G(opt)
        opt.netG = saved
        if not hasattr(opt, "isSkip"):           # same escape hatch as the reference (:195)
            netG = util.load_network(netG, "G", opt.which_epoch, opt)
            netM = util.load_network(netM, "M", opt.which_epoch, opt)
        return netM, netG, None

    def engine(self):
        from sketchedit_b200.engine import Engine
        key = self.netM._weights_key() + self.netG._weights_key()
        if self._engine is None or key != self._engine_key:
            eng = Engine()
            eng.load_state_dict("M", self.netM.state_dict())
            eng.load_state_dict("G", self.netG.state_dict())
            self.netG._configure_engine(eng)
            eng.finalize()
            self._engine, self._engine_key = eng, key
        return self._engine

    def preprocess_input(self, data):
        dev = torch.device("cuda")
        image = data["image"].to(dev, torch.float32, non_blocking=True)
        line = data["mask"].to(dev, torch.float32, non_blocking=True)
        return image, line

    def forward(self, data, mode, is_real_im=True):
        region = data["region"] if mode == "inpaint" else None
        image, line = self.preprocess_input(data)
        if mode == "inference":
            composed, mask, _ = self.engine().inference(image, line, precision=self.precision)
            return composed, mask
        if mode == "visualize":
            # reference :134-145 -- 'mask' is the BINARISED mask netG inpaints (mask_inpaint), 'composed' is blended
            # with the SOFT mask exactly like mode='inference'
            composed, _, ex = self.engine().inference(image, line, precision=self.precision,
                                                      want=("coarse", "fine", "mask_image", "mask_bin"))
            return {"mask": ex["mask_bin"], "maskim": ex["mask_image"], "coarse": ex["coarse"], "fine": ex["fine"],
                    "composed": composed}
        if mode == "inpaint":
            # the user chooses the region (data['region'] [B,1,H,W], 1 = edit here) instead of netM: the external-mask branch of the
            # reference's generate_fake (:340-352, 362-368) composed like :114. Returns (composed, region) like 'inference' does.
            region = region.to(image.device, torch.float32, non_blocking=True)
            composed, _ = self.engine().inpaint(image, line, region, precision=self.precision)
            return composed, region
        raise ValueError("|mode| is invalid or training-only: %r" % (mode,))

    def inference_stream(self, loader, depth=2, pinned_ring=True, gather=None, uint8=False, with_data=False):
        """Pipelined form of ``for data in loader: model(data, mode='inference')`` for throughput serving.

        Yields ``(composed, mask)`` per batch, in order, as PINNED CPU tensors (views of one packed [B,4,H,W] host
        buffer). The host->device copy of batch i+1 and the device->host copy of batch i-1 run on their own CUDA
        streams while batch i computes (``depth`` device buffers per tensor), so a step costs max(copy, compute)
        instead of their sum. Batches whose input tensors are in pinned memory (DataLoader(pin_memory=True)) overlap fully.

        uint8=True: the reference's host-side codecs run on the device (``Engine.inference_u8``): a batch supplies
        ``data['image_u8']`` [B,H,W,3] RGB uint8 and ``data['mask_u8']`` [B,H,W] uint8 (what the dataset holds before
        ToTensor/Normalize, reference data/testimage_dataset.py:89-103) and the results are ``(bgr_u8 [B,H,W,3], mask_u8
        [B,H,W])`` exactly as test.py:25-35 writes them: 4x fewer bytes over PCIe in each direction.

        with_data=True: yield ``(out0, out1, data)`` (test.py needs the batch's output paths).

        pinned_ring=True (default): results are views of a ring of ``depth + 2`` pinned buffers handed out round robin. The
        copy of batch i + depth - 1 is already in flight when result i is drawn, so a result stays intact while at most
        ``depth`` further results are drawn (you may hold the newest ``depth + 1``; consume or ``.clone()`` older ones);
        pinned_ring=False allocates fresh pinned tensors for every batch (a cudaHostAlloc per batch when the host
        allocator cannot recycle, which costs more than the copy itself).

        gather: a ``sketchedit_b200.parallel.OutputGather`` (data-parallel serving, one process per GPU; float mode): every
        batch's packed outputs are written into this rank's slice of the gather buffer and all-gathered over NCCL (async, in
        place) before this rank's shard is copied to the host; all ranks must feed equal batch sizes."""
        import collections
        eng = self.engine()
        if gather is not None and (gather.depth != depth or uint8):
            raise ValueError("gather= needs float mode and a ring depth equal to the stream depth (%d)" % depth)
        dev = torch.device("cuda")
        cur = torch.cuda.current_stream()
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
        slots = [None] * depth
        pending = collections.deque()
        ring = {}        # (B, H, W) -> [buffers, results handed out so far]

        def new_host(B, H, W):
            if uint8:
                return (torch.empty(B, H, W, 3, dtype=torch.uint8, pin_memory=True), torch.empty(B, H, W, dtype=torch.uint8, pin_memory=True))
            packed = torch.empty(B, 4, H, W, pin_memory=True)
            return (packed,)

        def host_out(B, H, W):
            if not pinned_ring:
                return new_host(B, H, W)
            entry = ring.setdefault((B, H, W), [[], 0])
            bufs, count = entry
            if len(bufs) < depth + 2:
                bufs.append(new_host(B, H, W))
            entry[1] = count + 1
            return bufs[count % (depth + 2)]       # strict round robin per shape: 0, 1, .., depth+1, 0, 1, ..

        def drain_one():
            host, ev, data = pending.popleft()
            ev.synchronize()
            res = (host[0], host[1]) if uint8 else (host[0][:, :3], host[0][:, 3:4])
            return res + (data,) if with_data else res

        in_keys = ("image_u8", "mask_u8") if uint8 else ("image", "mask")
        for i, data in enumerate(loader):
            img_h, line_h = data[in_keys[0]], data[in_keys[1]]
            B, H, W = (img_h.shape[0], img_h.shape[1], img_h.shape[2]) if uint8 else (img_h.shape[0], img_h.shape[2], img_h.shape[3])
            slot = slots[i % depth]
            if slot is None or slot["shape"] != (B, H, W):
                if slot is not None:   # shape change (ragged last batch): let the old buffers' users finish first
                    slot["ev_comp"].synchronize()
                    slot["ev_out"].synchronize()
                if uint8:
                    u8 = lambda *shape: torch.empty(*shape, device=dev, dtype=torch.uint8)
                    bufs = {"img": u8(B, H, W, 3), "line": u8(B, H, W), "out": (u8(B, H, W, 3), u8(B, H, W))}
                else:
                    f32 = lambda c: torch.empty(B, c, H, W, device=dev, dtype=torch.float32)
                    bufs = {"img": f32(3), "line": f32(1), "out": None if gather is not None else (f32(4),)}
                slot = dict(bufs, shape=(B, H, W), ev_in=torch.cuda.Event(), ev_comp=torch.cuda.Event(), ev_out=torch.cuda.Event())
                slots[i % depth] = slot
            s_in.wait_event(slot["ev_comp"])           # the previous user of these input buffers has been computed
            with torch.cuda.stream(s_in):
                slot["img"].copy_(img_h, non_blocking=True)
                slot["line"].copy_(line_h, non_blocking=True)
                slot["ev_in"].record(s_in)
            cur.wait_event(slot["ev_in"])
            cur.wait_event(slot["ev_out"])             # ... and its outputs have left the device buffers
            if gather is not None:
                if (B, H, W) != (gather.B,) + tuple(gather.bufs[0].shape[2:]):
                    raise ValueError("with gather= every batch must be [%d,*,%d,%d]" % ((gather.B,) + tuple(gather.bufs[0].shape[2:])))
                out = gather.next_slot()               # (waits, on `cur`, for the collective that last used this buffer)
                eng.inference_packed(slot["img"], slot["line"], precision=self.precision, out=out)
                k = gather.launch()
                slot["ev_comp"].record(cur)            # inputs are free again; the outputs follow the collective:
                with torch.cuda.stream(s_out):
                    gather.wait(k)                     # s_out waits for the all-gather of this batch
                    src = (gather.bufs[k][gather.rank * B:(gather.rank + 1) * B],)
            else:
                if uint8:
                    eng.inference_u8(slot["img"], slot["line"], precision=self.precision, out=slot["out"])
                else:
                    eng.inference_packed(slot["img"], slot["line"], precision=self.precision, out=slot["out"][0])
                slot["ev_comp"].record(cur)
                s_out.wait_event(slot["ev_comp"])
                src = slot["out"]
            with torch.cuda.stream(s_out):
                host = host_out(B, H, W)
                for h_t, d_t in zip(host, src):
                    h_t.copy_(d_t, non_blocking=True)
                slot["ev_out"].record(s_out)
                done = torch.cuda.Event()
                done.record(s_out)
            pending.append((host, done, data))
            if len(pending) >= depth:
                yield drain_one()
        while pending:
            yield drain_one()
