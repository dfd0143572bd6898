"""Engine: one fvhd handle + the torch-owned device memory it borrows (weights blob, workspace)."""
import ctypes as C

import torch

from . import lib as L

_DT = {torch.float32: L.F32, torch.float16: L.F16, torch.bfloat16: L.BF16}


def _img_dtype(t):
    if t.dtype not in _DT:
        raise L.FvhdError(f"images must be fp32/fp16/bf16, got {t.dtype}")
    return _DT[t.dtype]


class Engine:
    """Plan for one image size R (+ optional projector of hidden size H).

    Host plumbing only: PyTorch owns every buffer (packed weights, workspace, inputs, outputs) and
    supplies the current CUDA stream; all compute is in libfastvithd_b200.so.
    """

    def __init__(self, image_size, projector_hidden=0, projector_depth=2, max_batch=8):
        self.lib = L.load_library()
        self.cfg = L.FvhdConfig(int(image_size), int(projector_hidden), int(projector_depth), int(max_batch))
        self.handle = C.c_void_p()
        L.check(self.lib.fvhd_create(C.byref(self.cfg), C.byref(self.handle)), None)
        self.image_size = int(image_size)
        self.hidden = int(projector_hidden)
        self.max_batch = int(max_batch)
        self.num_tokens = self.lib.fvhd_num_tokens(self.handle)
        self.out_dim = self.lib.fvhd_out_dim(self.handle)
        self._weights = None       # keeps the device blob alive
        self._workspace = None
        self.device = None

    def __del__(self):
        try:
            if getattr(self, "handle", None) and self.handle.value:
                self.lib.fvhd_destroy(self.handle)
                self.handle = C.c_void_p()
        except Exception:
            pass

    # ------------------------------------------------------------------ introspection (no GPU needed)
    def weight_specs(self):
        out = []
        name, dt, n = C.c_char_p(), C.c_int(), C.c_int64()
        for i in range(self.lib.fvhd_num_weights(self.handle)):
            L.check(self.lib.fvhd_weight_spec(self.handle, i, C.byref(name), C.byref(dt), C.byref(n)), self.handle)
            out.append((name.value.decode(), dt.value, n.value))
        return out

    def units(self):
        out = []
        name = C.c_char_p()
        ie, oe = C.c_int64(), C.c_int64()
        oh, ow, oc = C.c_int(), C.c_int(), C.c_int()
        fl, mb = C.c_double(), C.c_double()
        for u in range(self.lib.fvhd_num_units(self.handle)):
            L.check(self.lib.fvhd_unit_info(self.handle, u, C.byref(name), C.byref(ie), C.byref(oe), C.byref(oh), C.byref(ow),
                                            C.byref(oc), C.byref(fl), C.byref(mb)), self.handle)
            out.append(dict(index=u, name=name.value.decode(), in_elems=ie.value, out_elems=oe.value, out_h=oh.value,
                            out_w=ow.value, out_c=oc.value, flops=fl.value, min_bytes=mb.value))
        return out

    def workspace_bytes(self, batch=None):
        return int(self.lib.fvhd_workspace_bytes(self.handle, int(batch or self.max_batch)))

    def launches_per_forward(self, batch=1):
        return int(self.lib.fvhd_launches_per_forward(self.handle, int(batch)))

    # ------------------------------------------------------------------ weights / workspace
    def load(self, packed, device):
        """`packed`: name -> CPU/GPU tensor from packer.pack_tower (+ pack_projector).  One H2D blob."""
        device = torch.device(device)
        if device.type != "cuda":
            raise L.FvhdError(f"libfastvithd_b200 computes on CUDA devices only (got {device}); there is no CPU path")
        if device.index is None:                       # 'cuda' -> the concrete current device, so tensor.device compares equal
            device = torch.device("cuda", torch.cuda.current_device())
        specs = self.weight_specs()
        offs, total = {}, 0
        for name, dt, numel in specs:
            if name not in packed:
                raise L.FvhdError(f"packed weights lack '{name}'")
            t = packed[name]
            want = {L.F32: torch.float32, L.F16: torch.float16, L.BF16: torch.bfloat16}[dt]
            if t.dtype != want or t.numel() != numel:
                raise L.FvhdError(f"packed '{name}': want {want} x {numel}, got {t.dtype} x {t.numel()}")
            offs[name] = total
            total += (t.numel() * t.element_size() + 255) // 256 * 256
        blob = torch.empty(total, dtype=torch.uint8, pin_memory=False)
        for name, dt, numel in specs:
            t = packed[name].detach().contiguous().cpu()
            nb = t.numel() * t.element_size()
            blob[offs[name]: offs[name] + nb] = t.view(-1).view(torch.uint8)
        with torch.cuda.device(device):
            dblob = blob.to(device)
            base = dblob.data_ptr()
            table = (L.FvhdTensor * len(specs))()
            keep = []
            for i, (name, dt, numel) in enumerate(specs):
                bname = name.encode()
                keep.append(bname)
                table[i] = L.FvhdTensor(bname, base + offs[name], dt, numel)
            L.check(self.lib.fvhd_load_weights(self.handle, table, len(specs)), self.handle)
            self._weights = dblob
            self.device = device
            ws = self.workspace_bytes()
            self._workspace = torch.empty(ws, dtype=torch.uint8, device=device)
            L.check(self.lib.fvhd_set_workspace(self.handle, self._workspace.data_ptr(), ws), self.handle)
        return self

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------ compute
    def _check_images(self, images, device):
        """Shape / dtype / placement of an image batch before its raw pointer goes to the C library; returns it contiguous."""
        if self.device is None:
            raise L.FvhdError("Engine.load() has not been called")
        if not torch.is_tensor(images) or images.dim() != 4 or images.shape[0] < 1 or images.shape[1] != 3 \
                or images.shape[2] != self.image_size or images.shape[3] != self.image_size:
            raise L.FvhdError(f"images must be [B>=1,3,{self.image_size},{self.image_size}], got {tuple(getattr(images, 'shape', ()))}")
        _img_dtype(images)
        if images.device != device:
            raise L.FvhdError(f"images on {images.device}, expected {device}")
        return images.contiguous()

    def _check_out(self, t, shape, what):
        if not torch.is_tensor(t) or t.dtype != torch.bfloat16 or tuple(t.shape) != tuple(shape) or not t.is_contiguous():
            raise L.FvhdError(f"{what} must be a contiguous bf16 tensor of shape {tuple(shape)}, got "
                              f"{getattr(t, 'dtype', None)} {tuple(getattr(t, 'shape', ()))}")

    def forward(self, images, want_tokens=True, want_projected=None):
        """images: CUDA tensor [B,3,R,R] (fp32/fp16/bf16) -> (tokens [B,N,3072] bf16 | None, projected [B,N,H] bf16 | None)."""
        if want_projected is None:
            want_projected = self.hidden > 0
        images = self._check_images(images, self.device)
        B = images.shape[0]
        with torch.cuda.device(self.device):
            tokens = torch.empty(B, self.num_tokens, 3072, dtype=torch.bfloat16, device=self.device) if want_tokens else None
            proj = torch.empty(B, self.num_tokens, self.hidden, dtype=torch.bfloat16, device=self.device) if want_projected else None
            L.check(self.lib.fvhd_forward(self.handle, self._stream(), images.data_ptr(), _img_dtype(images), B,
                                          tokens.data_ptr() if tokens is not None else None,
                                          proj.data_ptr() if proj is not None else None), self.handle)
        return tokens, proj

    def forward_into(self, images, embeds, position):
        """Write the projected visual tokens of image b straight into embeds[b, position:position+N, :]
        (embeds: [B, L, H] bf16 CUDA, contiguous).  The splice of llava_arch.py:251-271 as the projector's store."""
        if self.hidden <= 0:
            raise L.FvhdError("forward_into needs a plan with a projector")
        if embeds.dtype != torch.bfloat16 or not embeds.is_contiguous() or embeds.dim() != 3 or embeds.shape[2] != self.hidden:
            raise L.FvhdError(f"embeds must be contiguous bf16 [B, L, {self.hidden}], got {embeds.dtype} {tuple(embeds.shape)}")
        images = self._check_images(images, self.device)
        if embeds.device != self.device:
            raise L.FvhdError(f"embeds on {embeds.device}, engine on {self.device}")
        B, Lseq = embeds.shape[0], embeds.shape[1]
        if images.shape[0] != B or position < 0 or position + self.num_tokens > Lseq:
            raise L.FvhdError(f"cannot place {self.num_tokens} tokens at {position} in a sequence of {Lseq} (batch {images.shape[0]} vs {B})")
        with torch.cuda.device(self.device):
            dst = embeds.data_ptr() + position * self.hidden * 2
            L.check(self.lib.fvhd_forward_strided(self.handle, self._stream(), images.data_ptr(), _img_dtype(images), B, None, dst,
                                                  Lseq * self.hidden), self.handle)
        return embeds

    def encode_images_host(self, host_images, host_out=None):
        """HOST tensors in, HOST tensor out (bf16): the e2e entry (H2D + forward + D2H inside the call)."""
        host_images = self._check_images(host_images, torch.device("cpu"))
        B = host_images.shape[0]
        if host_out is None:
            host_out = torch.empty(B, self.num_tokens, self.out_dim, dtype=torch.bfloat16, pin_memory=True)
        if host_out.device.type != "cpu":
            raise L.FvhdError(f"host_out must be a CPU tensor, got {host_out.device}")
        self._check_out(host_out, (B, self.num_tokens, self.out_dim), "host_out")
        with torch.cuda.device(self.device):
            L.check(self.lib.fvhd_encode_images_host(self.handle, self._stream(), host_images.data_ptr(), _img_dtype(host_images), B,
                                                     host_out.data_ptr()), self.handle)
        return host_out

    def forward_scatter(self, images, dst_ptrs):
        """encode_images with image i's projected [N, H] block stored at device address dst_ptrs[i] (ints; dense rows): the
        general multi-<image> / ragged splice (llava_arch.py:233-271) as the projector's store.  The caller guarantees every
        destination is a writable bf16 region of N*H elements on this device."""
        if self.hidden <= 0:
            raise L.FvhdError("forward_scatter needs a plan with a projector")
        images = self._check_images(images, self.device)
        B = images.shape[0]
        if len(dst_ptrs) != B:
            raise L.FvhdError(f"{B} images but {len(dst_ptrs)} destinations")
        arr = (C.c_void_p * B)(*[C.c_void_p(int(p)) for p in dst_ptrs])
        with torch.cuda.device(self.device):
            L.check(self.lib.fvhd_forward_scatter(self.handle, self._stream(), images.data_ptr(), _img_dtype(images), B, arr), self.handle)

    def forward_gather(self, images, local_out, peer_ptrs):
        """encode_images of this rank's shard with the all-gather fused into the projector's store: the projected tokens
        are written to `local_out` ([b,N,H] bf16 view of this rank's slot in its own gathered buffer) AND, by the same
        kernel, to `peer_ptrs` (ints: peer-mapped device addresses of this rank's slot in every other GPU's gathered
        buffer).  The caller orders the readers (e.g. a symmetric-memory barrier) -- see parallel.GatheredEncoder."""
        if self.hidden <= 0:
            raise L.FvhdError("forward_gather needs a plan with a projector")
        images = self._check_images(images, self.device)
        B = images.shape[0]
        if local_out.device != self.device:
            raise L.FvhdError(f"local_out on {local_out.device}, engine on {self.device}")
        self._check_out(local_out, (B, self.num_tokens, self.hidden), "local_out")
        n = len(peer_ptrs)
        arr = (C.c_void_p * max(n, 1))(*[C.c_void_p(int(p)) for p in peer_ptrs])
        with torch.cuda.device(self.device):
            L.check(self.lib.fvhd_forward_gather(self.handle, self._stream(), images.data_ptr(), _img_dtype(images), B,
                                                 local_out.data_ptr(), arr, n), self.handle)
        return local_out

    def run_units(self, first, last, x, batch):
        """Run units [first,last]; x = NCHW images (first == 0) or bf16 NHWC activation.  Returns bf16 [B, out_elems]."""
        info = self.units()
        out = torch.empty(batch, info[last]["out_elems"], dtype=torch.bfloat16, device=self.device)
        x = x.contiguous()
        with torch.cuda.device(self.device):
            L.check(self.lib.fvhd_run_units(self.handle, self._stream(), first, last, x.data_ptr(),
                                            _img_dtype(x) if first == 0 else L.BF16, batch, out.data_ptr()), self.handle)
        return out

    def profile_units(self, images):
        n = self.lib.fvhd_num_units(self.handle)
        ms = (C.c_float * n)()
        images = images.contiguous()
        with torch.cuda.device(self.device):
            L.check(self.lib.fvhd_profile_units(self.handle, self._stream(), images.data_ptr(), _img_dtype(images), images.shape[0], ms, n),
                    self.handle)
        return [float(v) for v in ms]

    def steps(self, batch=1):
        """Kernel-level plan: [{kernel, unit, flops, bytes}] for `batch` images per pass (needs load())."""
        n = self.lib.fvhd_num_steps(self.handle, batch)
        if n < 0:
            L.check(n, self.handle)
        out = []
        k, u, fl, by = C.c_char_p(), C.c_int(), C.c_double(), C.c_double()
        for i in range(n):
            L.check(self.lib.fvhd_step_info(self.handle, batch, i, C.byref(k), C.byref(u), C.byref(fl), C.byref(by)), self.handle)
            out.append(dict(kernel=k.value.decode(), unit=u.value, flops=fl.value, bytes=by.value))
        return out

    def profile_steps(self, images):
        """Milliseconds of every kernel launch of one forward (CUDA events around each launch)."""
        images = images.contiguous()
        B = images.shape[0]
        n = self.lib.fvhd_num_steps(self.handle, B)
        if n < 0:
            L.check(n, self.handle)
        ms = (C.c_float * n)()
        with torch.cuda.device(self.device):
            L.check(self.lib.fvhd_profile_steps(self.handle, self._stream(), images.data_ptr(), _img_dtype(images), B, ms, n), self.handle)
        return [float(v) for v in ms]

    def gemm(self, A, W, bias=None, residual=None, act=0):
        """D = act(A @ W^T + bias) + residual on the tcgen05 GEMM (A [M,K] bf16, W [N,K] bf16)."""
        M, K = A.shape
        N = W.shape[0]
        D = torch.empty(M, N, dtype=torch.bfloat16, device=A.device)
        with torch.cuda.device(A.device):
            L.check(self.lib.fvhd_gemm(self.handle, C.c_void_p(torch.cuda.current_stream(A.device).cuda_stream), A.data_ptr(), W.data_ptr(),
                                       bias.data_ptr() if bias is not None else None,
                                       residual.data_ptr() if residual is not None else None, D.data_ptr(), M, N, K, int(act)), self.handle)
        return D

    def convffn2(self, z, w1, b1, w2, b2, resid):
        """Same operands as convffn(), on the second-generation fused kernel (convffn.cuh); w2 f16 (production) or bf16 (mixed-format test)."""
        M, Cc = z.shape
        out = torch.empty(M, Cc, dtype=torch.bfloat16, device=z.device)
        with torch.cuda.device(z.device):
            L.check(self.lib.fvhd_convffn_half(self.handle, C.c_void_p(torch.cuda.current_stream(z.device).cuda_stream), z.data_ptr(), w1.data_ptr(),
                                           b1.data_ptr(), w2.data_ptr(), 1 if w2.dtype == torch.float16 else 0, b2.data_ptr(), resid.data_ptr(),
                                           out.data_ptr(), M, Cc), self.handle)
        return out

    def attention(self, qkv, batch, n_tokens):
        """MHSA core on qkv [B*N, 3C] bf16 -> [B*N, C] bf16 (kernel per FVHD_ATTN as it was when the engine was created)."""
        Cc = qkv.shape[1] // 3
        out = torch.empty(qkv.shape[0], Cc, dtype=torch.bfloat16, device=qkv.device)
        with torch.cuda.device(qkv.device):
            L.check(self.lib.fvhd_attention(self.handle, C.c_void_p(torch.cuda.current_stream(qkv.device).cuda_stream), qkv.data_ptr(),
                                            out.data_ptr(), int(batch), int(n_tokens), Cc), self.handle)
        return out

    def mixer(self, x, w3, b3, w7, b7):
        """(y, z) = (dw3x3(x) + b3, dw7x7(y) + b7) on the mixer kernel FVHD_MIXER selected when the engine was created; x bf16 NHWC
        [B,H,W,C], weights fp32 tap-major."""
        B, H, W, Cc = x.shape
        y = torch.empty_like(x)
        z = torch.empty_like(x)
        with torch.cuda.device(x.device):
            L.check(self.lib.fvhd_mixer(self.handle, C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream), x.data_ptr(), w3.data_ptr(),
                                        b3.data_ptr(), w7.data_ptr(), b7.data_ptr(), y.data_ptr(), z.data_ptr(), B, H, W, Cc), self.handle)
        return y, z

    def convffn(self, z, w1, b1, w2, b2, resid, trace=None):
        """resid + fc2(GELU(fc1(z) + b1)) + b2 on the fused ConvFFN kernels (z, resid [M,C] bf16; w1 [4C,C], w2 [C,4C] bf16;
        b1, b2 fp32; C in {96, 192, 384}).  `trace`: optional int64 CUDA tensor, 64 entries per CTA (C = 384 only)."""
        M, Cc = z.shape
        out = torch.empty(M, Cc, dtype=torch.bfloat16, device=z.device)
        with torch.cuda.device(z.device):
            L.check(self.lib.fvhd_convffn(self.handle, C.c_void_p(torch.cuda.current_stream(z.device).cuda_stream), z.data_ptr(), w1.data_ptr(),
                                          b1.data_ptr(), w2.data_ptr(), b2.data_ptr(), resid.data_ptr(), out.data_ptr(), M, Cc,
                                          trace.data_ptr() if trace is not None else None), self.handle)
        return out
