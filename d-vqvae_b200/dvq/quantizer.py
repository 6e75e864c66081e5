"""``VectorQuantizer`` — drop-in for the reference's ``network/vqvae/quantizer.py:10-75``.

Same constructor ``(n_e, e_dim, beta, al)`` (:20), same parameter key
``embedding.weight`` ``[n_e, e_dim]`` with the ``U(-1/n_e, 1/n_e)`` init (:26-27), same
return order — train path ``(loss, z_q, perplexity, min_encodings, min_encoding_indices)``
(:67), inference path ``(min_encoding_indices, z_q)`` (:54) — and ``get_emb(idx, dim)`` (:68).
Everything between is one call into the C ABI (``dvq_vq_forward`` + ``dvq_vq_finalize``):
the N x K distance matrix, the host-built one-hot and the second GEMM of the reference do not
exist here.  There is no CPU path: inputs must be fp32 or bf16 CUDA tensors.

Differences that are deliberate and documented (SURVEY §0.7, §0.8):
* bf16 latents (what an encoder produces under ``torch.autocast(..., dtype=torch.bfloat16)``) are
  quantized natively, without an fp32 copy: the call is the fp32 call on ``z.float()`` — the same
  indices and histogram, loss and perplexity as fp32 scalars — with ``z_q`` returned in bf16 (the fp32
  result rounded to nearest even).  The codebook stays an fp32 parameter; in the backward ``dz`` is
  bf16 (the fp32 formulas on the upcast values, rounded once) and the codebook gradient fp32.  Other
  dtypes (fp16, fp64) raise ``TypeError``.
* ``min_encodings`` ([N,K] fp32 one-hot, 1 TiB at BASELINE config 4) is materialised only while
  it is at most ``onehot_limit_bytes`` (default 2 GiB); above that the 5-tuple carries a
  ``LazyOneHot`` that can still produce it on demand.  Both reference callers discard it
  (network/VQVAE.py:32).
* ``get_emb`` accepts a batch of indices (the reference's scatter/view is valid for B=1 only);
  for one index the result is identical.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _cabi
from . import dist as _dist


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class LazyOneHot:
    """Stand-in for ``min_encodings`` when N*K*4 bytes would be unreasonable to allocate."""

    def __init__(self, indices: torch.Tensor, n_e: int):
        self.indices = indices
        self.n_e = n_e
        self.shape = torch.Size((indices.shape[0], n_e))
        self.dtype = torch.float32
        self.device = indices.device

    def materialize(self) -> torch.Tensor:
        out = torch.empty(self.shape, dtype=torch.float32, device=self.device)
        _onehot_into(self.indices, self.n_e, out)
        return out

    def __repr__(self):
        return "LazyOneHot(shape=%s, device=%s)" % (tuple(self.shape), self.device)


def _onehot_into(indices: torch.Tensor, n_e: int, out: torch.Tensor) -> None:
    """quantizer.py:40-42 through ``dvq_onehot`` (one coalesced write pass, no memset+scatter)."""
    with torch.cuda.device(out.device):
        _cabi.check(_cabi.lib.dvq_onehot(indices.data_ptr(), indices.shape[0], n_e, out.data_ptr(),
                                         _stream_ptr(out.device)), "dvq_onehot")


class _VQFunction(torch.autograd.Function):
    """Autograd wrapper of the fused forward (SURVEY §8f-3).  Backward of
    ``loss = al*mean((sg[z_q]-z)^2) + beta*mean((z_q-sg[z])^2)`` and of the straight-through
    ``z + sg[z_q - z]`` (quantizer.py:56-60):
        dz = g_zq + g_loss * al   * 2 (z - e) / (N*D)
        dE[k] = sum_{n: idx_n = k} g_loss * beta * 2 (e - z) / (N*D)."""

    @staticmethod
    def forward(ctx, z, weight, module):
        loss, z_q, ppl, idx = module._forward_train_raw(z, weight)   # z_q has the dtype of z (fp32 or bf16)
        # rows the returned loss is a mean over: the local count, or — row-sharded — the all-reduced histogram total
        # (a device scalar: no host sync).  The gradients below are the exact partial derivatives of the RETURNED
        # (global) loss with respect to the local rows of z and the local rows' contribution to dE; summing dE over
        # the ranks (all-reduce SUM) gives the exact codebook gradient.
        if module.process_group is not None:
            n_rows = module.last_stats[:module.n_e].sum().to(torch.float32)
        else:
            n_rows = torch.tensor(float(z.numel() // weight.shape[1]), device=z.device)
        ctx.save_for_backward(z, weight, idx, n_rows)
        ctx.al, ctx.beta = float(module.al), float(module.beta)
        ctx.mark_non_differentiable(ppl, idx)
        return loss, z_q, ppl, idx

    @staticmethod
    def backward(ctx, g_loss, g_zq, _g_ppl, _g_idx):
        z, weight, idx, n_rows = ctx.saved_tensors
        d = weight.shape[1]
        want_z, want_e = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if g_loss is None:
            g_loss = torch.zeros((), device=z.device)
        gl = g_loss.detach().to(torch.float32).reshape(1).contiguous()
        rows = n_rows.reshape(1).contiguous()
        flat = z.detach().reshape(-1, d)
        n = flat.shape[0]
        # bf16 z: g_zq arrives in bf16 (the dtype of z_q) and dz is returned in bf16; the arithmetic is fp32
        bf16 = z.dtype == torch.bfloat16
        gq = None
        if g_zq is not None:
            gq = g_zq.detach().to(z.dtype).reshape(-1, d).contiguous()
        zal = 8 if bf16 else 16   # the kernel moves 4 elements of z / g_zq / dz at a time
        if d % 4 == 0 and flat.data_ptr() % zal == 0 and weight.data_ptr() % 16 == 0 and (gq is None or gq.data_ptr() % zal == 0):
            # one fused pass (dvq_vq_backward_ex): dz written once, dE by vector reductions
            gz = torch.empty_like(flat) if want_z else None
            gw = torch.zeros_like(weight) if want_e else None
            with torch.cuda.device(z.device):
                _cabi.check(_cabi.lib.dvq_vq_backward_ex(
                    flat.data_ptr(), weight.detach().data_ptr(), idx.data_ptr(), gq.data_ptr() if gq is not None else None,
                    gl.data_ptr(), rows.data_ptr(), n, weight.shape[0], d, ctx.al, ctx.beta, _cabi.DVQ_Z_BF16 if bf16 else 0,
                    gz.data_ptr() if gz is not None else None, gw.data_ptr() if gw is not None else None,
                    _stream_ptr(z.device)), "dvq_vq_backward_ex")
            return (gz.view_as(z) if gz is not None else None), gw, None
        # shapes the vector kernel does not take (e_dim not a multiple of 4, odd storage offsets): same formulas in torch,
        # in fp32 (dz is cast to the dtype of z once)
        e = weight.detach().index_select(0, idx.view(-1))
        diff = (flat.float() - e) * (2.0 / (rows * d))
        gz = gw = None
        if want_z:
            gz = (gl * ctx.al) * diff
            if gq is not None:
                gz = gz + gq.float()
            gz = gz.to(z.dtype).view_as(z)
        if want_e:
            gw = torch.zeros_like(weight)
            gw.index_add_(0, idx.view(-1), (-(gl * ctx.beta)) * diff)
        return gz, gw, None


class VectorQuantizer(nn.Module):
    """Discretisation bottleneck of the VQ-VAE (reference: network/vqvae/quantizer.py:10)."""

    onehot_limit_bytes = 2 << 30

    def __getstate__(self):     # deepcopy / pickle: the workspace is a cache, a process group cannot be pickled
        d = self.__dict__.copy()
        d["_ws"] = None
        d["_cb_key"] = None
        d["process_group"] = None
        d.pop("last_stats", None)
        return d

    def __init__(self, n_e, e_dim, beta, al):
        super().__init__()
        self.n_e = n_e
        self.e_dim = e_dim
        self.beta = beta
        self.al = al
        self.embedding = nn.Embedding(self.n_e, self.e_dim)
        self.embedding.weight.data.uniform_(-1.0 / self.n_e, 1.0 / self.n_e)
        self.path = _cabi.DVQ_PATH_AUTO      # DVQ_PATH_SIMT / DVQ_PATH_TC force a kernel
        self.process_group = None            # set by dvq.dist.shard_module for the multi-GPU path
        self._ws = None
        # The codebook preparation (code norms, FP16 operand image, scale / residual bounds: three small launches) lives
        # in the workspace and is reused while the codebook is unchanged: same storage and tensor version, same N,
        # same workspace.  In-place writes through `.data` do not bump the version — call invalidate_codebook_cache()
        # after such an edit, or set cache_codebook = False.
        self.cache_codebook = True
        self._cb_key = None

    def invalidate_codebook_cache(self):
        """Forget the cached codebook preparation (needed after editing ``embedding.weight.data`` in place)."""
        self._cb_key = None

    def _load_from_state_dict(self, *args, **kwargs):
        self._cb_key = None
        return super()._load_from_state_dict(*args, **kwargs)

    def _apply(self, fn, *args, **kwargs):
        self._cb_key = None
        return super()._apply(fn, *args, **kwargs)

    # ------------------------------------------------------------------ helpers
    def _check(self, z: torch.Tensor, weight: torch.Tensor):
        if not isinstance(z, torch.Tensor):
            raise TypeError("z must be a torch.Tensor")
        if z.dtype != torch.float32 and z.dtype != torch.bfloat16:
            raise TypeError("dvq.VectorQuantizer computes in fp32 and takes fp32 or bf16 latents; got %s" % z.dtype)
        if not z.is_cuda or not weight.is_cuda:
            raise ValueError("dvq.VectorQuantizer has no CPU path: z and the codebook must be CUDA tensors "
                             "(got z on %s, codebook on %s)" % (z.device, weight.device))
        if z.device != weight.device:
            raise ValueError("z (%s) and the codebook (%s) are on different devices" % (z.device, weight.device))
        if z.numel() % self.e_dim != 0:
            raise RuntimeError("shape '[-1, %d]' is invalid for input of size %d" % (self.e_dim, z.numel()))
        if weight.dtype != torch.float32 or not weight.is_contiguous() or tuple(weight.shape) != (self.n_e, self.e_dim):
            raise ValueError("embedding.weight must be a contiguous fp32 [n_e, e_dim] tensor")

    def _workspace(self, n: int, flags: int, device) -> torch.Tensor:
        need = _cabi.vq_workspace_bytes(n, self.n_e, self.e_dim, flags)
        ws = self._ws
        if ws is None or ws.device != device or ws.numel() < need:
            ws = torch.empty(max(need, 256), dtype=torch.uint8, device=device)
            self._ws = ws
        return ws

    def _launch(self, z, weight, flags, z_q, idx, onehot, stats):
        n = z.numel() // self.e_dim
        if z.dtype == torch.bfloat16:
            flags |= _cabi.DVQ_Z_BF16
        ws = self._workspace(n, flags, z.device)
        # (the 16-byte alignment of z decides between the tcgen05 and the FP32 kernel under AUTO: part of the key, since
        #  only the former builds the operand image; so is the dtype of z, so that a preparation is reused only by a call
        #  of the same kind)
        key = (weight.data_ptr(), weight._version, ws.data_ptr(), n, flags & _cabi.DVQ_PATH_MASK, str(z.device),
               z.data_ptr() % 16 == 0 and z_q.data_ptr() % 16 == 0, z.dtype)
        if self.cache_codebook and key == self._cb_key:
            flags |= _cabi.DVQ_CODEBOOK_CACHED
        self._cb_key = None          # (stays None if the launch raises)
        hist_ptr = stats.data_ptr() if stats is not None else None
        sse_ptr = stats.data_ptr() + 8 * self.n_e if stats is not None else None
        with torch.cuda.device(z.device):
            _cabi.check(_cabi.lib.dvq_vq_forward(
                z.data_ptr(), weight.data_ptr(), n, self.n_e, self.e_dim, flags,
                z_q.data_ptr(), idx.data_ptr(), onehot.data_ptr() if onehot is not None else None,
                hist_ptr, sse_ptr, ws.data_ptr(), ws.numel(), _stream_ptr(z.device)), "dvq_vq_forward")
        self._cb_key = key

    def last_counters(self, n: int, flags: int | None = None):
        """(rows refined by the exact FP32 kernel, tcgen05 pipeline error code) of the last forward
        over ``n`` rows — a synchronous diagnostic read, not part of the hot path."""
        import ctypes as C
        if self._ws is None:
            return 0, 0
        out = (C.c_int * 4)()
        # (the counters do not depend on the dtype of z: DVQ_Z_BF16 may be set in `flags` or not)
        with torch.cuda.device(self._ws.device):
            _cabi.check(_cabi.lib.dvq_vq_read_counters(self._ws.data_ptr(), n, self.n_e, self.e_dim,
                                                       self.path if flags is None else flags, out), "dvq_vq_read_counters")
        return int(out[0]), int(out[1])

    def _forward_train_raw(self, z, weight):
        n = z.numel() // self.e_dim
        dev = z.device
        z_q = torch.empty_like(z)
        idx = torch.empty((n, 1), dtype=torch.int64, device=dev)
        # stats = hist[K] (uint64) | sse (float64), one buffer so the all-reduce is one message
        stats = torch.zeros(self.n_e + 1, dtype=torch.int64, device=dev)
        if n > 0:   # (a rank with an empty shard still joins the collective below with zeroed stats)
            self._launch(z, weight, _cabi.DVQ_TRAIN | self.path, z_q, idx, None, stats)
        n_total = n
        if self.process_group is not None:
            n_total = _dist.allreduce_stats(stats, self.n_e, n, self.process_group)
        out = torch.empty(2, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _cabi.check(_cabi.lib.dvq_vq_finalize(
                stats.data_ptr(), stats.data_ptr() + 8 * self.n_e, n_total, self.n_e, self.e_dim,
                float(self.al), float(self.beta), out.data_ptr(), out.data_ptr() + 4, _stream_ptr(dev)),
                "dvq_vq_finalize")
        self.last_stats = stats
        return out[0], z_q, out[1], idx

    # ------------------------------------------------------------------ reference API
    def forward(self, z, istrain):
        weight = self.embedding.weight
        self._check(z, weight)
        if not z.is_contiguous():
            # the reference's .view(-1, e_dim) accepts stride-compatible slices (e.g. h[:, :256]) and raises for the
            # rest; the kernels read dense rows, so any layout is copied once (autograd flows through the copy)
            z = z.contiguous()
        n = z.numel() // self.e_dim
        if not istrain:
            # quantizer.py:44-54
            wd = weight.detach()
            z_q = torch.empty_like(z)
            idx = torch.empty((n, 1), dtype=torch.int64, device=z.device)
            self._launch(z.detach(), wd, self.path, z_q, idx, None, None)
            return idx, z_q

        # quantizer.py:35-43, 56-67
        if n == 0 and self.process_group is None:  # torch.mean over an empty tensor is NaN in the reference as well
            nan = torch.full((), float("nan"), device=z.device)
            return nan, torch.empty_like(z), nan.clone(), torch.empty((0, self.n_e), device=z.device), \
                torch.empty((0, 1), dtype=torch.int64, device=z.device)
        if torch.is_grad_enabled() and (z.requires_grad or weight.requires_grad):
            loss, z_q, ppl, idx = _VQFunction.apply(z, weight, self)
        else:
            loss, z_q, ppl, idx = self._forward_train_raw(z.detach(), weight.detach())
        if n * self.n_e * 4 <= self.onehot_limit_bytes:
            enc = torch.empty((n, self.n_e), dtype=torch.float32, device=z.device)
            _onehot_into(idx, self.n_e, enc)
        else:
            enc = LazyOneHot(idx, self.n_e)
        return loss, z_q, ppl, enc, idx

    # ------------------------------------------------------------------ training hooks (SURVEY §8f-3)
    # The reference trains its codebooks through the loss alone (quantizer.py:56-57).  These hooks are the usual
    # companions of a VQ bottleneck and run on what the fused forward already produced: the (all-reduced) usage
    # histogram in ``last_stats`` and the indices; the per-code input sums come from one scatter-add kernel.
    def code_sums(self, z, idx):
        """[n_e, e_dim] sum of the latents assigned to each code (``dvq_vq_code_sums``); summed over the ranks of a
        row-sharded module."""
        flat = z.detach().reshape(-1, self.e_dim).contiguous()
        bf16 = flat.dtype == torch.bfloat16   # bf16 latents are summed in fp32 (sums stay fp32)
        if self.e_dim % 4 != 0 or flat.data_ptr() % (8 if bf16 else 16) != 0:
            sums = torch.zeros(self.n_e, self.e_dim, device=flat.device)
            sums.index_add_(0, idx.view(-1), flat.float())
        else:
            sums = torch.zeros(self.n_e, self.e_dim, device=flat.device)
            with torch.cuda.device(flat.device):
                _cabi.check(_cabi.lib.dvq_vq_code_sums_ex(flat.data_ptr(), idx.contiguous().data_ptr(), flat.shape[0], self.n_e,
                                                          self.e_dim, _cabi.DVQ_Z_BF16 if bf16 else 0, sums.data_ptr(),
                                                          _stream_ptr(flat.device)), "dvq_vq_code_sums_ex")
        if self.process_group is not None and _dist.world_size(self.process_group) > 1:
            _dist.all_reduce_sum(sums, self.process_group)
        return sums

    @torch.no_grad()
    def ema_update(self, z, idx, decay: float = 0.99, eps: float = 1e-5):
        """Exponential-moving-average codebook update fed by the last forward's histogram (global on a row-sharded
        module): cluster_size <- decay * cluster_size + (1 - decay) * hist; ema_w <- decay * ema_w + (1 - decay) * sums;
        embedding <- ema_w / laplace-smoothed cluster_size.  State lives in (non-persistent) buffers created on first use."""
        hist = self.last_stats[:self.n_e].to(torch.float32)
        sums = self.code_sums(z, idx)
        if not hasattr(self, "ema_cluster_size"):
            self.register_buffer("ema_cluster_size", torch.zeros(self.n_e, device=hist.device), persistent=False)
            self.register_buffer("ema_w", self.embedding.weight.detach().clone(), persistent=False)
        self.ema_cluster_size.mul_(decay).add_(hist, alpha=1.0 - decay)
        self.ema_w.mul_(decay).add_(sums, alpha=1.0 - decay)
        total = self.ema_cluster_size.sum()
        smoothed = (self.ema_cluster_size + eps) / (total + self.n_e * eps) * total
        self.embedding.weight.copy_(self.ema_w / smoothed.unsqueeze(1))
        return hist

    @torch.no_grad()
    def reset_unused_codes(self, z, min_usage: int = 1, generator=None):
        """Re-seed the codes the last forward used fewer than ``min_usage`` times (global histogram) with latents
        drawn from ``z``; on a row-sharded module rank 0's draw is broadcast so the replicas stay identical.
        Returns the number of codes reset (a host int: this hook synchronises)."""
        hist = self.last_stats[:self.n_e]
        dead = (hist < min_usage).nonzero().view(-1)
        if dead.numel() == 0:
            return 0
        flat = z.detach().reshape(-1, self.e_dim)
        pick = torch.randint(0, flat.shape[0], (dead.numel(),), device=flat.device, generator=generator)
        new_rows = flat[pick].float().contiguous()   # (bf16 latents: the codebook stays fp32)
        if self.process_group is not None and _dist.world_size(self.process_group) > 1:
            _dist.broadcast0(new_rows, self.process_group)
        self.embedding.weight[dead] = new_rows
        if hasattr(self, "ema_w"):
            self.ema_w[dead] = new_rows
            self.ema_cluster_size[dead] = float(min_usage)
        return int(dead.numel())

    def get_emb(self, min_encoding_indices, dim):
        """quantizer.py:68-75: index -> embedding.  Returns ``[B, dim]`` (``[1, dim]`` for the
        reference's single-index call)."""
        weight = self.embedding.weight.detach()
        if not weight.is_cuda:
            raise ValueError("dvq.VectorQuantizer has no CPU path: the codebook must be on a CUDA device")
        idx = torch.as_tensor(min_encoding_indices, device=weight.device).reshape(-1).to(torch.int64).contiguous()
        if dim != self.e_dim:
            raise RuntimeError("shape '[1, %d]' is invalid for an embedding of width %d" % (dim, self.e_dim))
        out = torch.empty((idx.numel(), self.e_dim), dtype=torch.float32, device=weight.device)
        oob = torch.zeros(1, dtype=torch.int32, device=weight.device)
        with torch.cuda.device(weight.device):
            _cabi.check(_cabi.lib.dvq_gather(weight.data_ptr(), idx.data_ptr(), idx.numel(), self.n_e, self.e_dim,
                                             out.data_ptr(), oob.data_ptr(), _stream_ptr(weight.device)), "dvq_gather")
        # same failure mode as the reference's scatter_ on CUDA: a device-side assert
        torch._assert_async(oob[0] == 0, "dvq.get_emb: index out of range")
        return out.view(-1, dim)
