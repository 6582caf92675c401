"""Batched / multi-GPU inference harness around the model forward.

Restates the 10 lines of the reference inferencer methods that surround the model call
(speech_enhance/fullsubnet_plus/inferencer/inferencer.py:140-165 ``mag_complex_full_band_crm_mask`` and
:116-137 ``full_band_crm_mask``): STFT -> model -> decompress_cIRM -> complex multiply -> iSTFT, with STFT and
iSTFT kept in PyTorch on the GPU as BASELINE.json's north_star prescribes, for a BATCH of equal-length clips
(the reference is hard-wired to batch 1, audio_zen/inferencer/base_inferencer.py:65-69).

Multi-GPU: utterances are independent, so a batch is sharded across ranks (one process per GPU) with no
data-path collective; the only exchange is one all-gather of the enhanced waveforms (NCCL on GPUs, gloo in
the CPU tests of the host logic).
"""
import ctypes as C

import torch
import torch.distributed as dist

from . import _lib


def stft(y, n_fft=512, hop_length=256, win_length=512):
    """reference audio_zen/acoustics/feature.py:10-31.  y [B, L] -> complex [B, F, T]."""
    assert y.dim() == 2
    return torch.stft(y, n_fft, hop_length, win_length, window=torch.hann_window(n_fft, device=y.device),
                      return_complex=True)


_ISTFT_ENV = {}


def istft(spec, n_fft=512, hop_length=256, win_length=512, length=None):
    """reference audio_zen/acoustics/feature.py:34-65 (complex input) = torch.istft(spec, n_fft, hop, win, hann window, center=True).

    Restated with the same ATen operators torch.istft issues (irfft -> window -> overlap-add by ``fold`` -> division by the
    overlap-added squared window) but WITHOUT its "window overlap add min" check: that check reads a GPU scalar back to the host and
    therefore synchronises the calling thread with the stream on every call, which would serialise the pipelined harness
    (EnhancePipeline: the host must be able to enqueue batch i+1 while batch i is still on the GPU).  The envelope depends only on
    (n_fft, hop, window, frames), so it is built -- and checked -- once per geometry and cached.  CPU tensors use torch.istft."""
    if not spec.is_cuda or win_length != n_fft:
        return torch.istft(spec, n_fft, hop_length, win_length, window=torch.hann_window(n_fft, device=spec.device), length=length)
    B, F, T = spec.shape
    full = n_fft + hop_length * (T - 1)
    key = (n_fft, hop_length, T, spec.device)
    if key not in _ISTFT_ENV:
        window = torch.hann_window(n_fft, device=spec.device)
        env = torch.nn.functional.fold((window * window).view(1, n_fft, 1).expand(1, n_fft, T), output_size=(1, full),
                                       kernel_size=(1, n_fft), stride=(1, hop_length)).reshape(full)
        start = n_fft // 2
        if not bool(env[start: full - start].abs().min() > 1e-11):          # the check torch.istft makes on every call, made once here
            raise RuntimeError("istft: window overlap add min is zero for this n_fft / hop_length")
        _ISTFT_ENV[key] = (window, env)
    window, env = _ISTFT_ENV[key]
    frames = torch.fft.irfft(spec.transpose(1, 2), n=n_fft, dim=-1) * window              # [B, T, n_fft]
    y = torch.nn.functional.fold(frames.transpose(1, 2), output_size=(1, full), kernel_size=(1, n_fft),
                                 stride=(1, hop_length)).reshape(B, full)
    start = n_fft // 2
    end = start + length if length is not None else full - start
    if end > full:                                                                        # torch.istft pads with zeros up to `length`
        y = torch.nn.functional.pad(y, (0, end - full))
        envp = torch.nn.functional.pad(env, (0, end - full), value=1.0)
        return y[:, start:end] / envp[start:end]
    return y[:, start:end] / env[start:end]


def decompress_cIRM(mask, K=10, limit=9.9):
    """reference audio_zen/acoustics/mask.py:60-63."""
    mask = limit * (mask >= limit) - limit * (mask <= -limit) + mask * (torch.abs(mask) < limit)
    return -K * torch.log((K - mask) / (K + mask))


def apply_cirm(crm, X):
    """decompress_cIRM + complex multiply (reference inferencer.py:152-157): one fused CUDA kernel behind the C ABI for
    CUDA float32 inputs, the torch restatement otherwise (CPU tests of the harness)."""
    if crm.is_cuda and crm.dtype == torch.float32 and X.dtype == torch.complex64:
        crm = crm.contiguous()
        Xr = torch.view_as_real(X.contiguous())
        out = torch.empty_like(Xr)
        B, _, F, T = crm.shape
        with torch.cuda.device(crm.device):
            stream = C.c_void_p(torch.cuda.current_stream(crm.device).cuda_stream)
            _lib.check(_lib.load_library().fsn_apply_cirm(C.c_void_p(crm.data_ptr()), C.c_void_p(Xr.data_ptr()), C.c_void_p(out.data_ptr()),
                                                          B, F, T, stream))
        return torch.view_as_complex(out)
    m = decompress_cIRM(crm)                                   # [B, 2, F, T]
    return torch.complex(m[:, 0] * X.real - m[:, 1] * X.imag, m[:, 1] * X.real + m[:, 0] * X.imag)


@torch.no_grad()
def enhance_batch(model, noisy, n_fft=512, hop_length=256, win_length=512, complex_inputs=True):
    """noisy [B, L] float32 on the model's device -> enhanced [B, L].
    complex_inputs=True mirrors mag_complex_full_band_crm_mask (FullSubNet_Plus), False full_band_crm_mask (Model)."""
    X = stft(noisy, n_fft, hop_length, win_length)
    mag = X.abs().unsqueeze(1)
    if hasattr(model, "enhance_spectrum") and X.is_cuda:          # model + decompress + complex multiply in one call (fused epilogue)
        enh = model.enhance_spectrum(mag, X.real.unsqueeze(1).contiguous(), X.imag.unsqueeze(1).contiguous())
        return istft(enh, n_fft, hop_length, win_length, length=noisy.size(-1))
    if complex_inputs:
        crm = model(mag, X.real.unsqueeze(1).contiguous(), X.imag.unsqueeze(1).contiguous())
    else:
        crm = model(mag)
    return istft(apply_cirm(crm, X), n_fft, hop_length, win_length, length=noisy.size(-1))


def shard_range(n_items, rank, world_size):
    """Contiguous shard [lo, hi) of rank; sizes differ by at most one (ragged batches are allowed)."""
    base, rem = divmod(n_items, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def all_gather_enhanced(local, n_items, group=None):
    """Gather per-rank enhanced waveforms [n_local, L] into [n_items, L] on every rank with ONE collective
    (all_gather_into_tensor on equal shards, padded all_gather when the batch is ragged)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local
    world = dist.get_world_size(group)
    L = local.size(1)
    per = (n_items + world - 1) // world
    buf = local
    if local.size(0) != per:
        buf = torch.zeros((per, L), dtype=local.dtype, device=local.device)
        buf[: local.size(0)] = local
    out = torch.empty((world * per, L), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, buf.contiguous(), group=group)
    if per * world == n_items:
        return out
    pieces = []
    for r in range(world):
        lo, hi = shard_range(n_items, r, world)
        pieces.append(out[r * per: r * per + (hi - lo)])
    return torch.cat(pieces, 0)


@torch.no_grad()
def enhance_sharded(model, noisy_all, group=None, **kw):
    """Data-parallel enhancement: every rank holds the full list of clips (or at least its shard), enhances its
    contiguous shard and all-gathers the waveforms.  noisy_all [N, L] on the local device."""
    if dist.is_available() and dist.is_initialized():
        rank, world = dist.get_rank(group), dist.get_world_size(group)
    else:
        rank, world = 0, 1
    lo, hi = shard_range(noisy_all.size(0), rank, world)
    local = enhance_batch(model, noisy_all[lo:hi], **kw) if hi > lo else noisy_all.new_zeros((0, noisy_all.size(1)))
    return all_gather_enhanced(local, noisy_all.size(0), group)


class EnhancePipeline:
    """Enhancement of a STREAM of equal-shape batches with everything overlapped (what the reference's inferencer loop,
    base_inferencer.py:133-160, does one clip at a time):

        push(i):   [optional H2D of pinned host spectra on a copy stream] -> pipelined model call for batch i  (the front end of batch i
                   runs while the sub-band LSTM of batch i-1 is still running, see fsn_model_submit; with fused_post the LSTM epilogue
                   also does decompress_cIRM x noisy spectrum, fsn_model_submit_enhance)
                   then, on a side stream, for batch i-1: [cIRM post-processing if not fused] -> torch.istft ->
                   ONE all-gather of the enhanced waveforms over the process group (world > 1) [-> D2H into pinned host memory]
        flush():   post-process the last batch and synchronise; returns the list of results in push order.

    The collective therefore runs on the side stream underneath the NEXT batch's forward (SURVEY.md 2a C1), never on the
    critical path.  Results: device tensors [world * B, L] (gathered) or [B, L]; with ``to_host=True`` this rank's shard in
    pinned host memory.  Input / result buffers form a ring of NSLOT preallocated slots (no allocation on the steady-state path: a
    cudaMalloc would synchronise the device): a result is valid until NSLOT pushes later (copy it if kept longer).  The ring is
    deeper than the two batches in flight on purpose: reusing a slot waits for the post-processing that last read it, and with only
    two slots that wait would hold back the FRONT END of batch i+1 until the iSTFT of batch i-1 is done.
    """
    NSLOT = 4

    def __init__(self, model, length, n_fft=512, hop_length=256, win_length=512, complex_inputs=True, gather=True, to_host=False,
                 keep_results=True, group=None, fused_post=True):
        self.model, self.length, self.stft_args = model, length, (n_fft, hop_length, win_length)
        self.fused = fused_post
        self.complex_inputs, self.to_host, self.keep, self.group = complex_inputs, to_host, keep_results, group
        self.world = dist.get_world_size(group) if (gather and dist.is_available() and dist.is_initialized()) else 1
        self.dev = next(model.parameters()).device
        self.post, self.copy = torch.cuda.Stream(self.dev), torch.cuda.Stream(self.dev)
        self.pending = None                       # (lane, slot) of the batch whose LSTM may still be running
        self.n = 0
        ring = lambda: [None] * self.NSLOT
        self.inbuf, self.outbuf, self.post_done, self.host_out, self.gathered = ring(), ring(), ring(), ring(), ring()
        self.results = []
        self.last = None                          # result of the most recently finished batch (kept or not)

    def _slot(self, slot, B, F, T):
        if self.inbuf[slot] is None or tuple(self.inbuf[slot][0].shape) != (B, 1, F, T):
            self.inbuf[slot] = [torch.empty((B, 1, F, T), dtype=torch.float32, device=self.dev) for _ in range(3)]
            self.outbuf[slot] = (torch.empty((B, F, T), dtype=torch.complex64, device=self.dev) if self.fused else
                                 torch.empty((B, 2, F, T), dtype=torch.float32, device=self.dev))
            self.gathered[slot] = self.host_out[slot] = None
        return self.inbuf[slot], self.outbuf[slot]

    def _finish(self, item):
        lane, slot = item
        with torch.cuda.stream(self.post):
            self.model.wait_lane(lane, self.post)                       # the sub-band LSTM of that batch has written its output
            out = self.outbuf[slot]
            if out.is_complex():                                        # fused epilogue: the enhanced spectrum itself
                spec = out
            else:
                _, real, imag = self.inbuf[slot]
                spec = apply_cirm(out, torch.complex(real[:, 0], imag[:, 0]))
            enh = istft(spec, *self.stft_args, length=self.length)
            res = enh
            if self.world > 1:
                if self.gathered[slot] is None:
                    self.gathered[slot] = torch.empty((self.world * enh.size(0), enh.size(1)), dtype=enh.dtype, device=self.dev)
                dist.all_gather_into_tensor(self.gathered[slot], enh.contiguous(), group=self.group)
                res = self.gathered[slot]
            if self.to_host:
                if self.host_out[slot] is None:
                    self.host_out[slot] = torch.empty(tuple(enh.shape), dtype=enh.dtype).pin_memory()
                self.host_out[slot].copy_(enh, non_blocking=True)       # this rank's shard -> pinned host memory
                res = self.host_out[slot]
            if self.post_done[slot] is None:
                self.post_done[slot] = torch.cuda.Event()
            self.post_done[slot].record(self.post)
        self.last = res
        if self.keep:
            self.results.append(res)

    def push(self, X=None, host=None):
        """One batch: ``X`` complex64 [B, F, T] on the device, or ``host`` = (mag, real, imag) pinned CPU float32 [B, 1, F, T]
        (the C ABI's host-buffer layout)."""
        slot = self.n % self.NSLOT
        main = torch.cuda.current_stream(self.dev)
        if host is not None:
            B, _, F, T = host[0].shape
        else:
            B, F, T = X.shape
        (mag, real, imag), out = self._slot(slot, B, F, T)
        if self.post_done[slot] is not None:
            main.wait_event(self.post_done[slot])                       # input / output buffers of this slot are free again
        if host is not None:
            with torch.cuda.stream(self.copy):
                if self.post_done[slot] is not None:
                    self.copy.wait_event(self.post_done[slot])
                for d, h in zip((mag, real, imag), host):
                    if h is not None:
                        d.copy_(h, non_blocking=True)
                if getattr(self, "_h2d_ev", None) is None:
                    self._h2d_ev = [torch.cuda.Event() for _ in range(self.NSLOT)]
                self._h2d_ev[slot].record(self.copy)
            main.wait_event(self._h2d_ev[slot])
        else:
            torch.abs(X, out=mag[:, 0])
            real[:, 0].copy_(X.real)
            imag[:, 0].copy_(X.imag)
        if self.fused:                                                  # model + decompress_cIRM x spectrum in the LSTM epilogue
            self.model.enhance_spectrum(mag, real, imag, pipelined=True, out=out, hold=False)
        elif self.complex_inputs:
            self.model.submit(mag, real, imag, out=out, hold=False)
        else:
            self.model.submit(mag, out=out, hold=False)
        item = (self.model.last_lane, slot)
        if self.pending is not None:
            self._finish(self.pending)
        self.pending = item
        self.n += 1

    def flush(self):
        if self.pending is not None:
            self._finish(self.pending)
            self.pending = None
        self.post.synchronize()
        self.model.wait()
        out, self.results = self.results, []
        return out
