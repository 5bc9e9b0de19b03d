"""WaveRNNEngine: the torch-facing wrapper of one libb200tts context (one GPU).

PyTorch is only plumbing here (device memory, current stream); all arithmetic runs in
csrc/ through the C ABI.  Tensors in, tensors out.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import GenOpts, Rng, WaveRNNCfg


def _cfg_from_dims(dims: dict) -> WaveRNNCfg:
    c = WaveRNNCfg()
    c.rnn_dims, c.fc_dims, c.bits, c.pad = dims['rnn_dims'], dims['fc_dims'], dims['bits'], dims['pad']
    c.feat_dims, c.compute_dims = dims['feat_dims'], dims['compute_dims']
    c.res_out_dims, c.res_blocks = dims['res_out_dims'], dims['res_blocks']
    f = tuple(int(x) for x in dims['upsample_factors'])
    if not 1 <= len(f) <= 4:
        raise ValueError('upsample_factors must have 1..4 entries')
    c.n_upsample = len(f)
    for i, s in enumerate(f):
        c.upsample_factors[i] = s
    c.hop_length = dims['hop_length']
    return c


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class WaveRNNEngine:
    """Owns the packed weights of one model on one device."""

    def __init__(self, state_dict: dict, dims: dict, device: int | None = None):
        if not torch.cuda.is_available():
            raise RuntimeError('no CUDA device: the B200 WaveRNN path has no CPU fallback')
        self.lib = _lib.load()
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.dims = dict(dims)
        self.hop = int(dims['hop_length'])
        self.feat = int(dims['feat_dims'])
        self.res_out = int(dims['res_out_dims'])
        self.n_classes = 1 << int(dims['bits'])
        host = {}
        for k, v in state_dict.items():
            if hasattr(v, 'detach'):
                v = v.detach().cpu().numpy()
            v = np.asarray(v)
            if v.dtype.kind == 'f':
                host[k] = np.ascontiguousarray(v, dtype=np.float32)
        arr, keep = _lib.make_tensor_array(host)
        cfg = _cfg_from_dims(dims)
        h = C.c_void_p()
        _lib.check(self.lib.b200tts_wavernn_create(C.byref(h), self.device, C.byref(cfg), arr, len(arr)))
        del keep
        self._h = h

    def close(self):
        if getattr(self, '_h', None):
            self.lib.b200tts_wavernn_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -------------------------------------------------------------------------------------------
    def _dev(self):
        return torch.device('cuda', self.device)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _mel(self, mels):
        m = torch.as_tensor(mels)
        if m.dim() != 3 or m.shape[1] != self.feat:
            raise ValueError(f'mels must be [B, {self.feat}, T], got {tuple(m.shape)}')
        return m.to(device=self._dev(), dtype=torch.float32).contiguous()

    def upsample(self, mels, full_aux: bool = True):
        """[B, feat, T] -> (mels_up [B, T*hop, feat], aux [B, T*hop, res_out] or frame-rate [B, T, res_out])."""
        m = self._mel(mels)
        B, _, T = m.shape
        S = T * self.hop
        with torch.cuda.device(self.device):
            up = torch.empty(B, S, self.feat, device=self._dev(), dtype=torch.float32)
            auxf = torch.empty(B, T, self.res_out, device=self._dev(), dtype=torch.float32)
            aux = torch.empty(B, S, self.res_out, device=self._dev(), dtype=torch.float32) if full_aux else None
            _lib.check(self.lib.b200tts_wavernn_upsample(self._h, _ptr(m), B, T, _ptr(up), _ptr(auxf), _ptr(aux),
                                                         self._stream()))
        return up, (aux if full_aux else auxf)

    def generate(self, mels, *, seed: int = 0, utterance_offset: int = 0, utterance_ids=None, q=None, teacher=None,
                 return_logits: bool = False, want_wave: bool = True, mu_law: bool = True, kernel: str = 'auto',
                 max_steps: int = 0, fold=None, utt_frames=None, pack=None):
        """Runs the generation loop on the device.

        Returns dict(labels int16 [B,S] cuda, wave float64 [B,wave_len] cuda or None, logits [S,B,NC] or None).
        q: optional Exp(1) noise [S,B,NC] (torch/numpy) -> EXT_EXPONENTIAL mode; otherwise PHILOX(seed).
        pack: optional packed-row schedule dict(rows, utt int32 [rows, segs], start int32 [rows, segs+1], steps) from
        pipeline.pack_schedule: `rows` kernel rows run queues of the B utterances back to back (gen_opts.d_pack_*).
        """
        m = self._mel(mels)
        B, _, T = m.shape
        S = T * self.hop
        GB, GS = B, S                                     # rows / steps the generation kernels see
        if fold is not None:
            if B != 1:
                raise ValueError('fold-with-overlap generation takes exactly one utterance')
            GB, GS = self.fold_geometry(T, int(fold[0]), int(fold[1]))
        steps = max_steps if max_steps else GS
        dev = self._dev()
        with torch.cuda.device(self.device):
            labels = torch.zeros(GB, GS, device=dev, dtype=torch.int16)
            wave = None
            if want_wave and steps == GS:
                wave = torch.empty(B, (T - 1) * self.hop, device=dev, dtype=torch.float64)
            rng, opts, keep, logits = self._call_args(B, GB, GS, steps, seed=seed, utterance_offset=utterance_offset,
                                                      utterance_ids=utterance_ids, q=q, teacher=teacher, return_logits=return_logits,
                                                      mu_law=mu_law, kernel=kernel, max_steps=max_steps, fold=fold,
                                                      utt_frames=utt_frames, pack=pack)
            _lib.check(self.lib.b200tts_wavernn_generate(self._h, _ptr(m), B, T, C.byref(rng), C.byref(opts),
                                                         _ptr(labels), _ptr(wave), self._stream()))
            # keep inputs alive until the stream has consumed them
            for t in [m] + keep:
                t.record_stream(torch.cuda.current_stream(self.device))
        return dict(labels=labels, wave=wave, logits=logits, steps=steps)

    def _call_args(self, B, GB, GS, steps, *, seed, utterance_offset, utterance_ids, q, teacher, return_logits, mu_law, kernel,
                   max_steps, fold, utt_frames, pack):
        """Rng / GenOpts of a generate call, the device tensors they point to, and the logits buffer (or None)."""
        dev = self._dev()
        rng = Rng()
        rng.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        rng.utterance_offset = int(utterance_offset)
        ids = None
        if utterance_ids is not None:       # rows that are NOT consecutive utterances (length-sorted chunks): per-row global index
            ids = torch.as_tensor(np.asarray(utterance_ids, dtype=np.int64)).to(dev).contiguous()
            if tuple(ids.shape) != (B,) or fold is not None:
                raise ValueError('utterance_ids must be [B] (and cannot be combined with fold)')
            rng.d_utterance_ids = ids.data_ptr()
        qd = None
        if q is not None:
            qd = torch.as_tensor(q).to(device=dev, dtype=torch.float32).contiguous()
            if qd.dim() != 3 or tuple(qd.shape[1:]) != (GB, self.n_classes) or qd.shape[0] < steps:
                raise ValueError(f'q must be [>= {steps}, {GB}, {self.n_classes}], got {tuple(qd.shape)}')
            rng.mode = _lib.RNG_EXT_EXPONENTIAL
            rng.d_q = qd.data_ptr()
        else:
            rng.mode = _lib.RNG_PHILOX
        opts = GenOpts()
        opts.kernel = _lib.KERNELS[kernel]
        opts.mu_law = 1 if mu_law else 0
        opts.max_steps = int(max_steps)
        if fold is not None:
            opts.fold_target, opts.fold_overlap = int(fold[0]), int(fold[1])
        pk_u = pk_s = None
        if pack is not None:
            pk_u = torch.as_tensor(np.ascontiguousarray(pack['utt'], dtype=np.int32)).to(dev)
            pk_s = torch.as_tensor(np.ascontiguousarray(pack['start'], dtype=np.int32)).to(dev)
            rows, segs = pk_u.shape
            if tuple(pk_s.shape) != (rows, segs + 1) or rows != int(pack['rows']):
                raise ValueError('pack: utt must be [rows, segs], start [rows, segs + 1]')
            opts.d_pack_utt, opts.d_pack_start = pk_u.data_ptr(), pk_s.data_ptr()
            opts.pack_rows, opts.pack_segs, opts.pack_steps = rows, segs, int(pack['steps'])
        uf = None
        if utt_frames is not None:
            uf = torch.as_tensor(utt_frames).to(device=dev, dtype=torch.int32).contiguous()
            if tuple(uf.shape) != (B,):
                raise ValueError('utt_frames must be [B]')
            opts.d_utt_frames = uf.data_ptr()
        td = None
        if teacher is not None:
            td = torch.as_tensor(teacher).to(device=dev, dtype=torch.int16).contiguous()
            if tuple(td.shape) != (GB, GS):
                raise ValueError('teacher must be [B, S] ([n_folds, fold_len] when folding)')
            opts.d_teacher = td.data_ptr()
        logits = None
        if return_logits:
            logits = torch.empty(steps, GB, self.n_classes, device=dev, dtype=torch.float32)
            opts.d_logits = logits.data_ptr()
        return rng, opts, [t for t in (qd, td, uf, ids, pk_u, pk_s) if t is not None], logits

    def generate_stream(self, mels, *, seed: int = 0, utterance_offset: int = 0, utterance_ids=None, utt_frames=None,
                        mu_law: bool = True, q=None, teacher=None, chunk_steps: int | None = None, timeout_s: float = 30.0,
                        device_out: dict | None = None):
        """Generator: the wave of `generate` (same arguments, same bits) handed out WHILE the push kernel runs.

        Yields (start, chunk): chunk is a float64 numpy array [B, n] of the final samples [start, start + n) of every row, in
        order, until all (T-1)*hop samples have been yielded; a chunk is ready every `chunk_steps` lock-steps (default: one
        hop = one mel frame, 12.5 ms of audio).  1..32 rows, PHILOX or external noise; no folding / packing / max_steps.
        The launch happens at the first next().  Raises if the kernel gives up, if no progress is seen for `timeout_s`, or if
        the final check() fails.  A consumer that stops early still waits (on close) until the launch has finished writing the
        pinned buffers this generator owns.  device_out (a dict), if given, receives the call's device `labels` and `wave`.
        """
        m = self._mel(mels)
        B, _, T = m.shape
        S, L = T * self.hop, (T - 1) * self.hop
        chunk = self.hop if chunk_steps is None else int(chunk_steps)
        if chunk < 1:
            raise ValueError('chunk_steps must be >= 1')
        dev = self._dev()
        stream = torch.cuda.current_stream(self.device)
        with torch.cuda.device(self.device):
            labels = torch.zeros(B, S, device=dev, dtype=torch.int16)
            wave = torch.empty(B, L, device=dev, dtype=torch.float64)
            h_wave = torch.empty(B, L, dtype=torch.float64, pin_memory=True)
            h_prog = torch.zeros(1, dtype=torch.int64, pin_memory=True)
            rng, opts, keep, _ = self._call_args(B, B, S, S, seed=seed, utterance_offset=utterance_offset,
                                                 utterance_ids=utterance_ids, q=q, teacher=teacher, return_logits=False,
                                                 mu_law=mu_law, kernel='auto', max_steps=0, fold=None, utt_frames=utt_frames,
                                                 pack=None)
            _lib.check(self.lib.b200tts_wavernn_generate_stream(
                self._h, _ptr(m), B, T, C.byref(rng), C.byref(opts), chunk, C.c_void_p(h_wave.data_ptr()),
                C.c_void_p(h_prog.data_ptr()), _ptr(labels), _ptr(wave), C.c_void_p(stream.cuda_stream)))
        if device_out is not None:
            device_out.update(labels=labels, wave=wave)
        hw = h_wave.numpy()
        seen = C.c_int64()
        done, finished = 0, False
        try:
            while done < L:
                want = min(L, done + chunk)              # sample n is final once progress > n
                _lib.check(self.lib.b200tts_wavernn_stream_wait(C.c_void_p(h_prog.data_ptr()), want, int(timeout_s * 1000),
                                                                C.byref(seen)))
                p = int(seen.value)
                if p < 0:
                    self.check()                         # raises with the kernel's own message
                    raise _lib.B200TTSError(-2, 'streaming kernel gave up (a peer thread block did not answer)')
                if p < want:
                    raise TimeoutError(f'no streaming progress for {timeout_s} s (at {p} of {L} samples)')
                n = min(p, L)
                yield done, hw[:, done:n].copy()
                done = n
            self.check()
            finished = True
        finally:
            if not finished:
                stream.synchronize()                     # the kernel may still write h_wave / h_prog: never free them under it
            del keep, m, h_wave, h_prog

    def fold_geometry(self, T: int, target: int, overlap: int):
        """(n_folds, fold_len) of fold_with_overlap for a T-frame utterance."""
        nf, fl = C.c_int(), C.c_int()
        _lib.check(self.lib.b200tts_wavernn_fold_geometry(int(T), self.hop, int(target), int(overlap), C.byref(nf), C.byref(fl)))
        return nf.value, fl.value

    def generate_host(self, mels: np.ndarray, *, seed: int = 0, utterance_offset: int = 0, mu_law: bool = True,
                      kernel: str = 'auto', want_labels: bool = True, want_wave: bool = True):
        """HOST buffers in, HOST buffers out, synchronous: the call `wavernn_gen.py` makes end to end."""
        m = np.ascontiguousarray(mels, dtype=np.float32)
        if m.ndim != 3 or m.shape[1] != self.feat:
            raise ValueError(f'mels must be [B, {self.feat}, T], got {m.shape}')
        B, _, T = m.shape
        S = T * self.hop
        labels = np.empty((B, S), dtype=np.int16) if want_labels else None
        wave = np.empty((B, (T - 1) * self.hop), dtype=np.float64) if want_wave else None
        rng = Rng()
        rng.mode = _lib.RNG_PHILOX
        rng.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        rng.utterance_offset = int(utterance_offset)
        opts = GenOpts()
        opts.kernel = _lib.KERNELS[kernel]
        opts.mu_law = 1 if mu_law else 0
        _lib.check(self.lib.b200tts_wavernn_generate_host(
            self._h, m.ctypes.data_as(C.c_void_p), B, T, C.byref(rng), C.byref(opts),
            labels.ctypes.data_as(C.c_void_p) if labels is not None else C.c_void_p(0),
            wave.ctypes.data_as(C.c_void_p) if wave is not None else C.c_void_p(0)))
        return dict(labels=labels, wave=wave)

    def philox_exponential(self, seed: int, utterance_offset: int, B: int, step0: int, n_steps: int):
        """The Exp(1) noise the PHILOX mode draws, [n_steps, B, NC] on the device (for parity tests)."""
        with torch.cuda.device(self.device):
            q = torch.empty(n_steps, B, self.n_classes, device=self._dev(), dtype=torch.float32)
            _lib.check(self.lib.b200tts_philox_exponential(self.device, int(seed) & 0xFFFFFFFFFFFFFFFF, int(utterance_offset),
                                                           B, step0, n_steps, self.n_classes, _ptr(q), self._stream()))
        return q

    def debug_phase_cycles(self):
        """[6][2] mean cycles (compute, barrier) per phase of the last grid launch; needs B200TTS_GRID_PROF=1."""
        out = (C.c_double * 12)()
        _lib.check(self.lib.b200tts_wavernn_debug_phase_cycles(self._h, out))
        return np.array(list(out)).reshape(6, 2)

    def check(self):
        """Synchronises and raises if the last generate call's persistent kernel gave up waiting for a peer thread block
        (its wave is NaN-filled in that case).  Call after the point where the caller synchronises anyway."""
        _lib.check(self.lib.b200tts_wavernn_check(self._h))

    def fp32_peak_tflops(self) -> float:
        """Measured fp32 CUDA-core ceiling of this device (register-only FFMA2 loop), TFLOP/s."""
        v = C.c_double()
        _lib.check(self.lib.b200tts_debug_fp32_peak(self.device, C.byref(v)))
        return float(v.value)

    @property
    def launch_count(self) -> int:
        return int(self.lib.b200tts_wavernn_launch_count(self._h))

    KERNEL_NAMES = {0: None, 1: 'wavernn_utt_kernel', 2: 'wavernn_grid_kernel', 3: 'wavernn_push_kernel', 4: 'wavernn_pushmg_kernel',
                    5: 'wavernn_tc_kernel'}

    def last_kernel(self):
        """Name of the step kernel the last generate call ran."""
        return self.KERNEL_NAMES.get(int(self.lib.b200tts_wavernn_last_kernel(self._h)))

    def last_kernel_ms(self) -> float:
        ms = float(self.lib.b200tts_wavernn_last_kernel_ms(self._h))
        if ms < 0:
            raise _lib.B200TTSError(-1, self.lib.b200tts_last_error().decode())
        return ms
