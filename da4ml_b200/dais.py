"""Complete DAIS interpreter on the GPU: run any program of the reference's ``DAISInterpreter`` -- every opcode, lookup
tables included -- bit-identically, with the program loaded once and kept on the device.

    prog = DaisProgram(comb)          # a CombLogic (anything with .to_binary()), int32 words, or a path to a .bin file
    y = prog.predict(x)               # float64 numpy [n, n_in] -> numpy [n, n_out]; a CUDA float64 tensor -> CUDA tensor
    p = prog.profile(x)               # per op: value range, samples outside the declared dtype, samples wrapped
    v = prog.values(x, [3, 17])       # raw int64 values of ops 3 and 17: [n, 2], numpy or CUDA as x

``run_interp(bin_logic, data, n_threads=1)`` has the signature of the reference's ``dais_bin.run_interp``.
"""

from __future__ import annotations

import ctypes as C
import os
from typing import NamedTuple

import numpy as np

from . import _binary as B

INFO_FIELDS = ['n_in', 'n_out', 'n_ops', 'n_tables', 'n_slots', 'regime', 'tile', 'max_width']


class DaisProfile(NamedTuple):
    """What ``DaisProgram.profile`` found over ``n`` samples, per op (arrays of ``n_ops``):

    min, max        int64 extremes of the op's value, in units of 2^-fractionals (INT64_MAX / INT64_MIN when n = 0)
    outside         samples whose value lies outside the declared dtype's range (w = is_signed + integers + fractionals:
                    w <= 0 holds only 0, w >= 64 is unbounded); an op that does not quantize must never be outside
    wrapped         for the wrapping ops (-1, +-2, +-3, +-6): samples whose value the wrap step changed; 0 elsewhere
    first_outside   (sample, op) of the first value outside its range, sample order first; (-1, -1) when none
    width_declared  w of the declared dtype
    width_needed    the smallest width, signed or unsigned at the op's own fractional bits, that holds [min, max]
    """

    n: int
    min: np.ndarray
    max: np.ndarray
    outside: np.ndarray
    wrapped: np.ndarray
    first_outside: tuple
    width_declared: np.ndarray
    width_needed: np.ndarray


def _bit_length(v: np.ndarray) -> np.ndarray:
    """Bit length of non-negative int64 values."""
    return ((v[:, None] >> np.arange(64, dtype=np.int64)) != 0).sum(axis=1).astype(np.int64)


def width_needed(lo: np.ndarray, hi: np.ndarray) -> np.ndarray:
    """Smallest width that holds [lo, hi]: unsigned when lo >= 0, two's complement otherwise; 0 for an empty range."""
    lo, hi = np.asarray(lo, np.int64), np.asarray(hi, np.int64)
    unsigned = _bit_length(np.maximum(hi, 0))
    signed = 1 + np.maximum(_bit_length(np.maximum(hi, 0)), _bit_length(~np.minimum(lo, -1)))
    return np.where(lo > hi, 0, np.where(lo >= 0, unsigned, signed))


def _words(program) -> np.ndarray:
    if hasattr(program, 'to_binary'):
        program = program.to_binary()
    elif isinstance(program, (str, os.PathLike)):
        program = np.fromfile(program, dtype=np.int32)
    return np.ascontiguousarray(np.ravel(np.asarray(program)), dtype=np.int32)


def set_shared_budget(shared_bytes: int = 0, chunk_samples: int = 0):
    """Development switch for programs loaded afterwards: shared memory one CTA's value slots may use (a budget below
    32 samples' worth selects the global-memory regime) and samples per launch; 0 = automatic."""
    B._L.da4ml_dais_set_shared_budget(int(shared_bytes), int(chunk_samples))


class DaisProgram:
    """A DAIS program validated, compiled and resident on the current CUDA device."""

    def __init__(self, program):
        words = _words(program)
        h = B._vp()
        B._check(B._L.da4ml_dais_load(words.ctypes.data_as(B._i32p), words.size, C.byref(h)))
        self._h = h
        self._words = words
        out = np.zeros(8, np.int64)
        B._check(B._L.da4ml_dais_info(h, B._ip(out)))
        self.info = {k: int(v) for k, v in zip(INFO_FIELDS, out)}
        self.info['regime'] = 'shared' if self.info['regime'] == 0 else 'global'

    def __del__(self):
        h = getattr(self, '_h', None)
        if h:
            B._L.da4ml_dais_free(h)
            self._h = None

    @property
    def n_in(self) -> int:
        return self.info['n_in']

    @property
    def n_out(self) -> int:
        return self.info['n_out']

    @property
    def n_ops(self) -> int:
        return self.info['n_ops']

    @property
    def dtypes(self) -> np.ndarray:
        """[n_ops, 3] int64: (is_signed, integers, fractionals) of every op, from the program words."""
        w = self._words
        start = 6 + self.n_in + 3 * self.n_out
        return w[start : start + 8 * self.n_ops].reshape(-1, 8)[:, 5:8].astype(np.int64)

    def profile(self, x) -> DaisProfile:
        """Value ranges, out-of-range and wrap counts of every op over the samples (rows) of ``x``, computed on the GPU
        in one pass; ``x`` as for ``predict``.  A lookup index out of range raises the reference's error."""
        n_ops = self.n_ops
        stats = np.zeros((4, n_ops), np.int64)
        first = np.zeros(2, np.int64)
        if _is_cuda(x):
            xs = self._tensor_input(x)
            n = self._n_samples(xs.numel())
            with _on_stream(xs):
                B._check(B._L.da4ml_dais_profile_device(self._h, xs.data_ptr(), n, B._ip(stats), B._ip(first)))
        else:
            xs = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
            n = self._n_samples(xs.size)
            B._check(B._L.da4ml_dais_profile(self._h, xs.ctypes.data, n, B._ip(stats), B._ip(first)))
        dt = self.dtypes
        return DaisProfile(n=n, min=stats[0], max=stats[1], outside=stats[2], wrapped=stats[3], first_outside=(int(first[0]), int(first[1])),
                           width_declared=dt.sum(axis=1), width_needed=width_needed(stats[0], stats[1]))  # fmt: skip

    def values(self, x, ops):
        """Raw int64 values (the reference interpreter's ``buffer[op]``) of the ops listed in ``ops`` for every sample of
        ``x``: ``[n, len(ops)]``, a numpy array for host input and a CUDA tensor for a CUDA tensor.  Duplicates are
        allowed; an index outside ``[0, n_ops)`` raises ValueError."""
        idx = np.asarray(ops)
        if idx.ndim != 1 or (idx.size and idx.dtype.kind not in 'iu'):
            raise ValueError('ops must be a 1-D sequence of op indices')
        bad = idx[(idx < 0) | (idx >= self.n_ops)]
        if bad.size:
            raise ValueError(f'op index {int(bad[0])} out of range [0, {self.n_ops})')
        idx = np.ascontiguousarray(idx, np.int32)
        k = idx.size
        if _is_cuda(x):
            import torch

            xs = self._tensor_input(x)
            n = self._n_samples(xs.numel())
            out = torch.empty((n, k), dtype=torch.int64, device=xs.device)
            with _on_stream(xs):
                B._check(B._L.da4ml_dais_capture_device(self._h, xs.data_ptr(), n, idx.ctypes.data_as(B._i32p), k, out.data_ptr()))
            return out
        xs = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
        n = self._n_samples(xs.size)
        out = np.zeros((n, k), np.int64)
        B._check(B._L.da4ml_dais_capture(self._h, xs.ctypes.data, n, idx.ctypes.data_as(B._i32p), k, out.ctypes.data))
        return out

    def predict(self, x, n_threads: int = 1):
        """Outputs for every sample (row) of ``x``; ``n_threads`` is accepted for signature compatibility.  A CUDA tensor
        (float64, on the device the program was loaded on) is processed in place on the GPU on torch's current stream
        and the result is a CUDA tensor; anything else goes through float64 numpy."""
        if type(x).__module__.startswith('torch') and getattr(x, 'is_cuda', False):
            return self._predict_tensor(x)
        xs = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
        n = self._n_samples(xs.size)
        y = np.zeros((n, self.n_out), np.float64)
        B._check(B._L.da4ml_dais_infer(self._h, xs.ctypes.data, n, y.ctypes.data))
        return y

    def _n_samples(self, size: int) -> int:
        if self.n_in == 0:
            return 0
        if size % self.n_in:
            raise ValueError(f'Input size {size} is not divisible by {self.n_in}')
        return size // self.n_in

    def _tensor_input(self, x):
        import torch

        if x.dtype != torch.float64:
            raise TypeError('a CUDA input must be a float64 tensor')
        return x.contiguous()

    def _predict_tensor(self, x):
        import torch

        if x.dtype != torch.float64:
            raise TypeError('a CUDA input must be a float64 tensor')
        xs = x.contiguous()
        n = self._n_samples(xs.numel())
        y = torch.empty((n, self.n_out), dtype=torch.float64, device=xs.device)
        with torch.cuda.device(xs.device):
            B.set_stream(torch.cuda.current_stream().cuda_stream)
            B._check(B._L.da4ml_dais_infer_device(self._h, xs.data_ptr(), n, y.data_ptr()))
        return y


def _is_cuda(x) -> bool:
    return type(x).__module__.startswith('torch') and getattr(x, 'is_cuda', False)


class _on_stream:
    """torch's current device and stream of a CUDA tensor, made the library's for the duration of a call."""

    def __init__(self, xs):
        import torch

        self._dev = torch.cuda.device(xs.device)
        self._torch = torch

    def __enter__(self):
        self._dev.__enter__()
        B.set_stream(self._torch.cuda.current_stream().cuda_stream)

    def __exit__(self, *exc):
        return self._dev.__exit__(*exc)


def run_interp(bin_logic, data, n_threads: int = 1):
    """The reference's ``dais_bin.run_interp(bin_logic, data, n_threads=1)``: float64 ``[n_samples, n_out]``."""
    return DaisProgram(bin_logic).predict(data, n_threads)


__all__ = ['DaisProfile', 'DaisProgram', 'run_interp', 'set_shared_budget', 'width_needed']
