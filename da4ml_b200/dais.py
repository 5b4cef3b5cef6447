"""Complete DAIS interpreter on the GPU: run any program of the reference's ``DAISInterpreter`` -- every opcode, lookup
tables included -- bit-identically, with the program loaded once and kept on the device.

    prog = DaisProgram(comb)          # a CombLogic (anything with .to_binary()), int32 words, or a path to a .bin file
    y = prog.predict(x)               # float64 numpy [n, n_in] -> numpy [n, n_out]; a CUDA float64 tensor -> CUDA tensor

``run_interp(bin_logic, data, n_threads=1)`` has the signature of the reference's ``dais_bin.run_interp``.
"""

from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _binary as B

INFO_FIELDS = ['n_in', 'n_out', 'n_ops', 'n_tables', 'n_slots', 'regime', 'tile', 'max_width']


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


def run_interp(bin_logic, data, n_threads: int = 1):
    """The reference's ``dais_bin.run_interp(bin_logic, data, n_threads=1)``: float64 ``[n_samples, n_out]``."""
    return DaisProgram(bin_logic).predict(data, n_threads)


__all__ = ['DaisProgram', 'run_interp', 'set_shared_budget']
