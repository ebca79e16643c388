"""oracle/restate_engine.py — TEST INFRASTRUCTURE, not product code.

`QEngineRestate` = the host-side QEngine mirror (qrack_b200.qengine.QEngineHost) over the plain-C restatement of
the reference's QEngineCPU sweeps (oracle/qengine_restate.c), state held in numpy arrays on the host.  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline leg import this module.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile
from ctypes import POINTER, c_double, c_int, c_uint64, c_void_p

import numpy as np

from qrack_b200.qengine import QEngineHost

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "liboracle_restate.so")
_lib = None


def build_restatement(force: bool = False) -> str:
    """Compile liboracle_restate.so next to its sources when it is missing or older than they are; in a temporary directory
    when the tree is read-only (bench.py's baseline leg may run from one)."""
    src = [os.path.join(_HERE, f) for f in ("qengine_restate.c", "qengine_restate_impl.h", "qalu_restate_impl.h")]
    if not force and os.path.exists(_LIB) and os.path.getmtime(_LIB) >= max(os.path.getmtime(s) for s in src):
        return _LIB
    out = _LIB if os.access(_HERE, os.W_OK) else os.path.join(tempfile.mkdtemp(prefix="oracle_restate_"), os.path.basename(_LIB))
    subprocess.run(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-fno-fast-math", "-ffp-contract=off", src[0], "-lm",
                    "-o", out], check=True)
    return out


def _load():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build_restatement())
        for suf in ("_f32", "_f64"):
            for name in ("orc_prob_mask", "orc_prob_parity", "orc_collapse_parity", "orc_norm", "orc_expectation"):
                getattr(_lib, name + suf).restype = c_double
    return _lib


class _RestateBackend:
    def __init__(self, n_qubits: int, precision: int):
        self.lib = _load()
        self.suf = "_f32" if precision == 32 else "_f64"
        self.precision = precision
        self.cplx = np.complex64 if precision == 32 else np.complex128
        self.real = np.float32 if precision == 32 else np.float64
        self.creal = ctypes.c_float if precision == 32 else ctypes.c_double
        self.nq = n_qubits
        self.amps = None  # None == the zero state (reference: null stateVec)

    def fn(self, name):
        return getattr(self.lib, name + self.suf)

    def _p(self, a=None):
        a = self.amps if a is None else a
        return a.ctypes.data_as(c_void_p)

    def _alloc(self):
        if self.amps is None:
            self.amps = np.zeros(1 << self.nq, dtype=self.cplx)

    def resize_zero(self, n):
        self.nq = n
        self.amps = None

    def finish(self):
        pass

    def is_zero(self):
        return self.amps is None

    def zero(self):
        self.amps = None

    def set_permutation(self, perm, phase):
        self.amps = np.zeros(1 << self.nq, dtype=self.cplx)
        self.amps[perm] = phase

    def set_state(self, arr):
        self.amps = np.array(arr, dtype=self.cplx, copy=True)

    def get_state(self):
        return np.zeros(1 << self.nq, dtype=self.cplx) if self.amps is None else self.amps.copy()

    def get_probs(self):
        s = self.get_state()
        return (s.real.astype(self.real) ** 2 + s.imag.astype(self.real) ** 2).astype(self.real)

    def get_page(self, off, length):
        return self.get_state()[off:off + length]

    def set_page(self, arr, off):
        self._alloc()
        self.amps[off:off + arr.size] = arr

    def copy_page(self, src, src_off, dst_off, length):
        if self.amps is None and src.amps is None:
            return
        if src.amps is None and length == (1 << self.nq):
            self.amps = None
            return
        self._alloc()
        self.amps[dst_off:dst_off + length] = 0 if src.amps is None else src.amps[src_off:src_off + length]

    def shuffle(self, other):
        if self.amps is None and other.amps is None:
            return
        self._alloc()
        other._alloc()
        self.fn("orc_shuffle")(self._p(), other._p(), c_int(self.nq))

    def copy_state(self, src):
        self.nq = src.nq
        self.amps = None if src.amps is None else src.amps.copy()

    def get_amplitude(self, perm):
        return 0j if self.amps is None else complex(self.amps[perm])

    def set_amplitude(self, perm, amp):
        self._alloc()
        self.amps[perm] = amp

    def apply2x2(self, off1, off2, mtrx, pows, nrm, thresh, calc_norm):
        m = (self.creal * 8)()
        for k in range(4):
            m[2 * k] = mtrx[k].real
            m[2 * k + 1] = mtrx[k].imag
        pw = (c_uint64 * max(len(pows), 1))(*pows)
        out = c_double()
        self.fn("orc_apply2x2")(self._p(), c_int(self.nq), c_uint64(off1), c_uint64(off2), m, c_int(len(pows)), pw,
                                self.creal(nrm), self.creal(thresh), ctypes.byref(out) if calc_norm else None)
        return out.value if calc_norm else None

    def apply_gates(self, n, off1, off2, pmasks, mats8):
        """same call shape as the CUDA backend's batched submission (b200sv_apply_gates): here simply gate by gate"""
        for i in range(n):
            pm = int(pmasks[i])
            pows = [1 << b for b in range(pm.bit_length()) if (pm >> b) & 1]
            m = [complex(mats8[8 * i + 2 * k], mats8[8 * i + 2 * k + 1]) for k in range(4)]
            if self.precision == 32:
                m = [complex(np.float32(z.real), np.float32(z.imag)) for z in m]
            self.apply2x2(int(off1[i]), int(off2[i]), m, pows, 1.0, 0.0, False)

    def xmask(self, mask):
        self.fn("orc_xmask")(self._p(), c_int(self.nq), c_uint64(mask))

    def phase_parity(self, radians, mask):
        ang = self.real(radians / 2)
        self.fn("orc_phase_parity")(self._p(), c_int(self.nq), c_uint64(0), c_uint64(mask), self.creal(np.cos(ang)),
                                    self.creal(np.sin(ang)))

    def uniform_parity_rz(self, cmask, mask, angle):
        self.fn("orc_phase_parity")(self._p(), c_int(self.nq), c_uint64(cmask), c_uint64(mask),
                                    self.creal(np.cos(angle)), self.creal(np.sin(angle)))

    def phase_root_n_mask(self, n, mask):
        self.fn("orc_phase_root_n_mask")(self._p(), c_int(self.nq), c_int(n), c_uint64(mask))

    def apply_m(self, mask, result, nrm):
        self.fn("orc_apply_m")(self._p(), c_int(self.nq), c_uint64(mask), c_uint64(result), self.creal(nrm.real),
                               self.creal(nrm.imag))

    def collapse_parity(self, mask, result):
        return self.fn("orc_collapse_parity")(self._p(), c_int(self.nq), c_uint64(mask), c_int(int(result)))

    def prob_mask(self, mask, perm):
        return self.fn("orc_prob_mask")(self._p(), c_int(self.nq), c_uint64(mask), c_uint64(perm))

    def prob_parity(self, mask):
        return self.fn("orc_prob_parity")(self._p(), c_int(self.nq), c_uint64(mask))

    def prob_mask_all(self, mask):
        bits = [b for b in range(self.nq) if (mask >> b) & 1]
        out = np.zeros(1 << len(bits), dtype=self.real)
        for k in range(out.size):
            perm = 0
            for j, b in enumerate(bits):
                if (k >> j) & 1:
                    perm |= 1 << b
            out[k] = self.prob_mask(mask, perm) if self.amps is not None else 0
        return out

    def norm(self, thresh):
        return self.fn("orc_norm")(self._p(), c_int(self.nq), self.creal(thresh))

    def normalize(self, nrm, thresh, phase_arg):
        self.fn("orc_normalize")(self._p(), c_int(self.nq), self.creal(nrm), self.creal(thresh), self.creal(phase_arg))

    def inner(self, other):
        re, im = c_double(), c_double()
        self.fn("orc_inner")(self._p(), other._p(), c_int(self.nq), ctypes.byref(re), ctypes.byref(im))
        return complex(re.value, im.value)

    def expectation(self, start, length):
        return self.fn("orc_expectation")(self._p(), c_int(self.nq), c_int(start), c_int(length))

    # ---- QAlu family (oracle/qalu_restate_impl.h); the zero state is left untouched (CHECK_ZERO_SKIP) ----
    def _alu(self, name, *args):
        if self.amps is not None:
            self.fn(name)(self._p(), c_int(self.nq), *args)

    def alu_rol(self, shift, start, length):
        self._alu("orc_rol", c_int(shift), c_int(start), c_int(length))

    def alu_inc(self, to_add, start, length, ctrl_mask):
        self._alu("orc_inc", c_uint64(to_add), c_int(start), c_int(length), c_uint64(ctrl_mask))

    def alu_incdecc(self, to_mod, start, length, carry_index):
        self._alu("orc_incdecc", c_uint64(to_mod), c_int(start), c_int(length), c_int(carry_index))

    def alu_incs(self, to_add, start, length, overflow_index):
        self._alu("orc_incs", c_uint64(to_add), c_int(start), c_int(length), c_int(overflow_index))

    def alu_incdecsc(self, to_mod, start, length, overflow_index, carry_index):
        self._alu("orc_incdecsc", c_uint64(to_mod), c_int(start), c_int(length), c_int(overflow_index), c_int(carry_index))

    def alu_muldiv(self, inverse, to_mul, start, carry_start, length, ctrl_mask):
        self._alu("orc_muldiv", c_int(inverse), c_uint64(to_mul), c_int(start), c_int(carry_start), c_int(length),
                  c_uint64(ctrl_mask))

    def alu_modnout(self, kind, to_mod, mod_n, in_start, out_start, length, ctrl_mask):
        self._alu("orc_modnout", c_int(kind), c_uint64(to_mod), c_uint64(mod_n), c_int(in_start), c_int(out_start),
                  c_int(length), c_uint64(ctrl_mask))

    def alu_indexed(self, kind, index_start, index_length, value_start, value_length, carry_index, carry_in, values: bytes):
        self._alu("orc_indexed", c_int(kind), c_int(index_start), c_int(index_length), c_int(value_start),
                  c_int(value_length), c_int(carry_index), c_int(carry_in), ctypes.c_char_p(values))

    def alu_hash(self, start, length, values: bytes):
        self._alu("orc_hash", c_int(start), c_int(length), ctypes.c_char_p(values))

    def alu_phase_flip_if_less(self, greater_perm, start, length, flag_index):
        self._alu("orc_phase_flip_if_less", c_uint64(greater_perm), c_int(start), c_int(length), c_int(flag_index))

    def highest_prob(self):
        return 0 if self.amps is None else int(np.argmax(np.abs(self.amps) ** 2))

    def sample(self, rnd):
        # QEngineCPU::MAll, reference state.cpp:2026-2050
        n = 1 << self.nq
        if self.amps is None:
            return n - 1
        eps = 1.7763568394002505e-15 if self.precision == 32 else 6.310887241768095e-30
        fpeps = float(np.finfo(self.real).eps) / 4
        tot = 0.0
        last = n - 1
        pr = self.get_probs()
        for i in range(n):
            if pr[i] > eps:
                tot += float(pr[i])
                if tot > rnd or (1.0 - tot) <= fpeps:
                    return i
                last = i
        return last

    def compose(self, other, start):
        nq = self.nq + other.nq
        if self.amps is None or other.amps is None:
            self.amps = None
            self.nq = nq
            return
        out = np.empty(1 << nq, dtype=self.cplx)
        self.fn("orc_compose")(self._p(out), self._p(), c_int(self.nq), other._p(), c_int(other.nq), c_int(start))
        self.amps = out
        self.nq = nq

    def decompose(self, start, length, dest):
        nl = self.nq - length
        if self.amps is None:
            self.nq = nl
            if dest is not None:
                dest.amps = None
            return
        if nl == 0:
            if dest is not None:
                dest.amps = self.amps
                dest.nq = length
            self.amps = None
            self.nq = 0
            return
        floorv = 1.7763568394002505e-15 if self.precision == 32 else 6.310887241768095e-30
        rem = np.empty(1 << nl, dtype=self.cplx)
        part = np.empty(1 << length, dtype=self.cplx) if dest is not None else None
        self.fn("orc_decompose")(self._p(), c_int(self.nq), c_int(start), c_int(length), self._p(rem),
                                 self._p(part) if part is not None else None, self.creal(floorv))
        if dest is not None:
            dest.amps = part
            dest.nq = length
        self.amps = rem
        self.nq = nl

    def dispose_perm(self, start, length, perm):
        nl = self.nq - length
        if self.amps is None:
            self.nq = nl
            return
        out = np.empty(1 << nl, dtype=self.cplx)
        self.fn("orc_dispose_perm")(self._p(out), self._p(), c_int(self.nq), c_int(start), c_int(length), c_uint64(perm))
        self.amps = out
        self.nq = nl


class QEngineRestate(QEngineHost):
    """QEngineCPU restated: reference dispatch (host mirror) + reference sweeps (C restatement)."""

    def _make_backend(self, n_qubits: int):
        return _RestateBackend(n_qubits, self.precision)
