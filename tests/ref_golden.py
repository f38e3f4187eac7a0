"""The reference's kernels as the pin tests call them, without the reference.

``oracle.ref`` (oracle/_ref/liboracle_ref.so) is compiled from the reference's own sources, which a checkout of this
project does not carry.  What the tests asked of it is stored in tests/golden/ref_calls.npz: every call is keyed by a
digest of its method name, its arguments and (for the stateful multicorrelator) the state it was made in, and maps to
the outputs the reference returned.  ``Replay`` answers the same calls from that file; ``Recorder`` wraps the live
library and writes the file (tests/golden/make_golden.py runs the pin tests through it).

Outputs of more than ``INLINE_MAX`` elements are stored as a SHA-256 digest of their bytes (``Digest``): the tests
compare those bit for bit, and equal digests are equal bits.
"""
from __future__ import annotations

import hashlib
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_calls.npz")
INLINE_MAX = 256


class Digest:
    """Shape, dtype and SHA-256 of an array too large to store."""

    def __init__(self, shape, dtype, sha):
        self.shape, self.dtype, self.sha = tuple(shape), np.dtype(dtype), bytes(sha)

    @staticmethod
    def of(a) -> "Digest":
        a = np.ascontiguousarray(a)
        return Digest(a.shape, a.dtype, hashlib.sha256(a.tobytes()).digest())

    def __repr__(self):
        return f"Digest(shape={self.shape}, dtype={self.dtype}, sha256={self.sha.hex()[:16]}...)"


def same_bits(a, b) -> bool:
    """Bit-for-bit equality of two arrays, either of which may be a stored ``Digest``."""
    if isinstance(a, Digest) or isinstance(b, Digest):
        da = a if isinstance(a, Digest) else Digest.of(a)
        db = b if isinstance(b, Digest) else Digest.of(b)
        return da.shape == db.shape and da.dtype.itemsize == db.dtype.itemsize and da.sha == db.sha
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype.itemsize == b.dtype.itemsize and a.tobytes() == b.tobytes()


def _key(method, args, state=()):
    h = hashlib.sha1(method.encode())
    for x in tuple(state) + tuple(args):
        if isinstance(x, str):
            h.update(b"s" + x.encode())
            continue
        a = np.asarray(x)
        h.update(a.dtype.str.encode() + repr(a.shape).encode() + np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


class _Calls:
    """The ``oracle.ref`` methods the tests use; ``_answer(method, args, state, compute)`` supplies the outputs."""

    def __init__(self):
        self.arch = "a_avx"

    def select_arch(self, arch: str):
        self.arch = arch

    def resampler(self, variant, code, rem, step, shifts, n):
        return self._answer("resampler", (variant, _f32(code), rem, step, _f32(shifts), n))

    def hd_resampler(self, variant, code, rem, step, rate, shifts, n):
        return self._answer("hd_resampler", (variant, _f32(code), rem, step, rate, _f32(shifts), n))

    def rotator(self, variant, iq, phase_inc, phase, codes):
        return self._answer("rotator", (variant, _c64(iq), np.complex64(phase_inc), np.complex64(phase), _f32(codes)))

    def hd_rotator(self, variant, iq, phase_inc, phase_inc_rate, phase, codes):
        return self._answer("hd_rotator", (variant, _c64(iq), np.complex64(phase_inc), np.complex64(phase_inc_rate),
                                           np.complex64(phase), _f32(codes)))

    def sincos(self, variant, phase_inc, phase, n):
        return self._answer("sincos", (variant, np.float32(phase_inc), np.float32(phase), n))

    def index_max(self, variant, src):
        return self._answer("index_max", (variant, _f32(src)))

    # Cpu_Multicorrelator_Real_Codes: the handle carries what the correlate call depends on
    def mc_create(self, max_len, taps, high_dyn=False):
        return {"create": (max_len, taps, int(high_dyn))}

    def mc_set_code(self, h, code, shifts):
        h["code"] = (_f32(code), _f32(shifts))

    def mc_correlate(self, h, iq, taps, rem_carr, phase_step, phase_rate, rem_code, code_step, code_rate, n=None):
        iq = _c64(iq)
        n = len(iq) if n is None else n
        state = (self.arch,) + h["create"] + h["code"]
        return self._answer("mc_correlate", (iq[:n], taps, np.float32(rem_carr), np.float32(phase_step), np.float32(phase_rate),
                                             np.float32(rem_code), np.float32(code_step), np.float32(code_rate), n), state, h)

    def mc_destroy(self, h):
        pass


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _c64(a):
    return np.ascontiguousarray(a, dtype=np.complex64)


class Replay(_Calls):
    def __init__(self, path=GOLDEN):
        super().__init__()
        self.z = np.load(path)

    def _answer(self, method, args, state=(), h=None):
        k = _key(method, args, state)
        if f"{k}/n" not in self.z:
            raise KeyError(f"no stored reference output for this {method} call (re-run tests/golden/make_golden.py)")
        out = []
        for i in range(int(self.z[f"{k}/n"])):
            if f"{k}/{i}/sha" in self.z:
                out.append(Digest(self.z[f"{k}/{i}/shape"], str(self.z[f"{k}/{i}/dtype"]), self.z[f"{k}/{i}/sha"].tobytes()))
            else:
                v = self.z[f"{k}/{i}"]
                out.append(v[()] if v.ndim == 0 else v)
        return out[0] if int(self.z[f"{k}/single"]) else tuple(out)


class Recorder(_Calls):
    """Calls the live ``oracle.ref`` and keeps every answer; ``save()`` writes them."""

    def __init__(self, live, path=GOLDEN):
        super().__init__()
        self.live, self.path, self.rec = live, path, {}

    def select_arch(self, arch: str):
        super().select_arch(arch)
        self.live.select_arch(arch)

    def _answer(self, method, args, state=(), h=None):
        if method == "mc_correlate":
            (max_len, taps, hd), (code, shifts) = h["create"], h["code"]
            live = self.live.mc_create(max_len, taps, bool(hd))
            self.live.mc_set_code(live, code, shifts)
            res = self.live.mc_correlate(live, *args)
            self.live.mc_destroy(live)
        else:
            res = getattr(self.live, method)(*args)
        k = _key(method, args, state)
        single = not isinstance(res, tuple)
        outs = (res,) if single else res
        self.rec[f"{k}/n"] = np.array(len(outs))
        self.rec[f"{k}/single"] = np.array(int(single))
        for i, v in enumerate(outs):
            v = np.asarray(v)
            if v.size > INLINE_MAX:
                d = Digest.of(v)
                self.rec[f"{k}/{i}/sha"] = np.frombuffer(d.sha, np.uint8)
                self.rec[f"{k}/{i}/shape"] = np.array(d.shape, np.int64)
                self.rec[f"{k}/{i}/dtype"] = np.array(d.dtype.str)
            else:
                self.rec[f"{k}/{i}"] = v
        return res

    def save(self):
        np.savez_compressed(self.path, **self.rec)


def session_ref():
    """What the ``ref`` fixture hands out: a Recorder when B200_RECORD_REF_CALLS is set (make_golden.py), else a Replay."""
    if os.environ.get("B200_RECORD_REF_CALLS"):
        import atexit
        import oracle
        if oracle.ref is None:
            raise RuntimeError("recording needs oracle/_ref/liboracle_ref.so")
        r = Recorder(oracle.ref)
        atexit.register(r.save)
        return r
    return Replay()
