"""TEST INFRASTRUCTURE: load the CPU emulation build of the CUDA kernels (tests/emu/libdedalus_b200_emu.so)
and expose numpy-array wrappers with the same argument order as the C ABI.  Never imported by the product."""
import ctypes as C
import numpy as np
import pathlib, sys
ROOT = pathlib.Path(__file__).resolve().parents[2]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
from dedalus_b200 import lib as dlib
from dedalus_b200 import build as dbuild
from dedalus_b200.fftplan import HostPlan

_emu = None


def emu():
    global _emu
    if _emu is None:
        import fcntl
        # parallel test workers share one object directory: one builds, the others wait and then find it current
        with open(str(dbuild.EMU_LIB) + ".lock", "w") as lock:
            fcntl.flock(lock, fcntl.LOCK_EX)
            path = dbuild.build_emu()
        _emu = dlib.bind(path)
    return _emu


def ptr(a):
    if a is None:
        return None
    assert a.flags['C_CONTIGUOUS']
    return a.ctypes.data_as(C.c_void_p)


class EmuPlan:
    def __init__(self, n, kind):
        hp = HostPlan(n, kind)
        self.hp = hp
        self._keep = [np.ascontiguousarray(x) for x in (hp.tw, hp.twr, hp.twq, hp.perm, hp.iperm, hp.twn)]
        s = dlib.FftPlan()
        s.n, s.nc, s.half, s.nrad = hp.n, hp.nc, hp.half, len(hp.radices)
        for i, r in enumerate(hp.radices):
            s.rad[i] = r
        s.tw, s.twr, s.twq, s.perm, s.iperm, s.twn = [ptr(x) for x in self._keep]
        self.struct = s

    def ref(self):
        return C.byref(self.struct)


class EmuBackend:
    """TEST-ONLY stand-in for dedalus_b200.lib.CudaBackend: CPU tensors, no stream, the host build of the kernels."""

    def device(self):
        import torch
        return torch.device('cpu')

    def stream(self):
        return None

    def lib(self):
        return emu()

    def accepts(self, tensor):
        return True


_saved = None
_torch_saved = None


def _poison_uninitialised():
    """torch.empty / empty_like return NaN-filled floating tensors while the emulation is installed: freshly mapped host
    memory is usually zero, freshly allocated DEVICE memory is not -- code that relies on it must fail here too."""
    global _torch_saved
    import torch
    if _torch_saved is not None:
        return
    _torch_saved = (torch.empty, torch.empty_like)
    e, el = _torch_saved

    def empty(*a, **k):
        t = e(*a, **k)
        if t.is_floating_point() or t.is_complex():
            t.fill_(float('nan'))
        return t

    def empty_like(*a, **k):
        t = el(*a, **k)
        if t.is_floating_point() or t.is_complex():
            t.fill_(float('nan'))
        return t
    torch.empty, torch.empty_like = empty, empty_like


def install():
    """Route the product's C-ABI calls to the emulated kernels (CPU tensors). Test-only: swaps the backend object."""
    global _saved
    if _saved is None:
        _saved = dlib._BACKEND
    dlib._BACKEND = EmuBackend()
    _poison_uninitialised()


def uninstall():
    global _saved, _torch_saved
    if _saved is not None:
        dlib._BACKEND = _saved
        _saved = None
    if _torch_saved is not None:
        import torch
        torch.empty, torch.empty_like = _torch_saved
        _torch_saved = None
