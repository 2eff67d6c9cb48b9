"""ctypes binding of the C-ABI library (include/dsdf_b200.h).  No CPU fallback: a missing library is an error."""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libdsdf_b200.so')
_lib = None

c_p = ctypes.c_void_p
c_i = ctypes.c_int
c_d = ctypes.c_double
c_sz = ctypes.c_size_t
c_ll = ctypes.c_longlong

# name -> (restype, argtypes).  Must list every symbol include/dsdf_b200.h declares (tests/test_cabi.py checks).
SIGNATURES = {
    'dsdf_version': (c_i, []),
    'dsdf_lcp_workspace_bytes': (c_sz, [c_i, c_i, c_i, c_i]),
    'dsdf_lcp_smem_bytes': (c_sz, [c_i, c_i, c_i]),
    'dsdf_lcp_forward': (c_i, [c_p] * 8 + [c_i] * 5 + [c_d, c_i, c_i, c_i] + [c_p] * 8),
    'dsdf_lcp_backward': (c_i, [c_p] * 10 + [c_i] * 5 + [c_p] * 10),
    'dsdf_sdf_query': (c_i, [c_i, c_p, c_d, c_d, c_p, c_i, c_ll, c_p, c_i, c_i, c_i, c_p, c_p, c_p]),
    'dsdf_sdf_query_backward': (c_i, [c_i, c_p, c_d, c_d, c_p, c_i, c_ll, c_p, c_i, c_i, c_p, c_p, c_p, c_p]),
    'dsdf_integrate': (c_i, [c_p, c_p, c_p, c_p, c_i, c_i, c_p, c_p]),
    'dsdf_integrate_backward': (c_i, [c_p, c_p, c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_p]),
    'dsdf_contacts_detect': (c_i, [c_p, c_p, c_i, c_p, c_p, c_p, c_i, c_i, c_d, c_d, c_d, c_d, c_i, c_i, c_i]
                             + [c_p] * 11),
    'dsdf_contacts_phase_cycles': (c_i, [c_p, c_i]),
    'dsdf_dynamics_phase_cycles': (c_i, [c_p, c_i]),
    'dsdf_filter_contacts': (c_i, [c_p, c_p, c_p, c_i, c_i, c_d, c_p, c_p, c_p]),
    'dsdf_contact_geometry_backward': (c_i, [c_p, c_p, c_p, c_i, c_i, c_d, c_i, c_i] + [c_p] * 10),
    'dsdf_dynamics_assemble': (c_i, [c_p] * 12 + [c_i] * 4 + [c_p] * 7),
    'dsdf_dynamics_assemble_backward': (c_i, [c_p] * 12 + [c_i] * 6 + [c_p] * 17),
    'dsdf_dynamics_plan': (c_i, [c_i] * 7 + [c_p]),
    'dsdf_dynamics_solve': (c_i, [c_p] * 13 + [c_i] * 8 + [c_d, c_i, c_i] + [c_p] * 11),
    'dsdf_dynamics_solve_backward': (c_i, [c_p] * 13 + [c_i] * 10 + [c_p] * 15),
    'dsdf_toc_backward': (c_i, [c_i] * 3 + [c_p] * 9 + [c_d] + [c_p] * 7),
    'dsdf_attempt_commit': (c_i, [c_i] * 3 + [c_p] * 4 + [c_d, c_i, c_i] + [c_p] * 21),
    'dsdf_step_begin': (c_i, [c_p, c_p]),
    'dsdf_step_resume': (c_i, [c_p, c_p]),
    'dsdf_step_rounds': (c_i, [c_p, c_i, c_i, c_i, c_p]),
    'dsdf_step_profile': (c_i, [c_i]),
    'dsdf_step_profile_read': (c_i, [c_p, c_p]),
    'dsdf_fma_peaks': (c_i, [c_i, c_p, c_p, c_p, c_p]),
}


class DsdfLibraryError(RuntimeError):
    pass


def lib():
    """Load (once) the CUDA library; raise loudly if it is absent -- there is no other compute path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DsdfLibraryError(
                'libdsdf_b200.so not found at %s: build it with `python -m diffsdfsim_b200.build` '
                '(there is no CPU / PyTorch fallback for the stepping kernels)' % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


PROFILE = None      # set to {} to record (start, end) CUDA events around every entry-point call
LAUNCHES = {}       # name -> CUDA kernels its calls launched since reset_counters() (for bench.py's gpu_launches claim)


def reset_counters(profile=False):
    global PROFILE
    LAUNCHES.clear()
    PROFILE = {} if profile else None


def kernel_launches():
    return sum(LAUNCHES.values())


def call(name, *args, kernels=1):
    """Invoke an entry point of the library that launches ``kernels`` CUDA kernels (counted; optionally bracketed with
    CUDA events)."""
    fn = getattr(lib(), name)
    LAUNCHES[name] = LAUNCHES.get(name, 0) + kernels
    if PROFILE is None:
        return fn(*args)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    rc = fn(*args)
    e.record()
    PROFILE.setdefault(name, []).append((s, e))
    return rc


def profile_summary():
    """name -> (calls, total ms) from the recorded events (synchronises)."""
    torch.cuda.synchronize()
    return {k: (len(v), sum(s.elapsed_time(e) for s, e in v)) for k, v in (PROFILE or {}).items()}


def dynamics_plan(W, nb, neq, fric_dirs, ncontacts_small, ncontacts_large, force_cta=False):
    """(kernel launches, workspace bytes) of one dsdf_dynamics_solve / dsdf_dynamics_solve_backward call."""
    ws = ctypes.c_size_t(0)
    n = lib().dsdf_dynamics_plan(W, nb, neq, fric_dirs, ncontacts_small, ncontacts_large, int(force_cta),
                                 ctypes.byref(ws))
    if n == -2:
        raise DsdfLibraryError('world too large for the dynamics kernels: %d bodies' % nb)
    if n < 0:
        raise DsdfLibraryError('dsdf_dynamics_plan failed with status %d' % n)
    return n, ws.value


def ptr(t):
    """Device pointer of a tensor (None -> NULL).  Tensors must be contiguous."""
    if t is None:
        return None
    assert t.is_contiguous(), 'C ABI needs contiguous buffers'
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def check(rc, what):
    if rc != 0:
        if rc == -2:
            raise DsdfLibraryError('%s: problem too large for the shared-memory kernel' % what)
        raise DsdfLibraryError('%s failed with status %d' % (what, rc))


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise DsdfLibraryError('diffsdfsim_b200 kernels need CUDA tensors (got %s); there is no CPU fallback'
                                   % t.device)
