"""Shared by the top-K path tests: the plan query (`b200rec_debug_topk_plan`, a development entry point that the public
header does not declare) and a context manager that sets the library's development knobs for a block of code.

The library reads its knobs from the environment once per process; `topk_knobs` re-reads them on entry and again on
exit, after the environment is restored, so later tests in the same process see the default plans."""
import contextlib
import ctypes as C
import os

PLAN_KEYS = ("sms", "v2", "nq", "bn", "stages", "ks", "grid", "max_parts", "S", "T", "W", "R", "n_main", "Tmain", "Tt",
             "sample_m", "sample_gw", "cap", "flush")

KNOBS = ("B200REC_TOPK_V2", "B200REC_TOPK_NQ", "B200REC_TOPK_NOSAMPLE", "B200REC_SCHED")

# The instantiation the default plan picks on 148 SMs, by row width ld (bf16 elements) and query count.
# -ks1: the 2-CTA pair kernel with one 64-column atom per ring stage (odd ld / 64).
DEFAULT_MAP = {
    64: ("bn256", "pair1-ks1", "pair2-ks1"), 128: ("bn256", "pair1", "pair2"), 192: ("bn256", "pair1-ks1", "pair2-ks1"),
    256: ("bn256", "pair1", "pair2"), 320: ("bn256", "pair1-ks1", "pair2-ks1"), 384: ("bn256", "pair1", "pair1"),
    448: ("bn64", "pair1-ks1", "pair1-ks1"), 512: ("bn64", "bn64", "bn64"), 576: ("bn64", "pair1-ks1", "pair1-ks1"),
    640: ("bn64", "bn64", "bn64"), 704: ("bn64", "bn64", "bn64"),
}


def default_path(ld: int, q: int) -> str:
    """DEFAULT_MAP's cell for (ld, q): Q <= 128, 128 < Q <= 256, Q > 256."""
    return DEFAULT_MAP[ld][0 if q <= 128 else (1 if q <= 256 else 2)]


def _lib():
    from b200rec import _native
    lib = _native.lib()
    fn = lib.b200rec_debug_topk_plan
    fn.restype = C.c_int
    fn.argtypes = [C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_longlong), C.c_int]
    return lib


def plan(n: int, ld: int, q: int, k: int, shards: int = 1) -> dict:
    """The plan a search of (n, ld, q, k) runs with under the knobs in force; RuntimeError when there is none."""
    from b200rec import _native
    out = (C.c_longlong * len(PLAN_KEYS))()
    if _lib().b200rec_debug_topk_plan(n, ld, q, k, shards, out, len(PLAN_KEYS)) != 0:
        raise RuntimeError(_native.last_error())
    return dict(zip(PLAN_KEYS, out))


def path_name(p: dict) -> str:
    """Kernel instantiation of a plan: pair2 / pair1 (2-CTA kernel, NQ2 = 2 / 1, suffix -ks1 for one atom per stage),
    nq2bn128 (single-CTA NQ = 2, BN = 128), bn256 / bn64 (single-CTA NQ = 1)."""
    if p["v2"]:
        return f"pair{p['v2']}" + ("-ks1" if p["ks"] == 1 else "")
    return "nq2bn128" if p["nq"] == 2 else f"bn{p['bn']}"


def decomposition(p: dict) -> str:
    """Work split of a pair-kernel plan: 'contiguous' (no time-aligned sweep), 'aligned-idle' (leftover units idle or
    none left over) or 'aligned-working' (leftover units share the tail tiles)."""
    if p["n_main"] == 0:
        return "contiguous"
    return "aligned-working" if p["Tt"] > 0 else "aligned-idle"


def reload() -> None:
    _lib().b200rec_debug_reload_env()


@contextlib.contextmanager
def topk_knobs(**env):
    """Set development knobs (B200REC_* names, values str()-ed; None unsets) for the block; the environment and the
    library's knobs and plan cache are restored on exit, also when the block raises."""
    saved = {name: os.environ.get(name) for name in env}
    try:
        for name, value in env.items():
            if value is None:
                os.environ.pop(name, None)
            else:
                os.environ[name] = str(value)
        reload()
        yield
    finally:
        for name, value in saved.items():
            if value is None:
                os.environ.pop(name, None)
            else:
                os.environ[name] = value
        reload()
