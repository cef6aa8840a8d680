"""Shared by the loss path tests: the plan query (`b200rec_debug_loss_plan`, a development entry point that the public
header does not declare), which reports the forward log-sum-exp plan and the fused backward plan of an in-batch loss
shape without launching anything."""
import ctypes as C

LSE_KEYS = ("nq", "bn", "stages", "grid", "S", "T", "W", "max_parts")
GRAD_KEYS = ("supported", "smem", "NST", "units_u", "splits_u", "splits_v", "atomic_u", "atomic_v")
PLAN_KEYS = ("sms",) + tuple("lse_" + k for k in LSE_KEYS) + tuple("grad_" + k for k in GRAD_KEYS)


def pad64(n: int) -> int:
    return (n + 63) // 64 * 64


def _lib():
    from b200rec import _native
    lib = _native.lib()
    fn = lib.b200rec_debug_loss_plan
    fn.restype = C.c_int
    fn.argtypes = [C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_longlong), C.c_int]
    return lib


def plan(B: int, NI: int, ld: int = 0, E: int = 0, nprod_s: int = 0, nprod_g: int = 0) -> dict:
    """Both plans of an in-batch loss of B users against NI items: the forward on operands of row width ld (bf16
    elements), the backward at embedding width E with (nprod_s, nprod_g) piece products.  RuntimeError on bad sizes."""
    from b200rec import _native
    out = (C.c_longlong * len(PLAN_KEYS))()
    if _lib().b200rec_debug_loss_plan(B, NI, ld, E, nprod_s, nprod_g, out, len(PLAN_KEYS)) != 0:
        raise RuntimeError(_native.last_error())
    return dict(zip(PLAN_KEYS, out))


def lse_path(B: int, NI: int, ld: int) -> str:
    """Forward kernel of (B, NI, ld): stream_scores_kernel<NQ, BN, LseEpi> as 'nq{NQ}bn{BN}', or 'fallback' (the chunked
    GEMM + lse_rows_kernel)."""
    p = plan(B, NI, ld)
    return f"nq{p['lse_nq']}bn{p['lse_bn']}" if p["lse_nq"] else "fallback"


def grad_plan(B: int, NI: int, E: int, nprod_s: int, nprod_g: int) -> dict:
    """The fused backward's plan (keys without the grad_ prefix); supported == 0 means the chunked path."""
    p = plan(B, NI, 0, E, nprod_s, nprod_g)
    return {k: p["grad_" + k] for k in GRAD_KEYS}
