"""TEST INFRASTRUCTURE ONLY: `hqq_b200_reload_env()` on the emulated library -- the HQQ_B200_* knobs are cached per process and
parsed again only after a reload.  Observable without a GPU: HQQ_B200_DECODE1=0 removes the one-token kernel, and with it the fused
activation prologues (`hqq_b200_decode_linear_fwd` with x_op != 0 answers HQQ_E_UNSUPPORTED).  Prints one JSON line."""
import ctypes
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import build_emu  # noqa: E402
from run_small import F16, P, aligned, dev, make_layer  # noqa: E402


def main():
    for k in [k for k in os.environ if k.startswith("HQQ_B200_")]:
        del os.environ[k]
    lib = ctypes.CDLL(build_emu.build())
    lib.hqq_b200_last_error.restype = ctypes.c_char_p
    i64, VP = ctypes.c_int64, ctypes.c_void_p
    rng = np.random.default_rng(7)
    N, K, nbits = 64, 1024, 4
    A, B = make_layer(rng, N, K, nbits, 64), make_layer(rng, N, K, nbits, 64)
    xd, x2d = dev(rng.standard_normal((1, K)).astype(np.float16)), dev((rng.standard_normal((1, K)) * 0.5).astype(np.float16))
    arr = lambda vals: (VP * 2)(*[v.ctypes.data if v is not None else None for v in vals])  # noqa: E731
    Ns = (i64 * 2)(N, N)

    def call():
        ya, yb = aligned((1, N), np.float16), aligned((1, N), np.float16)
        rc = lib.hqq_b200_decode_linear_fwd(P(xd), 2, P(x2d), None, None, ctypes.c_float(1e-5), 2, arr([A["Wq"], B["Wq"]]),
                                            arr([A["scale"], B["scale"]]), arr([A["zero"], B["zero"]]), arr([None, None]), arr([ya, yb]), Ns,
                                            i64(K), 64, nbits, F16, None)
        return rc, np.concatenate([ya, yb]).tobytes()

    out = {}
    rc0, y0 = call()
    out["default_rc"] = rc0
    os.environ["HQQ_B200_DECODE1"] = "0"
    rc, y = call()
    out["cached_rc"], out["cached_same"] = rc, y == y0          # knob changed, no reload: still the cached choice
    lib.hqq_b200_reload_env()
    out["reloaded_rc"] = call()[0]                               # one-token kernel switched off -> prologue unsupported
    del os.environ["HQQ_B200_DECODE1"]
    lib.hqq_b200_reload_env()
    rc, y = call()
    out["restored_rc"], out["restored_same"] = rc, y == y0
    print("RELOAD " + json.dumps(out))


if __name__ == "__main__":
    main()
