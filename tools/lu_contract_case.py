"""Factors the matrices of an .npz file with the dense LU entry points in a fresh process.

    python tools/lu_contract_case.py IN.npz OUT.npz

The LU schedule switches (SCB_LU_Q, SCB_LU_LAT, ... DESIGN.md section 6) are read once per process, so
tests/test_dense_lu_contract.py runs one worker per setting with the switch in its environment.  IN.npz
holds ``a<i>`` (n_pad x n_pad float64, row-major) and ``kind<i>`` ("sym", "gen" or "piv") for i = 0 ..
count - 1.  OUT.npz receives per case ``lu<i>`` (the factored workspace), ``dinv<i>`` (the block
inverses, [nb][2][128][128]), ``info<i>`` and, for "piv", ``piv<i>`` and ``perm<i>``.  Each matrix gets
buffers of its own and is factored twice through them; the second result is kept (for n_pad <= 12288 the
unpivoted LU captures its second call into a CUDA graph unless SCB_LU_GRAPH=0).  Nothing is left running
when it returns.
"""
from __future__ import annotations

import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def main(src: str, dst: str) -> None:
    import numpy as np
    import torch

    from superscreen_b200 import _lib

    L = _lib.lib()
    cases = np.load(src)
    out = {}
    count = sum(1 for k in cases.files if k.startswith("a"))
    for i in range(count):
        kind = str(cases[f"kind{i}"])
        A = cases[f"a{i}"]
        n_pad = A.shape[0]
        A_dev = torch.tensor(A).cuda()
        M = torch.empty_like(A_dev)
        dinv = torch.zeros(int(L.scb_getrf_dinv_bytes(n_pad)) // 8, dtype=torch.float64, device="cuda")
        info = torch.zeros(1, dtype=torch.int32, device="cuda")
        piv = torch.empty(n_pad, dtype=torch.int32, device="cuda")
        perm = torch.empty(n_pad, dtype=torch.int32, device="cuda")
        for _ in range(2):
            M.copy_(A_dev)
            sp = _lib.stream_ptr()
            if kind == "piv":
                _lib.check(L.scb_getrf_piv(n_pad, _lib.ptr(M), _lib.ptr(dinv), _lib.ptr(piv), _lib.ptr(perm),
                                           _lib.ptr(info), sp))
            else:
                getrf = L.scb_getrf_sym_nopiv if kind == "sym" else L.scb_getrf_nopiv
                _lib.check(getrf(n_pad, _lib.ptr(M), _lib.ptr(dinv), _lib.ptr(info), sp))
        torch.cuda.synchronize()
        if kind == "piv":
            out[f"piv{i}"] = piv.cpu().numpy()
            out[f"perm{i}"] = perm.cpu().numpy()
        nb = n_pad // 128
        out[f"lu{i}"] = M.cpu().numpy()
        out[f"dinv{i}"] = dinv[: nb * 2 * 128 * 128].cpu().numpy().reshape(nb, 2, 128, 128)
        out[f"info{i}"] = np.int32(info.item())
    np.savez(dst, **out)


if __name__ == "__main__":
    if len(sys.argv) != 3:
        sys.exit(__doc__)
    main(sys.argv[1], sys.argv[2])
