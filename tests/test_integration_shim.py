"""CPU: the binding INTEGRATION.md documents for a reference maintainer (section 1: register ctypes-backed stand-ins for the
two native extension modules before the reference is imported) is EXECUTED here -- the shim text is taken verbatim from the
document, and the calls the reference's own autograd Functions make into the two modules (selective_scan_fn forward and
backward, causal_conv1d_fn forward and backward, recorded from the unmodified reference by oracle/gen_golden_shim.py) are
replayed against it.  The CUDA-only raw ops the shim calls are replaced by CPU fakes built on the oracle, so what is verified
is the glue: module / function names, argument order, the layout of the returned lists, the state handed from fwd to bwd."""
import json
import sys

import torch

from oracle import gen_golden_shim as gs
from util import gold


def _replay(g):
    """Each recorded call on the registered module; an argument recorded as an element of an earlier result is that element."""
    results = []
    for call in json.loads(bytes(g["trace_json"]).decode()):
        args = []
        for kind, *ref in call["args"]:
            if kind == "arr":
                args.append(torch.from_numpy(g[ref[0]]))
            elif kind == "ret":
                args.append(results[ref[0]][ref[1]])
            else:
                args.append(ref[0])
        res = getattr(sys.modules[call["module"]], call["fn"])(*args)
        results.append(list(res) if isinstance(res, (list, tuple)) else [res])
    return results


def test_integration_md_shim_runs_under_the_reference_interfaces(monkeypatch):
    g = gold("integration_shim")
    saved_mods = {n: sys.modules.get(n) for n in gs.SHIM_MODULES}
    try:
        calls = gs.install_shim(monkeypatch.setattr)
        fwd, bwd, conv_fwd, conv_bwd = _replay(g)
    finally:
        for n, m in saved_mods.items():
            if m is None:
                sys.modules.pop(n, None)
            else:
                sys.modules[n] = m
    assert calls == ["scan_fwd", "scan_fwd", "scan_bwd", "conv_fwd", "conv_bwd"], calls
    want = lambda k: torch.from_numpy(g["want_" + k])

    # the reference reads `out, x, *rest = fwd(...)`, returns rest[0] (out_z) and x[:, :, -1, 1::2] as the last state
    # (selective_scan_interface.py:37-47); `du, ddelta, dA, dB, dC, dD, ddelta_bias, *rest = bwd(...)` with dz = rest[0] and
    # dB, dC squeezed back to the 3-D shape they came in (:62-68); against its own selective_scan_ref
    assert len(fwd) == 3
    assert torch.allclose(fwd[2], want("scan_out"), rtol=1e-4, atol=1e-5)
    assert torch.allclose(fwd[1][:, :, -1, 1::2], want("scan_last"), rtol=1e-4, atol=1e-5)
    du, ddelta, dA, dB, dC, dD, ddelta_bias, *rest = bwd
    got = dict(u=du, delta=ddelta, A=dA, B=dB.squeeze(1), C=dC.squeeze(1), D=dD, z=rest[0], delta_bias=ddelta_bias)
    for k in gs.SCAN_INPUTS:
        assert torch.allclose(got[k], want("scan_grad_" + k), rtol=1e-3, atol=1e-4), k

    # causal_conv1d_interface.py:20 returns the fwd result as is; :31 reads `dx, dweight, dbias = bwd(...)`; against causal_conv1d_ref
    assert torch.allclose(conv_fwd[0], want("conv_y"), atol=1e-6)
    assert len(conv_bwd) == 3
    for k, v in zip(("x", "w", "b"), conv_bwd):
        assert torch.allclose(v, want("conv_grad_" + k), atol=1e-5), k
