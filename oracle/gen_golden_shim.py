"""TEST INFRASTRUCTURE ONLY -- golden call trace for tests/test_integration_shim.py.

Registers the two shim modules of INTEGRATION.md section 1 (their raw ops replaced by CPU stand-ins built on the
oracle), loads the UNMODIFIED reference ``selective_scan_interface.py`` and ``causal_conv1d`` package on top of them
(build container only), runs the reference's autograd Functions forward and backward, and records every call they make
into ``selective_scan_cuda`` / ``causal_conv1d_cuda``: the function name and each positional argument, either by value
or as an element of what an earlier call returned.  Next to the trace it stores the reference's own pure-PyTorch results
for the same inputs (``selective_scan_ref``, ``causal_conv1d_ref``, outputs and gradients), after checking that the
reference's Functions running through the shim reproduce them.  Writes tests/golden/integration_shim.npz; the test
replays the recorded calls against the shim and compares what comes back with those results.

    python oracle/gen_golden_shim.py
"""
import importlib.util
import json
import os
import re
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF_ROOT = os.environ.get("ZIGMA_REFERENCE_ROOT", "/root/reference")
GOLD = os.path.join(ROOT, "tests", "golden", "integration_shim.npz")

# modules the shim registers, and the reference's modules loaded on top of it (restored afterwards)
SHIM_MODULES = ["selective_scan_cuda", "causal_conv1d_cuda", "causal_conv1d", "causal_conv1d.causal_conv1d_interface",
                "_ref_ssi_under_shim"]
SCAN_INPUTS = ("u", "delta", "A", "B", "C", "D", "z", "delta_bias")
BT, E, L, N = 2, 6, 24, 4


def shim_text():
    """The shim module exactly as INTEGRATION.md prints it."""
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    blocks = re.findall(r"```python\n(.*?)```", text, flags=re.S)
    return next(b for b in blocks if "zigma_shims.py" in b)


def install_shim(setattr_):
    """Replaces the raw ops the shim calls by CPU stand-ins (through `setattr_`, e.g. pytest's monkeypatch.setattr),
    executes the shim text and returns the list the stand-ins append their names to."""
    from oracle import zigma_oracle as zo
    import zigma_b200.causal_conv1d_interface as zci
    import zigma_b200.selective_scan_interface as zsi
    calls = []

    def fake_scan_fwd(u, delta, A, B, C, D=None, z=None, delta_bias=None, delta_softplus=False, z_rowmap=None,
                      want_last_state=True, want_ckpt=False, out=None, dt_proj=None):
        calls.append("scan_fwd")
        o, last = zo.selective_scan(u, delta, A, B[:, 0] if B.dim() == 4 else B, C[:, 0] if C.dim() == 4 else C, D, z, delta_bias,
                                    delta_softplus, return_last_state=True)
        return o, (last if want_last_state else None), ("CKPT" if want_ckpt else None), (u, delta, z, B, C, D, delta_bias, A)

    def fake_scan_bwd(saved, ckpt, dout, delta_softplus, dz_out=None, z_rowmap=None):
        calls.append("scan_bwd")
        assert ckpt == "CKPT", "the checkpoint object of the forward must reach the backward"
        u, delta, z, B, C, D, delta_bias, A = saved
        leaves = [t.detach().clone().requires_grad_() if t is not None else None for t in (u, delta, A, B, C, D, delta_bias, z)]
        lu, ld, lA, lB, lC, lD, lb, lz = leaves
        with torch.enable_grad():      # (called from inside an autograd Function's backward: grad mode is off there)
            o = zo.selective_scan(lu, ld, lA, lB[:, 0], lC[:, 0], lD, lz, lb, delta_softplus)
        o.backward(dout)
        g = lambda t: None if t is None else t.grad
        return g(lu), g(ld), g(lA), g(lB), g(lC), g(lD), g(lb), g(lz)

    def fake_conv_fwd(x, w, b, silu, x_rowmap=None, out=None):
        calls.append("conv_fwd")
        return zo.causal_conv1d(x, w, b, "silu" if silu else None)

    def fake_conv_bwd(x, w, b, dout, silu, dx_out=None, x_rowmap=None):
        calls.append("conv_bwd")
        lx, lw = x.detach().clone().requires_grad_(), w.detach().clone().requires_grad_()
        lb = None if b is None else b.detach().clone().requires_grad_()
        with torch.enable_grad():
            yy = zo.causal_conv1d(lx, lw, lb, "silu" if silu else None)
        yy.backward(dout)
        return lx.grad, lw.grad, None if lb is None else lb.grad

    setattr_(zsi, "_scan_fwd", fake_scan_fwd)
    setattr_(zsi, "_scan_bwd", fake_scan_bwd)
    setattr_(zci, "_conv_fwd", fake_conv_fwd)
    setattr_(zci, "_conv_bwd", fake_conv_bwd)
    exec(compile(shim_text(), "INTEGRATION.md:zigma_shims.py", "exec"), {"__name__": "zigma_shims"})
    assert "selective_scan_cuda" in sys.modules and "causal_conv1d_cuda" in sys.modules
    return calls


def inputs():
    torch.manual_seed(0)
    mk = lambda *s: torch.randn(*s, dtype=torch.float32)
    scan = dict(u=mk(BT, E, L), delta=0.5 * torch.rand(BT, E, L), A=-torch.rand(E, N) - 0.1, B=mk(BT, N, L), C=mk(BT, N, L), D=mk(E),
                z=mk(BT, E, L), delta_bias=0.3 * mk(E))
    conv = dict(x=mk(BT, E, L), w=mk(E, 4), b=mk(E))
    return scan, conv


def run_scan(fn, base):
    """`fn` (the reference's selective_scan_fn or selective_scan_ref) forward and backward of sum(out^2)."""
    a = {k: v.clone().requires_grad_() for k, v in base.items()}
    out, last = fn(*(a[k] for k in SCAN_INPUTS[:6]), z=a["z"], delta_bias=a["delta_bias"], delta_softplus=True, return_last_state=True)
    out.square().sum().backward()
    return out.detach(), last.detach(), {k: v.grad for k, v in a.items()}


def run_conv(fn, base):
    """`fn` (the reference's causal_conv1d_fn or causal_conv1d_ref) with SiLU, forward and backward of sum(y)."""
    x, w, b = (base[k].clone().requires_grad_() for k in ("x", "w", "b"))
    y = fn(x, w, b, "silu")
    y.sum().backward()
    return y.detach(), {"x": x.grad, "w": w.grad, "b": b.grad}


class Recorder:
    """Wraps the functions of the registered shim modules and records each call: positional arguments are stored by value,
    unless a tensor is (a view with the same storage, shape and strides as) an element of an earlier call's result."""

    def __init__(self):
        self.trace, self.arrays, self.results = [], {}, []

    def encode(self, v, key):
        if isinstance(v, torch.Tensor):
            for i, res in enumerate(self.results):
                for j, r in enumerate(res):
                    if (isinstance(r, torch.Tensor) and r.data_ptr() == v.data_ptr() and r.shape == v.shape and r.stride() == v.stride()
                            and r.dtype == v.dtype):
                        return ["ret", i, j]
            self.arrays[key] = v.detach().numpy().copy()
            return ["arr", key]
        assert v is None or isinstance(v, (bool, int, float, str)), type(v)
        return ["val", v]

    def wrap(self, module, fname):
        mod = sys.modules[module]
        fn = getattr(mod, fname)

        def recorded(*args):
            i = len(self.trace)
            self.trace.append({"module": module, "fn": fname,
                               "args": [self.encode(a, f"call{i}_arg{j}") for j, a in enumerate(args)]})
            res = fn(*args)
            self.results.append(list(res) if isinstance(res, (list, tuple)) else [res])
            return res
        setattr(mod, fname, recorded)


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path, submodule_search_locations=[os.path.dirname(path)] if path.endswith("__init__.py") else None)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def main():
    sys.path.insert(0, ROOT)
    saved_attrs, saved_mods = [], {n: sys.modules.get(n) for n in SHIM_MODULES}

    def setattr_(obj, name, value):
        saved_attrs.append((obj, name, getattr(obj, name)))
        setattr(obj, name, value)
    try:
        calls = install_shim(setattr_)
        rec = Recorder()
        for module, fname in (("selective_scan_cuda", "fwd"), ("selective_scan_cuda", "bwd"),
                              ("causal_conv1d_cuda", "causal_conv1d_fwd"), ("causal_conv1d_cuda", "causal_conv1d_bwd")):
            rec.wrap(module, fname)
        _load("causal_conv1d", os.path.join(REF_ROOT, "dis_causal_conv1d", "causal_conv1d", "__init__.py"))
        ssi = _load("_ref_ssi_under_shim", os.path.join(REF_ROOT, "dis_mamba", "mamba_ssm", "ops", "selective_scan_interface.py"))
        conv = sys.modules["causal_conv1d"]
        conv_iface = sys.modules["causal_conv1d.causal_conv1d_interface"]
        scan_in, conv_in = inputs()

        out, last, grads = run_scan(ssi.selective_scan_fn, scan_in)       # reference autograd Function -> shim -> stand-ins
        ref_out, ref_last, ref_grads = run_scan(ssi.selective_scan_ref, scan_in)
        y, cgrads = run_conv(conv.causal_conv1d_fn, conv_in)
        ref_y, ref_cgrads = run_conv(conv_iface.causal_conv1d_ref, conv_in)
        assert calls == ["scan_fwd", "scan_fwd", "scan_bwd", "conv_fwd", "conv_bwd"], calls
        assert torch.allclose(out, ref_out, rtol=1e-4, atol=1e-5) and torch.allclose(last, ref_last, rtol=1e-4, atol=1e-5)
        for k in SCAN_INPUTS:
            assert torch.allclose(grads[k], ref_grads[k], rtol=1e-3, atol=1e-4), k
        assert torch.allclose(y, ref_y, atol=1e-6)
        for k in cgrads:
            assert torch.allclose(cgrads[k], ref_cgrads[k], atol=1e-5), k
    finally:
        for obj, name, value in reversed(saved_attrs):
            setattr(obj, name, value)
        for n, m in saved_mods.items():
            if m is None:
                sys.modules.pop(n, None)
            else:
                sys.modules[n] = m

    want = {"scan_out": ref_out, "scan_last": ref_last, "conv_y": ref_y}
    want.update({f"scan_grad_{k}": v for k, v in ref_grads.items()})
    want.update({f"conv_grad_{k}": v for k, v in ref_cgrads.items()})
    arrays = dict(rec.arrays, **{f"want_{k}": v.numpy() for k, v in want.items()})
    np.savez_compressed(GOLD, trace_json=np.frombuffer(json.dumps(rec.trace).encode(), dtype=np.uint8), **arrays)
    print(f"wrote {GOLD}: {len(rec.trace)} calls, {len(arrays)} arrays, {os.path.getsize(GOLD)} bytes")
    for c in rec.trace:
        print(f"  {c['module']}.{c['fn']}({', '.join(a[0] if a[0] != 'val' else repr(a[1]) for a in c['args'])})")


if __name__ == "__main__":
    main()
