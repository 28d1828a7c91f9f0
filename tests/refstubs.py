"""
Test harness only: the few names the REFERENCE'S OWN modules import from the rest of its package (config defaults, the
process-global scratch cache, the Hadamard helpers of its quantizer), provided as minimal stand-ins so that the
reference's exllamav3/modules/quant/exl3.py can be loaded unmodified with its `ext` bound to exllamav3_b200.ext
(oracle/gen_golden_callsites.py), and the call recorder and seeded inputs that the generator and
tests/test_reference_callsites.py share.  Nothing in the product imports this file.
"""
import hashlib, inspect
import numpy as np
import torch

RECORDED_OPS = ("exl3_gemm", "had_r_128", "reconstruct", "reconstruct_slice", "reconstruct_had_slice", "hgemm")


def install_recorders(ext, setattr_fn):
    """Replace ext's qgemm entry points (via setattr_fn) by recorders that bind each call against the real signature and
    log (name, argument shapes / values); returns the log.  No kernel runs."""
    calls = []

    def wrap(name):
        sig = inspect.signature(getattr(ext, name))

        def f(*a, **kw):
            sig.bind(*a, **kw)                                    # the caller's argument list fits the shim's signature
            calls.append((name,) + tuple(tuple(t.shape) if isinstance(t, torch.Tensor) else t for t in a))
            return 210
        return f

    for name in RECORDED_OPS:
        setattr_fn(ext, name, wrap(name))
    return calls


def jsonable(calls):
    """A call log in the form it takes after a JSON round trip (tuples become lists)."""
    return [[list(v) if isinstance(v, tuple) else v for v in c] for c in calls]


def linear_tensors(k, n, K=4):
    g = torch.Generator().manual_seed(1)
    tr = torch.randint(0, 32767, (k // 16, n // 16, 16 * K), generator=g, dtype=torch.int32).to(torch.int16)
    return dict(suh=torch.ones(k, dtype=torch.half), svh=torch.ones(n, dtype=torch.half), trellis=tr, mul1=torch.zeros((), dtype=torch.int))


def tp_tensors(k, n):
    """Inputs of the tensor-parallel split comparison: random trellis, scales and bias."""
    t = linear_tensors(k, n)
    g = torch.Generator().manual_seed(5)
    t["suh"] = torch.randn(k, generator=g).half(); t["svh"] = torch.randn(n, generator=g).half()
    return t, torch.randn(n, generator=g).half()


def digest(t):
    """[dtype, shape, sha256 of the values] of a tensor, or None."""
    if t is None:
        return None
    return [str(t.dtype), list(t.shape), hashlib.sha256(t.contiguous().numpy().tobytes()).hexdigest()]


class InferParams:
    no_reconstruct = False


class NullConfig:
    def __init__(self):
        self.infer_params = InferParams()


class TensorCache:
    def __init__(self):
        self.d = {}

    def get(self, device, shape, dtype):
        return self.d.setdefault((str(device), tuple(shape), dtype), torch.empty(shape, dtype=torch.half, device=device))


g_tensor_cache = TensorCache()


def _h(n, ref):
    from oracle import exl3_oracle as orc
    assert n == 128
    return torch.from_numpy(orc.hadamard_matrix_128() / np.sqrt(128.0)).to(ref.device, ref.dtype)


def preapply_had_l(x, had_dim):
    k, n = x.shape
    return (_h(had_dim, x) @ x.view(k // had_dim, had_dim, n)).view(k, n)


def preapply_had_r(x, had_dim):
    k, n = x.shape
    return (x.view(k, n // had_dim, had_dim) @ _h(had_dim, x)).view(k, n)
