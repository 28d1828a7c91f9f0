"""
TEST INFRASTRUCTURE (oracle).  Generates tests/golden/ref_callsites.json by running the reference's OWN Python modules
(unmodified, loaded from a checkout of turboderp-org/exllamav3; nothing is copied) with their `ext` import bound to this
repo's shim (exllamav3_b200.ext), exactly what INTEGRATION.md's three-line patch does.  The shim's qgemm entry points are
replaced by recorders that bind every call against the real signature (no kernel runs).  Recorded:

  * constants       AUTO_RECONSTRUCT_THRESHOLD, MAX_RECONSTRUCT_SLICE_N             modules/quant/exl3.py:10-11
  * bc_ctor         the arguments LinearEXL3 passes to ext.BC_LinearEXL3            modules/quant/exl3.py:81-90
  * linear, wide    the extension calls (argument shapes / values) of LinearEXL3.forward per input shape and params,
                    and with the output slicing window narrowed to 256 columns
  * multilinear     which tensor each entry of MultiLinear's pointer tables addresses   modules/multilinear.py:30-32
  * callsites       every `ext.<op>(...)` call of the qgemm surface in the reference's Python sources (file, line, argument
                    count, keyword names)
  * use_mgemm       InferParams.use_mgemm for an int8-GEMV K cap of 0 (this shim) and 6 (the reference's extension on
                    sm_100)                                                          model/config.py:48-64
  * tp_split        LinearEXL3.tp_export / tp_import_split per shard: metadata and digests of the shard tensors
                                                                                    modules/quant/exl3.py:268-330

tests/test_reference_callsites.py replays the same inputs through this repo's own caller (QLinear, pointer_tables,
tp.tp_slice) and the shim's signatures, and compares with this file.

usage: python oracle/gen_golden_callsites.py <exllamav3 checkout>
"""
import ast, importlib.util, inspect, json, os, sys, types
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, "tests", "golden", "ref_callsites.json")
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from exllamav3_b200 import ext, tp  # noqa: E402
import refstubs  # noqa: E402

AUDITED_OPS = ["exl3_gemm", "exl3_mgemm", "reconstruct", "reconstruct_slice", "reconstruct_had_slice", "had_r_128", "hgemm",
               "exl3_gemv", "g_get_cc", "g_get_num_sms", "exl3_gemv_int8_max_k", "exl3_gemm_num_kernel_shapes",
               "exl3_gemm_shape_compat"]


def stub(name, **attrs):
    m = types.ModuleType(name)
    m.__path__ = []
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m


def load(pkg, name, rel):
    spec = importlib.util.spec_from_file_location(name, os.path.join(pkg, *rel.split("/")))
    m = importlib.util.module_from_spec(spec)
    sys.modules[name] = m
    spec.loader.exec_module(m)
    return m


def load_exl3(pkg):
    class Config: pass
    stub("exllamav3"); stub("exllamav3.model")
    stub("exllamav3.model.config", Config=Config, NullConfig=refstubs.NullConfig)
    stub("exllamav3.ext", exllamav3_ext=ext)
    stub("exllamav3.util", profile_opt=lambda f: f)
    stub("exllamav3.util.tensor", g_tensor_cache=refstubs.g_tensor_cache)
    stub("exllamav3.modules"); stub("exllamav3.modules.quant"); stub("exllamav3.modules.quant.exl3_lib")
    stub("exllamav3.modules.quant.exl3_lib.quantize", preapply_had_l=refstubs.preapply_had_l,
         preapply_had_r=refstubs.preapply_had_r, had_k=128, had_n=128)
    return load(pkg, "exllamav3.modules.quant.exl3", "modules/quant/exl3.py")


def dtype_name(dt):
    return None if dt is None else str(dt).replace("torch.", "")


def linear_section(mod, calls):
    ctor = {}
    real = ext.BC_LinearEXL3

    def bc(*a, **kw):
        inspect.signature(real).bind(*a, **kw)
        ctor.update(args=[list(t.shape) if isinstance(t, torch.Tensor) else t for t in a], kwargs=sorted(kw))
        return real(*a, **kw)
    ext.BC_LinearEXL3 = bc
    k, n = 256, 384
    lin = mod.LinearEXL3(None, k, n, key="q", **refstubs.linear_tensors(k, n))
    ext.BC_LinearEXL3 = real
    assert isinstance(lin.bc, real)
    cases = []
    for (shape, params, out_dtype) in (((1, k), {}, None), ((144, k), {}, torch.float), ((3, 7, k), {}, None),
                                       ((145, k), {}, None), ((1, k), {"reconstruct": True}, None), ((1024, k), {}, torch.float),
                                       ((2, k), {}, None)):
        calls.clear()
        y = lin.forward(torch.zeros(shape, dtype=torch.half), params, out_dtype)
        cases.append(dict(shape=list(shape), params=params, out_dtype=dtype_name(out_dtype), calls=refstubs.jsonable(calls),
                          y_shape=list(y.shape), y_dtype=dtype_name(y.dtype)))
    linear = dict(k=k, n=n, K=lin.K, mcg=lin.mcg, mul1=lin.mul1, cases=cases)

    mod.MAX_RECONSTRUCT_SLICE_N = 256
    k, n = 128, 640
    lin = mod.LinearEXL3(None, k, n, **refstubs.linear_tensors(k, n))
    wide = dict(slice_n=256, k=k, n=n, cases=[])
    for rows in (200, 2048):
        calls.clear()
        lin.forward(torch.zeros((rows, k), dtype=torch.half), {})
        wide["cases"].append(dict(rows=rows, calls=refstubs.jsonable(calls)))
    mod.MAX_RECONSTRUCT_SLICE_N = 32768
    return ctor, linear, wide


def multilinear_section(pkg, mod):
    src = open(os.path.join(pkg, "modules", "multilinear.py")).read()
    ns = {}
    exec(compile(src.replace("from . import Linear", "Linear = object"), "multilinear_ref", "exec"), ns)   # in memory, not copied
    k, n = 128, 256
    inners = [mod.LinearEXL3(None, k, n, **refstubs.linear_tensors(k, n)) for _ in range(3)]

    class Lin:                                                  # the reference wraps LinearEXL3 in modules.Linear (.inner)
        def __init__(self, inner):
            self.inner, self.quant_type, self.softcap, self.post_scale = inner, "exl3", 0.0, 1.0
            self.in_features, self.out_features = inner.in_features, inner.out_features
    ml = ns["MultiLinear"]("cpu", [Lin(i) for i in inners])
    where = {getattr(i, a).data_ptr(): [a, j] for j, i in enumerate(inners) for a in ("trellis", "suh", "svh")}
    tables = {}
    for a in ("ptrs_trellis", "ptrs_suh", "ptrs_svh"):
        t = getattr(ml, a)
        tables[a] = dict(dtype=dtype_name(t.dtype), entries=[where[p] for p in t.tolist()])
    return dict(k=k, n=n, count=len(inners), tables=tables, K=ml.K, mcg=ml.mcg, mul1=ml.mul1,
                in_features=ml.in_features, out_features=ml.out_features)


def callsites_section(checkout):
    sites, files = [], 0
    for root, dirs, names in os.walk(checkout):                 # the package, science/ (qgemm_benchmark.py), tests/, eval/
        dirs.sort()
        if "exllamav3_ext" in root:
            continue
        for nm in sorted(names):
            if not nm.endswith(".py"):
                continue
            path = os.path.join(root, nm)
            try:
                tree = ast.parse(open(path).read())
            except SyntaxError:
                continue
            files += 1
            for node in ast.walk(tree):
                if (isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and node.func.attr in AUDITED_OPS
                        and isinstance(node.func.value, ast.Name) and node.func.value.id == "ext"):
                    if any(isinstance(a, ast.Starred) for a in node.args) or any(kw.arg is None for kw in node.keywords):
                        continue
                    sites.append(dict(path=os.path.relpath(path, checkout), line=node.lineno, op=node.func.attr,
                                      nargs=len(node.args), kwargs=[kw.arg for kw in node.keywords]))
    sites.sort(key=lambda s: (s["path"], s["line"], s["op"]))
    return dict(ops=AUDITED_OPS, files=files, sites=sites)


def use_mgemm_section(pkg):
    stub("exllamav3"); stub("exllamav3.model"); stub("exllamav3.util")
    stub("exllamav3.util.rope", RopeSettings=object, RopeStyle=object)
    stub("exllamav3.loader", SafetensorsCollection=object)
    stub("exllamav3.util.file", read_dict=None, no_value=None, no_default=None)
    stub("exllamav3.ext", exllamav3_ext=ext)
    for v in ("EXL3_INT8_GEMV", "EXL3_MGEMM_K_THRESHOLD", "EXL3_MGEMM_N_THRESHOLD"):
        os.environ.pop(v, None)
    cfg = load(pkg, "exllamav3.model.config", "model/config.py")
    ip = cfg.InferParams()
    real = ext.exl3_gemv_int8_max_k
    out = []
    for cap in (0, 6):
        ext.exl3_gemv_int8_max_k = lambda dev, cap=cap: cap
        for K in range(1, 9):
            for n in (14336, 1024):
                for mul1 in (True, False):
                    out.append(dict(int8_max_k=cap, K=K, out_features=n, mul1=mul1,
                                    fused=bool(ip.use_mgemm(K, n, mul1=mul1, device="cuda:0"))))
    ext.exl3_gemv_int8_max_k = real
    return out


def tp_section(mod):
    class Producer:
        def send(self, t): return t

    class Consumer:
        def recv(self, t, cuda=False, slice_dim=None, first=None, last=None):
            if t is None:
                return None
            return t if slice_dim is None else t.narrow(slice_dim, first, last - first).contiguous()

    k, n, world = 512, 768, 3
    tens, bias = refstubs.tp_tensors(k, n)
    full = mod.LinearEXL3(None, k, n, bias=bias, out_dtype=torch.float, **tens)
    exported = full.tp_export(None, Producer())
    ctx = {"consumer": Consumer(), "device": "cpu"}
    splits = [(True, a, b) for (a, b) in tp.split_ranges(n, world)] + [(False, a, b) for (a, b) in tp.split_ranges(k, world)] + [None]
    out = []
    for split in splits:
        r = mod.LinearEXL3.tp_import_split(ctx, exported, None, split)
        out.append(dict(split=None if split is None else list(split), in_features=r.in_features, out_features=r.out_features,
                        K=r.K, mcg=r.mcg, mul1=r.mul1, out_dtype=dtype_name(r.out_dtype),
                        trellis=refstubs.digest(r.trellis), suh=refstubs.digest(r.suh), svh=refstubs.digest(r.svh),
                        bias=refstubs.digest(r.bias)))
    return dict(k=k, n=n, world=world, splits=out)


def main():
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    checkout = os.path.abspath(sys.argv[1])
    pkg = os.path.join(checkout, "exllamav3")
    mod = load_exl3(pkg)
    calls = refstubs.install_recorders(ext, setattr)
    ctor, linear, wide = linear_section(mod, calls)
    out = dict(
        constants=dict(AUTO_RECONSTRUCT_THRESHOLD=mod.AUTO_RECONSTRUCT_THRESHOLD, MAX_RECONSTRUCT_SLICE_N=mod.MAX_RECONSTRUCT_SLICE_N),
        bc_ctor=ctor, linear=linear, wide=wide, multilinear=multilinear_section(pkg, mod), callsites=callsites_section(checkout),
        tp_split=tp_section(mod), use_mgemm=use_mgemm_section(pkg))
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote", os.path.abspath(OUT))


if __name__ == "__main__":
    main()
