"""
Drop-in check at the Python level against the REFERENCE'S OWN modules (`exllamav3/modules/quant/exl3.py` LinearEXL3,
`modules/multilinear.py`, `model/config.py`): oracle/gen_golden_callsites.py ran them unmodified with their `ext` import bound
to this repo's shim (`exllamav3_b200.ext`), exactly what INTEGRATION.md's three-line patch does, and recorded every extension
call they made (bound against the shim's real signatures) in tests/golden/ref_callsites.json.  Here this repo's own minimal
caller (QLinear, pointer_tables, tp.tp_slice) runs on the same inputs and must issue the same extension calls with the same
argument shapes, and every recorded call must still fit the shim's signatures.  No kernel runs: the shim's entry points are
wrapped by recorders after their signatures have been checked.
"""
import inspect, json, os
import pytest
import torch

import refstubs
from conftest import GOLDEN

REF = json.load(open(os.path.join(GOLDEN, "ref_callsites.json")))
DTYPES = {None: None, "float16": torch.half, "float32": torch.float}


@pytest.fixture()
def recorded(monkeypatch):
    from exllamav3_b200 import ext
    return refstubs.install_recorders(ext, monkeypatch.setattr)


def _qlin(t, **kw):
    from exllamav3_b200 import QLinear
    return QLinear(t["trellis"], t["suh"], t["svh"], mul1=True, **kw)


def _fits_shim(calls):
    """Every recorded call of the reference still binds against the shim's current signature."""
    from exllamav3_b200 import ext
    for c in calls:
        inspect.signature(getattr(ext, c[0])).bind(*c[1:])


def test_reference_linear_exl3_runs_on_the_shim_and_matches_the_mirror(recorded):
    from exllamav3_b200 import ext, qlinear
    calls = recorded
    assert REF["constants"]["AUTO_RECONSTRUCT_THRESHOLD"] == qlinear.KERNEL_MAX_ROWS == 144
    assert REF["constants"]["MAX_RECONSTRUCT_SLICE_N"] == qlinear.DENSE_WINDOW_COLS == 32768
    lin = REF["linear"]
    k, n = lin["k"], lin["n"]
    # the reference constructs ext.BC_LinearEXL3 from the shim: its arguments bind against the shim's constructor
    ctor = REF["bc_ctor"]
    inspect.signature(ext.BC_LinearEXL3).bind(*ctor["args"], **{kw: None for kw in ctor["kwargs"]})
    t = refstubs.linear_tensors(k, n)
    assert ctor["args"][:3] == [list(t["trellis"].shape), [k], [n]] and ctor["args"][3:7] == [4, None, False, True]
    assert isinstance(ext.BC_LinearEXL3(t["trellis"], t["suh"], t["svh"], 4, None, False, True, None), ext.BC_LinearEXL3)
    assert lin["K"] == 4 and lin["mul1"] and not lin["mcg"]
    mir_lin = _qlin(t)
    for case in lin["cases"]:
        _fits_shim(case["calls"])
        calls.clear()
        ym = mir_lin.forward(torch.zeros(case["shape"], dtype=torch.half), case["params"], DTYPES[case["out_dtype"]])
        seq_mir = refstubs.jsonable(calls)
        assert case["calls"] == seq_mir and len(seq_mir) >= 1, case      # same extension calls, same argument shapes
        assert case["y_shape"] == list(ym.shape) == case["shape"][:-1] + [n] and DTYPES[case["y_dtype"]] == ym.dtype
    # the kernel path hands exl3_gemm the reference's 10 arguments: (A, B, C, suh, A_had, svh, -1, mcg, mul1, 0)
    two_rows = next(c for c in lin["cases"] if c["shape"] == [2, k] and not c["params"])
    assert two_rows["calls"][0][0] == "exl3_gemm" and two_rows["calls"][0][7:] == [-1, False, True, 0]


def test_reference_wide_output_slicing_matches_the_mirror(recorded, monkeypatch):
    from exllamav3_b200 import qlinear
    calls = recorded
    wide = REF["wide"]
    monkeypatch.setattr(qlinear, "DENSE_WINDOW_COLS", wide["slice_n"])
    mir_lin = _qlin(refstubs.linear_tensors(wide["k"], wide["n"]))
    assert [c["rows"] for c in wide["cases"]] == [200, 2048]
    for case in wide["cases"]:
        _fits_shim(case["calls"])
        calls.clear(); mir_lin.forward(torch.zeros((case["rows"], wide["k"]), dtype=torch.half), {})
        assert case["calls"] == refstubs.jsonable(calls) and sum(c[0] == "hgemm" for c in case["calls"]) == 3


def test_reference_multilinear_tables_match_the_mirror():
    """modules/multilinear.py builds the pointer tables exl3_mgemm reads; pointer_tables must build the same ones."""
    from exllamav3_b200 import pointer_tables
    ml_ref = REF["multilinear"]
    k, n = ml_ref["k"], ml_ref["n"]
    inners = [_qlin(refstubs.linear_tensors(k, n)) for _ in range(ml_ref["count"])]
    where = {getattr(i, a).data_ptr(): [a, j] for j, i in enumerate(inners) for a in ("trellis", "suh", "svh")}
    ml = dict(zip(("ptrs_trellis", "ptrs_suh", "ptrs_svh"), pointer_tables("cpu", inners)))
    for a in ("ptrs_trellis", "ptrs_suh", "ptrs_svh"):
        assert ml[a].dtype == torch.long and ml_ref["tables"][a]["dtype"] == "int64"
        assert [where.get(p) for p in ml[a].tolist()] == ml_ref["tables"][a]["entries"]
    i0 = inners[0]
    assert (ml_ref["K"], ml_ref["mcg"], ml_ref["mul1"], ml_ref["in_features"], ml_ref["out_features"]) == \
           (i0.K, i0.mcg, i0.mul1, i0.in_features, i0.out_features) == (4, False, True, k, n)


def test_every_reference_call_site_of_the_qgemm_surface_fits_the_shim():
    """Static audit: every `ext.<op>(...)` call in the reference's Python sources, for the ops of the qgemm path, is bound
    (by argument count and keyword names) against the shim's signature.  SURVEY.md 8b lists these callers."""
    from exllamav3_b200 import ext
    audit = REF["callsites"]
    sigs = {o: inspect.signature(getattr(ext, o)) for o in audit["ops"]}
    seen = {o: 0 for o in audit["ops"]}
    for s in audit["sites"]:
        try:
            sigs[s["op"]].bind(*([None] * s["nargs"]), **{kw: None for kw in s["kwargs"]})
        except TypeError as e:
            raise AssertionError(f"{s['path']}:{s['line']}: ext.{s['op']} call does not fit the shim: {e}")
        seen[s["op"]] += 1
    assert audit["files"] > 50
    assert seen["exl3_gemm"] >= 1 and seen["exl3_gemm_num_kernel_shapes"] >= 1 and seen["exl3_gemm_shape_compat"] >= 1   # science/qgemm_benchmark.py
    # the call sites SURVEY.md 8b names exist and were checked
    assert seen["exl3_mgemm"] >= 8 and seen["hgemm"] >= 3 and seen["had_r_128"] >= 2 and seen["reconstruct"] >= 2
    assert seen["reconstruct_had_slice"] >= 2 and seen["reconstruct_slice"] >= 1 and seen["exl3_gemv_int8_max_k"] >= 1


def test_reference_use_mgemm_policy_with_the_shims_answer(monkeypatch):
    """model/config.py:48-64, the reference's OWN policy function, evaluated with this shim's exl3_gemv_int8_max_k (0): k+v and
    gate+up stay fused for every bitrate -- the launch list bench.py times (161 launches) -- whereas with the reference
    extension's answer on Blackwell (6) the wide 4-bpw gate+up pair is unfused (225-launch variant, bench.py --no-fuse)."""
    from exllamav3_b200 import ext
    monkeypatch.setattr(ext, "_check", lambda rc: 148)                      # no device here: the index check is not under test
    shim = ext.exl3_gemv_int8_max_k(0)
    assert shim == 0
    fused = {(u["int8_max_k"], u["K"], u["out_features"], u["mul1"]): u["fused"] for u in REF["use_mgemm"]}
    for K in range(1, 9):
        assert fused[(shim, K, 14336, True)]                                # gate/up: fused at every bitrate
        assert fused[(shim, K, 1024, True)]                                 # k/v
        assert fused[(shim, K, 14336, False)]                               # other codebooks are always fused
    assert not fused[(6, 4, 14336, True)]                                   # the reference's own extension on sm_100: wide 4 bpw pair unfused
    assert fused[(6, 4, 1024, True)]                                        # narrow outputs stay fused either way
    assert fused[(6, 7, 14336, True)]


def test_reference_tp_import_split_equals_tp_slice():
    """The reference's OWN shard construction (LinearEXL3.tp_export / tp_import_split, modules/quant/exl3.py:268-330), run with a
    trivial in-process stand-in for its SHM producer / consumer transport, against this repo's tp.tp_slice."""
    from exllamav3_b200 import tp
    ref = REF["tp_split"]
    k, n, world = ref["k"], ref["n"], ref["world"]
    tens, bias = refstubs.tp_tensors(k, n)
    mir_full = _qlin(tens, bias=bias, out_dtype=torch.float)
    splits = [(True, a, b) for (a, b) in tp.split_ranges(n, world)] + [(False, a, b) for (a, b) in tp.split_ranges(k, world)] + [None]
    assert [None if s is None else list(s) for s in splits] == [r["split"] for r in ref["splits"]]
    for split, r in zip(splits, ref["splits"]):
        m = tp.tp_slice(mir_full, split)
        assert (r["in_features"], r["out_features"], r["K"], r["mcg"], r["mul1"], DTYPES[r["out_dtype"]]) == \
               (m.in_features, m.out_features, m.K, m.mcg, m.mul1, m.out_dtype)
        for a in ("trellis", "suh", "svh", "bias"):
            assert refstubs.digest(getattr(m, a)) == r[a], (split, a)
        assert m.trellis.is_contiguous()
