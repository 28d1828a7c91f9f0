"""
bench.py's host logic without a GPU: the per-rank launch list of a token (what the reference's model code issues through the
operator surface: q+k+v as one fan-out exl3_mgemm (or q, k+v like the reference's Llama module), o, gate+up as one exl3_mgemm, down
per layer, then lm_head; SURVEY.md 8d / a14),
the tensor-parallel shard shapes, the algorithmic byte count of the roofline, and the control flow of Token.run() for the
NCCL and the fused row-parallel variants -- with a recording stand-in for the extension (no kernel runs here).
"""
import os, sys
import pytest
import torch
from conftest import ROOT

sys.path.insert(0, ROOT)
import bench

TINY = dict(hidden=256, inter=512, q=256, kv=128, layers=2, vocab=640, K=4, head_K=6)


class Recorder:
    def __init__(self):
        self.calls = []

    def exl3_gemm(self, A, B, C, suh, A_had, svh, fsi, mcg, mul1, fns):
        assert A.shape[-1] == B.shape[0] * 16 and C.shape[-1] == B.shape[1] * 16 and mul1 and not mcg
        self.calls.append(("gemm", A.shape[-1], C.shape[-1]))
        return 210

    def exl3_gemm_allreduce(self, A, B, C, suh, A_had, svh, mcg, mul1):
        assert A_had is None and mul1 and not mcg
        self.calls.append(("gemm_ar", A.shape[-1], C.shape[-1]))
        return 211

    def exl3_mgemm(self, A, B, C, suh, A_had, svh, indices, weights, K, fsi, mcg, mul1, mn, mx, fns, num_tokens=1, size_n_list=None, c_ptrs=None):
        assert indices is None and weights is None and mn == -1 and mx == -1 and num_tokens == 1
        if size_n_list is not None:
            # fan-out: per-matrix widths, outputs through c_ptrs, C carries dtype and the maximum width
            assert B.numel() == c_ptrs.numel() == size_n_list.numel() == C.shape[0] and C.shape[-1] == int(size_n_list.max())
            assert size_n_list.dtype == torch.int and c_ptrs.dtype == torch.long and A_had.shape[0] == B.numel()
            self.calls.append(("fanout", A.shape[-1]) + tuple(int(v) for v in size_n_list))
            return 210
        assert B.numel() == 2 and C.shape[0] == 2 and c_ptrs is None
        self.calls.append(("mgemm", A.shape[-1], C.shape[-1]))
        return 210


@pytest.mark.parametrize("tp", [1, 2, 4])
def test_token_launch_list_and_run_control_flow(tp, monkeypatch):
    dev = torch.device("cpu")
    tok = bench.Token(TINY, tp, 0, dev)
    sh = lambda x: max(128, (x // tp) // 128 * 128) if tp > 1 else x
    assert len(tok.mats) == 7 * TINY["layers"] + 1
    # default: q+k+v as one fan-out exl3_mgemm, gate+up as one exl3_mgemm: 129 launches for the 32-layer model; the reference's
    # Llama launch list (q, then k+v) stays available for the same-run comparison: 161 launches
    assert len(tok.launches) == 4 * TINY["layers"] + 1 and len(tok.launches_ref) == 5 * TINY["layers"] + 1
    ref_layer = [("gemm", 256, sh(256)), ("mgemm", 256, sh(128)), ("gemm", sh(256), 256), ("mgemm", 256, sh(512)), ("gemm", sh(512), 256)]
    per_layer = [("fanout", 256, sh(256), sh(128), sh(128))] + ref_layer[2:]
    head = ("gemm", 256, sh(640) if tp > 1 else 640)
    rec = Recorder(); tok.ext = rec; tok.skip_reduce = True
    tok.run(tok.launches_ref)
    assert rec.calls == ref_layer * TINY["layers"] + [head]
    assert tok.list_alg_bytes(tok.launches_ref) - tok.alg_bytes == 2 * 256 * TINY["layers"]        # one more read of the shared input per layer
    nofan = bench.Token(TINY, tp, 0, dev, fanout=False)
    assert len(nofan.launches) == 5 * TINY["layers"] + 1 and nofan.launches_ref is nofan.launches

    # (1) kernels only (the single-GPU bench, or --tp-shapes): no collective
    rec = Recorder(); tok.ext = rec; tok.skip_reduce = True
    tok.run()
    assert rec.calls == per_layer * TINY["layers"] + [head]

    # (2) NCCL variant: one all_reduce after every row-parallel output (o, down) when tp > 1
    import torch.distributed as dist
    reduced = []
    monkeypatch.setattr(dist, "all_reduce", lambda t, *a, **k: reduced.append(tuple(t.shape)))
    rec = Recorder(); tok.ext = rec; tok.skip_reduce = False
    tok.run()
    assert rec.calls == per_layer * TINY["layers"] + [head]
    assert len(reduced) == (2 * TINY["layers"] if tp > 1 else 0) and all(s == (1, 256) for s in reduced)

    # (3) fused variant: the row-parallel GEMMs become exl3_gemm_allreduce, nothing else changes, no NCCL call
    if tp > 1:
        reduced.clear()
        rec = Recorder(); tok.ext = rec; tok.fused_reduce = True
        tok.run()
        fused_layer = [c if i not in (1, 3) else ("gemm_ar",) + c[1:] for i, c in enumerate(per_layer)]
        assert rec.calls == fused_layer * TINY["layers"] + [head]
        assert reduced == []


def test_algorithmic_bytes_match_survey_8d():
    # 4096 x 4096, K = 4, m = 1, fp16 out: 8,388,608 + 8,192 + 8,192 + 16,384 = 8,421,376 B (SURVEY.md 8d)
    assert bench.alg_bytes(1, 4096, 4096, 4, False) == 8421376
    cfg = bench.MODELS["llama-3.1-8b"]
    layer, head = bench.token_plan(cfg, 1)
    total = cfg["layers"] * sum(bench.alg_bytes(1, k, n, K, f) for (_, k, n, K, f, _) in layer) + bench.alg_bytes(1, *head[1:5])
    assert abs(total / 1e9 - 3.884) < 0.02                       # "Llama-8B token: 3.884 GB"
    assert bench.weights_per_token(cfg) == 32 * 218103808 + 4096 * 128256
    # TP shards are multiples of 128 channels and never empty
    for tp in (2, 4, 8):
        for model in bench.MODELS.values():
            layer, head = bench.token_plan(model, tp)
            for (_, k, n, _, _, _) in layer + [head]:
                assert k % 128 == 0 and n % 128 == 0 and k >= 128 and n >= 128


def test_qgemm_section_control_flow(monkeypatch):
    """bench.py's supplementary section (per-shape decode GB/s, prefill TFLOP/s) with every CUDA facility stubbed: checks the
    Python control flow, the shapes it times and the keys it reports -- so that a typo cannot cost the round's bench line."""
    import contextlib
    import exllamav3_b200
    from exllamav3_b200 import ext, QLinear

    class Ev:
        def __init__(self, enable_timing=True): pass
        def record(self, s=None): pass
        def synchronize(self): pass
        def elapsed_time(self, other): return 1.0           # ms

    class Graph:
        def replay(self): pass

    class Stream:
        def synchronize(self): pass

    calls = []
    monkeypatch.setenv("EXL3B_BENCH_NO_REF_CUDA", "1")       # the same-run reference-kernel leg spawns a GPU process
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "graph", lambda g, stream=None: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "CUDAGraph", Graph)
    monkeypatch.setattr(torch.cuda, "Event", Ev)
    monkeypatch.setattr(ext, "exl3_gemm", lambda *a: calls.append(("gemm", a[0].shape[-1], a[2].shape[-1])) or 210)
    monkeypatch.setattr(ext, "reconstruct", lambda *a: calls.append(("rec",)))
    monkeypatch.setattr(ext, "reconstruct_had_slice", lambda *a: calls.append(("rec_had",)))
    monkeypatch.setattr(QLinear, "forward", lambda self, x, params, out_dtype=None: calls.append(("prefill", tuple(x.shape), self.out_features)) or x)
    tok = bench.Token(TINY, 1, 0, torch.device("cpu"))
    out = bench.qgemm_section(tok, TINY, Stream(), 6576.1)
    assert set(out["decode_hbm"]) == {"q", "k", "v", "o", "gate", "up", "down", "lm_head"}
    q = out["decode_hbm"]["q"]
    assert (q["k"], q["n"], q["K"]) == (256, 256, 4) and q["us_per_launch"] > 0 and q["GBps"] > 0 and q["frac_of_hbm_peak"] >= 0
    # every shape: one warm-up pass + one captured pass over its layer instances; the batch-8 / 32 leg adds the same for q twice
    # (q and o share the shape); the codebook leg adds the same for q twice more (3INST, MCG)
    assert calls.count(("gemm", 256, 256)) == 2 * 2 * TINY["layers"] + 2 * 2 * TINY["layers"] + 2 * 2 * TINY["layers"]
    assert set(out["decode_codebooks"]) == {"q_3inst", "q_mcg", "gate_3inst"}
    assert set(out["decode_batch"]) == {"q_m8", "q_m32", "gate_m8", "gate_m32", "down_m8", "down_m32"}
    assert out["decode_batch"]["q_m8"]["tag"] == 210 and "reference_cuda" in out
    assert set(out["reconstruct"]) == {"reconstruct_256x256", "reconstruct_had_256x256", "reconstruct_256x512", "reconstruct_had_256x512"}
    assert calls.count(("gemm", 256, 640)) >= 2
    pre = [c for c in calls if c[0] == "prefill"]
    assert {(c[1], c[2]) for c in pre} == {((65536, 256), 256), ((16384, 256), 512)} and len(pre) == 2 * 7
    for v in out["prefill_tensor"].values():
        assert v["tflops"] > 0 and v["frac_of_measured_bf16_burst"] > 0 and v["rows"] in (65536, 16384)


def test_ncu_capture_parser_is_unit_aware(tmp_path):
    # the committed capture: 29.485056 Mbyte read, 0 byte written, for 29.46 MB of algorithmic bytes (no re-reads)
    b = bench.ncu_dram_bytes(os.path.join(ROOT, bench.NCU_CAPTURE))
    assert 29.4e6 < b < 29.6e6 and abs(b / bench.alg_bytes(1, 4096, 14336, 4, True) - 1.0) < 2e-3
    f = tmp_path / "cap.csv"
    f.write_text("metric,unit,value\ndram__bytes_read.sum,Gbyte,1.5\ndram__bytes_write.sum,Kbyte,2\n")
    assert bench.ncu_dram_bytes(str(f)) == 1.5e9 + 2e3


@pytest.mark.parametrize("fanout", [True, False])
def test_dumped_outputs_are_what_each_launch_wrote(fanout, tmp_path):
    """--dump-outputs: every projection's output as float32, stacked over layers, taken from the buffer its launch writes
    (a two-matrix exl3_mgemm's own output, otherwise the matrix's y); within 64 MB for both bench models."""
    import numpy as np
    tok = bench.Token(TINY, 1, 0, torch.device("cpu"), fanout=fanout)
    for i, mt in enumerate(tok.mats):
        mt["y"].fill_(i)
    pair = {}
    for ln in tok.launches:
        for j, mt in enumerate(ln.get("mats", ())):
            i = next(i for i, t in enumerate(tok.mats) if t is mt)
            ln["y"][j].fill_(1000 + i); pair[i] = True
    names = ["q", "k", "v", "o", "gate", "up", "down"]
    assert {tok.mats[i]["name"] for i in pair} == ({"gate", "up"} if fanout else {"k", "v", "gate", "up"})
    bench.dump_outputs(tok, str(tmp_path))
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(f"{n}.npy" for n in names + ["lm_head"])
    for name in names + ["lm_head"]:
        a = np.load(tmp_path / f"{name}.npy")
        idx = [i for i, t in enumerate(tok.mats) if t["name"] == name]
        assert a.dtype == np.float32 and a.shape == (len(idx), 1, tok.mats[idx[0]]["n"])
        assert [float(v) for v in a[:, 0, 0]] == [1000.0 + i if i in pair else float(i) for i in idx]
    for cfg in bench.MODELS.values():
        layer, head = bench.token_plan(cfg, 1)
        assert 4 * (cfg["layers"] * sum(n for (_, _, n, _, _, _) in layer) + head[2]) <= 64 << 20
