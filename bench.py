#!/usr/bin/env python
"""
bench.py -- decode tok/s of the EXL3 qgemm hot path on Llama-3.1-8B shapes @ 4.0 bpw, batch 1 (BASELINE.json metric).

A "step" is one token's worth of quantized GEMMs: 32 layers x (q, k, v, o, gate, up, down) + lm_head (K=6), m = 1,
executed back to back over DISTINCT synthetic weight buffers (3.88 GB >> 126 MB L2, so nothing is cache-resident
between steps).  Attention / norm / rope are not part of the hot path (SURVEY.md 8) and are not executed.

  value      tok/s with inputs resident in HBM when the timed region starts (CUDA-graph replay of the token)
  e2e        same, through the reference-facing operator surface with HOST buffers: every step copies the token's
             hidden state from pinned host memory, runs the token, and reads the lm_head logits back to the host
  roofline   algorithmic bytes of the step (SURVEY.md 8d: k*n*K/8 + 2mk + mn*{2|4} + 2(k+n) per GEMM) / step time,
             against the measured HBM copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline   the oracle port of the reference's torch dequant+matmul path (LinearEXL3.get_weight_tensor semantics)
             timed on the host cores on a bounded sample (rank 0, N=1)
  qgemm      (N=1) the other half of BASELINE.json's metric, measured after the timed token: per matrix shape the batch-1
             qgemm's HBM GB/s and fraction of the measured copy peak, and the batch-32 prefill sibling's TFLOP/s against the
             measured dense bf16 peaks (supplementary: a failure there is reported in the key, never loses the line)

N > 1 (torchrun): the same token, tensor-parallel: q/k/v/gate/up column-sharded, o/down row-sharded with one
all-reduce (sum) per row-parallel output, lm_head column-sharded ("scaling": "strong").

--impl reference: the CPU path only (the reference has no CPU qgemm: its torch dequant+matmul semantics restated
in oracle/ are timed with all host threads), same metric/config, "impl": "reference".
"""
from __future__ import annotations
import argparse, json, os, sys, time, subprocess, threading, statistics

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODELS = {
    "llama-3.1-8b": dict(hidden=4096, inter=14336, q=4096, kv=1024, layers=32, vocab=128256, K=4, head_K=6),
    "llama-3.1-70b": dict(hidden=8192, inter=28672, q=8192, kv=1024, layers=80, vocab=128256, K=4, head_K=6),
}


def token_plan(cfg, tp=1):
    """[(name, k, n, K, c_fp32, reduce)] per rank for one layer, + head.  Sharding as modules/quant/exl3.py:284-330."""
    h, it, q, kv = cfg["hidden"], cfg["inter"], cfg["q"], cfg["kv"]
    K = cfg["K"]
    sh = lambda x: max(128, (x // tp) // 128 * 128) if tp > 1 else x
    layer = [
        ("q", h, sh(q), K, False, False), ("k", h, sh(kv), K, False, False), ("v", h, sh(kv), K, False, False),
        ("o", sh(q), h, K, True, tp > 1),
        ("gate", h, sh(it), K, True, False), ("up", h, sh(it), K, True, False),
        ("down", sh(it), h, K, True, tp > 1),
    ]
    vs = cfg["vocab"] // 128 * 128
    head = ("lm_head", h, sh(vs) if tp > 1 else vs, cfg["head_K"], True, False)
    return layer, head


def alg_bytes(m, k, n, K, c_fp32):
    return k * n * K // 8 + 2 * m * k + m * n * (4 if c_fp32 else 2) + 2 * (k + n)


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    def __init__(self, index=0):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index),
                 "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "25"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm (oracle port of the reference's torch dequant + matmul path)
# ---------------------------------------------------------------------------------------------------------------------

def cpu_path_time(cfg, budget_s=None):
    """
    Reference semantics: W = get_weight_tensor() (decode -> H128 left -> *suh -> H128 right -> *svh, torch fp32
    matmuls with the 128x128 Hadamard, modules/quant/exl3.py:227-237 + quantize.py:340-357), then x @ W in fp32.
    Sample: ALL seven matrices of layer 0 (q, k, v, o, gate, up, down), always the same work (budget_s = None), so that two
    runs differ only by the host they ran on; a budget cuts the sample short (used by nothing but quick local checks).
    Returns (weights_per_second, cores, sample_description, (y, name, k, n) of the first matrix for validation).
    """
    import ctypes, numpy as np, torch
    from oracle import exl3_oracle as orc
    so = os.path.join(ROOT, "oracle", "libexl3oracle.so")
    if not os.path.exists(so):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "libexl3oracle.so"])
    lib = ctypes.CDLL(so)
    lib.exl3o_reconstruct_f32.argtypes = [ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 5
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    layer, _ = token_plan(cfg, 1)
    H = torch.from_numpy((orc.hadamard_matrix_128() / np.sqrt(128.0)).astype(np.float32))
    done_w, t_total, names, first = 0, 0.0, [], None
    for (name, k, n, K, c_fp32, _) in layer:
        tr, suh, svh, x = orc.make_synthetic(k, n, K)
        w = np.empty((k, n), dtype=np.float32)
        t0 = time.perf_counter()
        lib.exl3o_reconstruct_f32(w.ctypes.data, tr.ctypes.data, k, n, K, 2, cores)
        wt = torch.from_numpy(w)
        wt = (H @ wt.view(k // 128, 128, n)).view(k, n)
        wt *= torch.from_numpy(suh.astype(np.float32)).unsqueeze(1)
        wt = (wt.view(k, n // 128, 128) @ H).view(k, n)
        wt *= torch.from_numpy(svh.astype(np.float32)).unsqueeze(0)
        y = torch.from_numpy(x.astype(np.float32)) @ wt
        dt = time.perf_counter() - t0
        t_total += dt; done_w += k * n; names.append(name)
        if first is None:
            first = (y.numpy().copy(), name, k, n, K)
        if budget_s is not None and t_total > budget_s:
            break
    return done_w / t_total, cores, f"layer-0 matrices {'+'.join(names)} ({done_w / 1e6:.1f} M weights, {t_total:.1f} s)", first


def weights_per_token(cfg):
    layer, head = token_plan(cfg, 1)
    return cfg["layers"] * sum(k * n for (_, k, n, _, _, _) in layer) + head[1] * head[2]


def run_reference_arm(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wps, cores, sample, _ = cpu_path_time(cfg, budget_s=5.0)    # warm-up / page-in
    vals = []
    evals = max(1, min(args.steps, 3))                          # each evaluation is the whole fixed sample (~10-30 s of CPU work)
    for _ in range(evals):
        wps, cores, sample, _ = cpu_path_time(cfg)
        vals.append(wps / weights_per_token(cfg))
    v = statistics.median(vals)
    sample += f"; median of {evals} evaluations"
    line = {
        "impl": "reference", "metric": "decode tok/s Llama-3.1-8B 4.0bpw b=1 (qgemm path)", "value": v, "unit": "tok/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 / v,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.model} EXL3 4.0bpw b=1 decode, qgemm path; CPU torch dequant+matmul "
                               "(reference LinearEXL3.get_weight_tensor semantics, oracle port) on a bounded sample",
                   "sample": sample},
        "cpu_baseline": {"value": v, "unit": "tok/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------

class Token:
    """All quantized linears of one token for one TP rank, with their input/output/scratch buffers."""

    def __init__(self, cfg, tp, rank, dev, seed=1234, fuse=True, mode="ops", fanout=True):
        import torch
        from exllamav3_b200 import ext
        self.ext, self.torch, self.dev, self.tp = ext, torch, dev, tp
        self.mode = mode
        self.skip_reduce = False
        self.fused_reduce = False           # row-parallel outputs: one kernel (GEMM + NVLink exchange) instead of GEMM + NCCL
        g = torch.Generator(device=dev); g.manual_seed(seed + rank)
        layer, head = token_plan(cfg, tp)
        self.mats = []
        self.alg_bytes = 0
        plan = [(l, spec) for l in range(cfg["layers"]) for spec in layer] + [(-1, head)]
        for (l, (name, k, n, K, c_fp32, red)) in plan:
            tr = torch.randint(0, 65536, (k // 16, n // 16, 16 * K), generator=g, device=dev, dtype=torch.int32).to(torch.int16)
            sgn = lambda sz: (torch.randint(0, 2, (sz,), generator=g, device=dev) * 2 - 1).float()
            suh = (sgn(k) * (0.5 + 1.5 * torch.rand(k, generator=g, device=dev)) / (k * tp) ** 0.5).half()
            svh = (sgn(n) * (0.5 + 1.5 * torch.rand(n, generator=g, device=dev))).half()
            x = torch.randn((1, k), generator=g, device=dev).half()
            y = torch.empty((1, n), dtype=torch.float if c_fp32 else torch.half, device=dev)
            xh = torch.empty((1, k), dtype=torch.half, device=dev)
            self.mats.append(dict(name=name, layer=l, k=k, n=n, K=K, tr=tr, suh=suh, svh=svh, x=x, y=y, xh=xh,
                                  c_fp32=c_fp32, reduce=red))
            self.alg_bytes += alg_bytes(1, k, n, K, c_fp32)
        self.first_x = self.mats[0]["x"]
        self.logits = self.mats[-1]["y"]
        # launch list.  k+v and gate+up share their input and shape: the reference's model code issues them as ONE
        # exl3_mgemm each at bsz*q_len <= 32 (modules/attn.py:603-631 multi_kv, modules/mlp.py:726-760 multi_gu) whenever
        # config.use_mgemm() says so (model/config.py:48-64): always for narrow outputs (k+v), and for gate+up when
        # ext.exl3_gemv_int8_max_k(device) < K -- the reference's own extension answers 6 on Blackwell (its separate int8 GEMVs
        # beat its fused kernel), this library's shim answers 0 (the fused launch is the faster one here), so through the
        # drop-in boundary the model issues exactly this launch list.  --no-fuse times one launch per projection.
        #
        # Fan-out (default; --no-fanout = the list above): q, k and v read the same input too, but q is wider than k / v.  The
        # reference's exl3_mgemm takes per-matrix output widths for exactly this (size_n_list + c_ptrs, exl3_gemm.cu:402-447,
        # exl3_gemm_kernel.cuh:172-181) and its fused attention issues its same-input projections that way
        # (libtorch/dsv4_attn.cpp:88-99 "fan"); its Llama attention module does not (q_proj, then multi_kv: modules/attn.py:555-631).
        # With fan-out the three projections are ONE operator call: 4 launches per layer instead of 5.  INTEGRATION.md shows the
        # module-side change; the bench line carries the token time of BOTH launch lists.
        self.fanout = bool(fanout and fuse)
        self.launches = self._launch_list(fuse, self.fanout)
        self.launches_ref = self._launch_list(fuse, False) if self.fanout else self.launches
        self.alg_bytes = self.list_alg_bytes(self.launches)

        if mode != "ops":
            self.build_chains(mode)

    def _launch_list(self, fuse, fanout):
        torch, dev = self.torch, self.dev
        out = []
        i = 0
        while i < len(self.mats):
            a = self.mats[i]
            b = self.mats[i + 1] if i + 1 < len(self.mats) else None
            c = self.mats[i + 2] if i + 2 < len(self.mats) else None
            if (fanout and c is not None and (a["name"], b["name"], c["name"]) == ("q", "k", "v") and a["layer"] == c["layer"]
                    and a["k"] == b["k"] == c["k"] and a["K"] == b["K"] == c["K"] and a["y"].dtype == b["y"].dtype == c["y"].dtype):
                grp = (a, b, c)
                ptr = lambda key: torch.tensor([t[key].data_ptr() for t in grp], dtype=torch.long, device=dev)
                out.append(dict(kind="mgemm", x=a["x"].view(1, 1, -1), K=a["K"], reduce=False, B=ptr("tr"), suh=ptr("suh"), svh=ptr("svh"),
                                y=torch.empty((3, 1, max(t["n"] for t in grp)), dtype=a["y"].dtype, device=dev),     # dtype / max-width carrier
                                xh=torch.empty((3, 1, a["k"]), dtype=torch.half, device=dev),
                                snl=torch.tensor([t["n"] for t in grp], dtype=torch.int, device=dev), cp=ptr("y"), shared_inputs=3))
                i += 3
            elif fuse and b is not None and (a["name"], b["name"]) in (("k", "v"), ("gate", "up")) and a["layer"] == b["layer"]:
                ptr = lambda key: torch.tensor([a[key].data_ptr(), b[key].data_ptr()], dtype=torch.long, device=dev)
                y2 = torch.empty((2, 1, a["n"]), dtype=a["y"].dtype, device=dev)
                xh2 = torch.empty((2, 1, a["k"]), dtype=torch.half, device=dev)
                out.append(dict(kind="mgemm", x=a["x"].view(1, 1, -1), y=y2, xh=xh2, K=a["K"], reduce=False,
                                B=ptr("tr"), suh=ptr("suh"), svh=ptr("svh"), snl=None, cp=None, shared_inputs=2, mats=(a, b)))
                i += 2
            else:
                out.append(dict(kind="gemm", mt=a, reduce=a["reduce"]))
                i += 1
        return out

    def list_alg_bytes(self, launches):
        """Algorithmic bytes of a launch list: every matrix's own bytes, a shared input counted once (SURVEY.md 8d)."""
        b = sum(alg_bytes(1, t["k"], t["n"], t["K"], t["c_fp32"]) for t in self.mats)
        for ln in launches:
            if ln["kind"] == "mgemm":
                b -= 2 * ln["x"].shape[-1] * (ln["shared_inputs"] - 1)
        return b

    def outputs(self):
        """What the caller of the timed launch list receives after a step: every projection's output as float32, stacked
        over layers ({"q": (layers, 1, n), ..., "lm_head": (1, 1, vocab)}).  A two-matrix exl3_mgemm writes its own (2, 1, n)
        output; every other launch writes the matrix's y."""
        out_of = {id(mt): mt["y"] for mt in self.mats}
        if self.mode == "ops":
            for ln in self.launches:
                for j, mt in enumerate(ln.get("mats", ())):
                    out_of[id(mt)] = ln["y"][j]
        by_name = {}
        for mt in self.mats:
            by_name.setdefault(mt["name"], []).append(out_of[id(mt)])
        return {name: self.torch.stack(ys).float().cpu().numpy() for name, ys in by_name.items()}

    def build_chains(self, mode):
        """
        The same quantized linears as GEMM chains (ext.GemmChain, one persistent launch per chain) at the granularity of
          blocks   the reference's C++ block modules: q + k + v | o | gate + up -> silu * mul -> down  (BC_Attention's projections,
                   libtorch/attention.cpp:286-365; BC_GatedMLP, libtorch/mlp.cpp:14-91) + lm_head: 3 launches per layer
          layer    one launch per layer (q, k, v -> o -> gate, up -> down as four dependent stages), + lm_head
          token    the whole token as one launch
        with the data flow the shapes allow: o reads q's output (stand-in for the attention output, same shape), down reads
        silu(gate) * up of the gate / up outputs; where the model has non-GEMM ops in between (norms, attention) the chain still
        carries the DEPENDENCY (the next stage starts only after every output of the previous one is written), its input is the
        resident buffer of that matrix.  Row-parallel outputs (N > 1) end their chain: the all-reduce follows as its own launch.
        """
        ext = self.ext
        by_layer = {}
        for mt in self.mats:
            by_layer.setdefault(mt["layer"], {})[mt["name"]] = mt
        op = lambda mt, **kw: dict(trellis=mt["tr"], suh=mt["suh"], svh=mt["svh"], y=mt["y"], mul1=True, **kw)
        self.chain_items = []                 # (GemmChain, matrix whose output is all-reduced afterwards or None)
        token_ops = []
        nlayers = max(by_layer) + 1
        tp_on = self.tp > 1
        for l in range(nlayers):
            m_ = by_layer[l]
            q_in = m_["q"]["x"]
            qkv = [op(m_["q"], x=q_in), op(m_["k"], x=q_in), op(m_["v"], x=q_in)]
            o_ = op(m_["o"], x=m_["q"]["y"])
            gu_in = m_["gate"]["x"]
            gu = [op(m_["gate"], x=gu_in), op(m_["up"], x=gu_in)]
            dn = op(m_["down"], gate=m_["gate"]["y"], up=m_["up"]["y"], new_stage=True)
            if mode == "blocks" or tp_on:
                self.chain_items += [(ext.GemmChain(qkv), None), (ext.GemmChain([o_]), m_["o"] if m_["o"]["reduce"] else None),
                                     (ext.GemmChain(gu + [dn]), m_["down"] if m_["down"]["reduce"] else None)]
            else:
                ops = [dict(qkv[0], new_stage=l > 0 and mode == "token")] + qkv[1:] + [dict(o_, new_stage=True), dict(gu[0], new_stage=True), gu[1], dn]
                if mode == "layer":
                    self.chain_items.append((ext.GemmChain(ops), None))
                else:
                    token_ops += ops
        hd = by_layer[-1]["lm_head"]
        if mode == "token" and not tp_on:
            token_ops.append(op(hd, x=hd["x"], new_stage=True))
            self.chain_items.append((ext.GemmChain(token_ops), None))
        else:
            self.chain_items.append((ext.GemmChain([op(hd, x=hd["x"])]), None))
        self.launches = self.chain_items

    def run(self, launches=None):
        ext, dist = self.ext, None
        if self.mode != "ops":
            for ch, red in self.chain_items:
                ch.run()
                if red is not None and not self.skip_reduce:
                    import torch.distributed as dist
                    dist.all_reduce(red["y"])
            return
        for ln in (self.launches if launches is None else launches):
            if ln["kind"] == "gemm":
                mt = ln["mt"]
                if mt["reduce"] and self.fused_reduce:
                    ext.exl3_gemm_allreduce(mt["x"], mt["tr"], mt["y"], mt["suh"], None, mt["svh"], False, True)
                    continue
                ext.exl3_gemm(mt["x"], mt["tr"], mt["y"], mt["suh"], mt["xh"], mt["svh"], -1, False, True, 0)
                if mt["reduce"] and not self.skip_reduce:
                    import torch.distributed as dist
                    dist.all_reduce(mt["y"])
            else:
                ext.exl3_mgemm(ln["x"], ln["B"], ln["y"], ln["suh"], ln["xh"], ln["svh"], None, None, ln["K"], -1,
                               False, True, -1, -1, 0, 1, ln["snl"], ln["cp"])


def qgemm_section(tok, cfg, stream, hbm_peak):
    """
    The second half of BASELINE.json's metric, measured live on rank 0 at N = 1 AFTER the timed token (never inside it):
      decode_hbm      per matrix shape of the model, the batch-1 qgemm's achieved HBM GB/s = algorithmic bytes (SURVEY.md 8d) /
                      launch time, from one CUDA-graph replay of that shape's 32 layer instances back to back (distinct weight
                      buffers, 67-940 MB per shape; weights are loaded evict-first), CUDA events on the launching stream
      prefill_tensor  the prefill sibling of the same linear (reconstruct_had + tcgen05 dense GEMM, QLinear.forward for
                      rows > 144) at batch 32 x 2048 rows: achieved TFLOP/s (2 m k n) against the measured dense bf16 peaks
    """
    import torch
    from exllamav3_b200 import ext, QLinear
    out = {"decode_hbm": {}, "prefill_tensor": {}}
    by_name = {}
    for mt in tok.mats:
        by_name.setdefault(mt["name"], []).append(mt)
    for name, mats in by_name.items():
        def run():
            for mt in mats:
                ext.exl3_gemm(mt["x"], mt["tr"], mt["y"], mt["suh"], mt["xh"], mt["svh"], -1, False, True, 0)
        with torch.cuda.stream(stream):
            run()
        stream.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            run()
        reps = 3 if len(mats) > 1 else 6
        best = None
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                e0.record(stream)
                for _ in range(reps):
                    g.replay()
                e1.record(stream)
            e1.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / (reps * len(mats))
            best = us if best is None else min(best, us)
        mt = mats[0]
        b = alg_bytes(1, mt["k"], mt["n"], mt["K"], mt["c_fp32"])
        out["decode_hbm"][name] = {"k": mt["k"], "n": mt["n"], "K": mt["K"], "us_per_launch": round(best, 2),
                                   "GBps": round(b / best / 1e3, 1), "frac_of_hbm_peak": round(b / best / 1e3 / hbm_peak, 3),
                                   "distinct_weight_MB": round(len(mats) * mt["k"] * mt["n"] * mt["K"] / 8 / 1e6)}
        del g
    # batch 8 / 32 decode (BASELINE config 3) on the default path: exact tcgen05 kernel, one launch per call
    out["decode_batch"] = {}
    for name in ("q", "gate", "down"):
        mats = by_name[name]
        for m in (8, 32):
            mt0 = mats[0]
            xb = torch.randn((m, mt0["k"]), device=tok.dev).half(); xhb = torch.empty_like(xb)
            yb = torch.empty((m, mt0["n"]), dtype=torch.float if mt0["c_fp32"] else torch.half, device=tok.dev)
            tag = [0]
            def runb():
                for mt in mats:
                    tag[0] = ext.exl3_gemm(xb, mt["tr"], yb, mt["suh"], xhb, mt["svh"], -1, False, True, 0)
            with torch.cuda.stream(stream):
                runb()
            stream.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                runb()
            best = None
            for _ in range(3):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                with torch.cuda.stream(stream):
                    e0.record(stream); g.replay(); g.replay(); e1.record(stream)
                e1.synchronize()
                us = e0.elapsed_time(e1) * 1e3 / (2 * len(mats))
                best = us if best is None else min(best, us)
            b = alg_bytes(m, mt0["k"], mt0["n"], mt0["K"], mt0["c_fp32"])
            out["decode_batch"][f"{name}_m{m}"] = {"us_per_launch": round(best, 2), "GBps": round(b / best / 1e3, 1),
                                                    "frac_of_hbm_peak": round(b / best / 1e3 / hbm_peak, 3), "tag": int(tag[0])}
            del g
    # the other two codebooks at batch 1 (default path: exact tcgen05 kernel): same bytes, different decode
    out["decode_codebooks"] = {}
    for name in ("q", "gate"):
        mats = by_name[name]
        for cbn, mcg in (("3inst", False), ("mcg", True)):
            if name == "gate" and cbn == "mcg":
                continue
            tag = [0]
            def runc():
                for mt in mats:
                    tag[0] = ext.exl3_gemm(mt["x"], mt["tr"], mt["y"], mt["suh"], mt["xh"], mt["svh"], -1, mcg, False, 0)
            with torch.cuda.stream(stream):
                runc()
            stream.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                runc()
            best = None
            for _ in range(3):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                with torch.cuda.stream(stream):
                    e0.record(stream); g.replay(); g.replay(); e1.record(stream)
                e1.synchronize()
                us = e0.elapsed_time(e1) * 1e3 / (2 * len(mats))
                best = us if best is None else min(best, us)
            mt0 = mats[0]
            b = alg_bytes(1, mt0["k"], mt0["n"], mt0["K"], mt0["c_fp32"])
            out["decode_codebooks"][f"{name}_{cbn}"] = {"us_per_launch": round(best, 2), "GBps": round(b / best / 1e3, 1),
                                                        "frac_of_hbm_peak": round(b / best / 1e3 / hbm_peak, 3), "tag": int(tag[0])}
            del g
    # the reference's own CUDA kernels (unmodified sources compiled for sm_100a, oracle/_ref) on this GPU in this run, its default
    # configuration, same shapes and method (graph replay over >= 512 MB of rotated weight copies): the bar the kernels are held to
    ref_so = os.path.join(ROOT, "oracle", "_ref", "exl3_ref_ext.so")
    if os.path.exists(ref_so) and not os.environ.get("EXL3B_BENCH_NO_REF_CUDA"):
        try:
            import tempfile
            with tempfile.TemporaryDirectory() as td:
                env = dict(os.environ); env.update(REF_BENCH_SHAPES="decode", REF_BENCH_OUT=td, EXLLAMAV3_TUNE_CACHE=os.path.join(td, "tune"))
                r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "bench_ref_gpu.py"), "int8"], env=env,
                                   capture_output=True, text=True, timeout=300)
                res = json.load(open(os.path.join(td, "ref_bench_int8.json")))
            out["reference_cuda"] = {"what": "unmodified reference kernels (exllamav3_ext, default settings: its int8 GEMV for mul1 at m <= 2, "
                                             "mma.sync kernels otherwise), same GPU, same run, outside every timed region",
                                     "shapes": {(d["shape"] if " m=" in d["shape"] else f"{d['shape']} m={d['m']}"): {"us": round(d["us"], 2), "GBps": round(d["gbps"], 1)} for d in res}}
        except Exception as e:
            out["reference_cuda"] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
    else:
        out["reference_cuda"] = {"unavailable": "oracle/_ref/exl3_ref_ext.so not present (built only where the reference checkout exists)"}
    # weight materialisation kernels of the prefill sibling (reconstruct / reconstruct_had): write-dominated, K/8 + 2 bytes per weight
    out["reconstruct"] = {}
    for (k, n) in ((cfg["hidden"], cfg["q"]), (cfg["hidden"], cfg["inter"])):
        mt = next(t for t in tok.mats if t["k"] == k and t["n"] == n)
        w = torch.empty((k, n), dtype=torch.half, device=tok.dev)
        for nm, fn in (("reconstruct", lambda: ext.reconstruct(w, mt["tr"], mt["K"], False, True)),
                       ("reconstruct_had", lambda: ext.reconstruct_had_slice(w, mt["tr"], mt["suh"], mt["svh"], mt["K"], False, True, 0))):
            with torch.cuda.stream(stream):
                fn(); fn()
            stream.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                e0.record(stream)
                for _ in range(10):
                    fn()
                e1.record(stream)
            e1.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / 10
            b = k * n * (mt["K"] / 8 + 2)
            out["reconstruct"][f"{nm}_{k}x{n}"] = {"us": round(us, 2), "GBps": round(b / us / 1e3, 1), "frac_of_hbm_peak": round(b / us / 1e3 / hbm_peak, 3)}
        del w
    # prefill: batch 32 x seq 2048 rows through the reference-facing linear (rows > 144 -> reconstruct + dense GEMM)
    peaks = {}
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peaks = {"burst": float(d["bf16_tflops"]), "sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"]))}
    except Exception:
        peaks = {"burst": 2250.0, "sustained": 2250.0}          # nominal dense bf16 (B200_PROFILING.md fallback)
    dev = tok.dev
    gen = torch.Generator(device=dev); gen.manual_seed(7)
    h = cfg["hidden"]
    for (k, n, m) in ((h, cfg["q"], 32 * 2048), (h, cfg["inter"], 8 * 2048)):
        mt = next(t for t in tok.mats if t["k"] == k and t["n"] == n)
        lin = QLinear(mt["tr"], mt["suh"], mt["svh"], mul1=True)
        x = torch.randn((m, k), generator=gen, device=dev).half()
        with torch.cuda.stream(stream):
            for _ in range(2):
                y = lin.forward(x, {})
        stream.synchronize()
        it = 5
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(it):
                y = lin.forward(x, {})
            e1.record(stream)
        e1.synchronize()
        ms = e0.elapsed_time(e1) / it
        tf = 2.0 * m * k * n / ms / 1e9
        out["prefill_tensor"][f"{k}x{n}_m{m}"] = {"rows": m, "ms": round(ms, 3), "tflops": round(tf, 1),
                                                   "frac_of_measured_bf16_burst": round(tf / peaks["burst"], 3),
                                                   "frac_of_measured_bf16_sustained": round(tf / peaks["sustained"], 3),
                                                   "path": "reconstruct_had + tcgen05 dense GEMM (includes the weight reconstruction every call)"}
        del x, y, lin
    return out


NCU_CAPTURE = os.path.join("profiles", "r02_ncu_gate.csv")     # metric,unit,value rows of one --set full capture


def ncu_dram_bytes(path):
    """dram__bytes_read.sum + dram__bytes_write.sum of the committed ncu capture, in bytes (units as ncu printed them)."""
    import csv
    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    cap = {r[0]: (r[1], r[2]) for r in csv.reader(open(path)) if len(r) == 3}
    total = 0.0
    for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
        unit, val = cap[key]
        total += float(val) * mult[unit]
    return total


def ncu_traffic_per_launch(tok):
    """DRAM traffic of the dominant kernel from the committed ncu capture (profiles/): measured bytes / algorithmic bytes of
    the captured launch (gate shape), applied to the average launch of this step; None if the capture is missing."""
    try:
        return ncu_dram_bytes(os.path.join(ROOT, NCU_CAPTURE)) / alg_bytes(1, 4096, 14336, 4, True) * tok.alg_bytes / len(tok.launches)
    except Exception:
        return None


def dump_outputs(tok, out_dir):
    """The outputs of the last timed step as out_dir/<projection>.npy (float32; Llama-3.1-8B: 6.0 MB, 70B: 27.4 MB).  The inputs
    come from the seeded generator of Token, so two builds run with the same arguments can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in tok.outputs().items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def run_gpu_arm(args, cfg):
    import torch
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch N>1 with torch.distributed.run)"
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the EXL3 path has no CPU implementation (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from exllamav3_b200 import ext

    tok = Token(cfg, world if not args.tp_shapes else args.tp_shapes, rank, dev, fuse=not args.no_fuse, mode=args.mode, fanout=not args.no_fanout)
    if world > 1 and not args.nccl_allreduce and args.mode == "ops" and not args.tp_shapes:
        from exllamav3_b200 import tp as _tp
        try:
            _tp.enable_fused_allreduce(max_elems=4 * cfg["hidden"])
            tok.fused_reduce = True
        except Exception as e:                  # no peer access / IPC: every rank fails alike (collective setup), NCCL it is
            if rank == 0:
                print(f"# fused all-reduce unavailable ({type(e).__name__}: {e}); using NCCL", file=sys.stderr)
    if args.tp_shapes:
        # single-GPU dry run of ONE rank's shard of a TP-N token (kernel shapes only, no collective): not a bench result
        tok.skip_reduce = True
    stream = torch.cuda.Stream(device=dev)
    launches0 = ext.launch_count()
    with torch.cuda.stream(stream):
        for _ in range(2):
            tok.run()                       # eager warm-up: lazy context init, NCCL channels
    stream.synchronize()
    launches_per_step = (ext.launch_count() - launches0) // 2

    graph = None
    if not args.no_graph:
        try:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=stream):
                tok.run()
        except Exception as e:                # capture unsupported (e.g. NCCL config): eager launches
            if rank == 0:
                print(f"# graph capture failed ({type(e).__name__}: {e}); timing eager launches", file=sys.stderr)
            graph = None
            torch.cuda.synchronize()

    def step():
        if graph is not None:
            graph.replay()
        else:
            tok.run()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(steps):
                fn()
            e1.record(stream)
        e1.synchronize()
        barrier()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # clocks are sampled from the warm-up on (same load as the timed steps), so that even a short timed region has samples
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)                     # nvidia-smi start-up
    with torch.cuda.stream(stream):
        for _ in range(max(3, args.warmup)):
            step()
        if args.steps < 200:                # short timed region: keep the GPU under the same load a little longer first
            for _ in range(200):
                step()
    stream.synchronize()
    ms = timed(step, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = ms / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(tok, args.dump_outputs)

    # ---- the same token with the reference's Llama launch list (q, k+v as two calls), same run, same weights ----
    ref_list = None
    if tok.fanout and args.mode == "ops" and tok.launches_ref is not tok.launches:
        with torch.cuda.stream(stream):
            for _ in range(2):
                tok.run(tok.launches_ref)
        stream.synchronize()
        ref_fn = lambda: tok.run(tok.launches_ref)
        if graph is not None:
            try:
                g2 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g2, stream=stream):
                    tok.run(tok.launches_ref)
                ref_fn = g2.replay
            except Exception:
                torch.cuda.synchronize()
        with torch.cuda.stream(stream):
            for _ in range(3):
                ref_fn()
        ref_ms = timed(ref_fn, args.steps) / args.steps
        ref_list = {"launches": len(tok.launches_ref), "ms_per_step": ref_ms, "value": 1000.0 / ref_ms, "unit": "tok/s",
                    "what": "q_proj and k+v (exl3_mgemm) as two operator calls per layer, as modules/attn.py:555-631 issues them"}

    # ---- end-to-end through the operator surface with host buffers ----
    hx = torch.randn((1, cfg["hidden"])).half().pin_memory()
    hlogits = torch.empty(tuple(tok.logits.shape), dtype=tok.logits.dtype).pin_memory()

    def e2e_step():
        tok.first_x.copy_(hx, non_blocking=True)
        step()
        hlogits.copy_(tok.logits, non_blocking=True)
        stream.synchronize()                 # the host consumes the logits every token

    with torch.cuda.stream(stream):
        for _ in range(3):
            e2e_step()
    e2e_ms = timed(e2e_step, args.steps) / args.steps     # events bracket the loop; host round trips are inside
    # the same without the CUDA graph: one Python -> ctypes -> C ABI call per launch, what the reference's eager module path does
    e2e_eager_ms = None
    if graph is not None:
        def e2e_eager_step():
            tok.first_x.copy_(hx, non_blocking=True)
            tok.run()
            hlogits.copy_(tok.logits, non_blocking=True)
            stream.synchronize()
        n_eager = max(3, min(args.steps, 50))
        with torch.cuda.stream(stream):
            for _ in range(2):
                e2e_eager_step()
        e2e_eager_ms = timed(e2e_eager_step, n_eager) / n_eager

    peak, peak_src = read_peaks()
    achieved = tok.alg_bytes / (ms_per_step * 1e-3) / 1e9          # per rank (each rank streams its own shard)
    # DRAM traffic of the dominant kernel from the committed ncu capture (profiles/): measured bytes / algorithmic bytes
    # of the captured launch, applied to the average launch of this step
    traffic = ncu_traffic_per_launch(tok)
    cpu_baseline = None
    check = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        wps, cores, sample, first = cpu_path_time(cfg, budget_s=args.cpu_budget if args.cpu_budget > 0 else None)
        cpu_baseline = {"value": wps / weights_per_token(cfg), "unit": "tok/s", "cores": cores, "kind": "port",
                        "sample": sample}
        # validate the GPU path on the same matrix the CPU arm just computed (oracle as checker only)
        import numpy as np
        from oracle import exl3_oracle as orc
        y_cpu, name, k, n, K = first
        tr, suh, svh, x = orc.make_synthetic(k, n, K)
        T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        C = torch.empty((1, n), dtype=torch.float, device=dev)
        ext.exl3_gemm(T(x), T(tr), C, T(suh), torch.empty((1, k), dtype=torch.half, device=dev), T(svh), -1, False, True, 0)
        err = float(np.abs(C.cpu().numpy() - y_cpu).max() / np.abs(y_cpu).max())
        check = {"matrix": name, "max_rel_err_vs_cpu_path": err}
        assert err < 1e-2, f"GPU result deviates from the CPU path: {err}"

    qgemm = None
    if rank == 0 and world == 1 and not args.tp_shapes and not args.no_qgemm:
        try:
            qgemm = qgemm_section(tok, cfg, stream, peak)
        except Exception as e:                   # never lose the bench line over the supplementary section
            qgemm = {"error": f"{type(e).__name__}: {e}"}
            try:
                torch.cuda.synchronize()
            except Exception:
                pass

    if rank == 0:
        line = {
            "metric": "decode tok/s Llama-3.1-8B 4.0bpw b=1 (qgemm path)", "value": 1000.0 / ms_per_step, "unit": "tok/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": f"{args.model} EXL3 4.0bpw (lm_head 6bpw) b=1 decode: "
                                   f"{len(tok.mats)} quantized matrices/token in {len(tok.launches)} launches "
                                   + ("(q+k+v as one fan-out exl3_mgemm with per-matrix widths -- the operator's size_n_list / c_ptrs arguments, "
                                      "exl3_gemm.cu:402-447, used like the reference's libtorch/dsv4_attn.cpp:88-99 -- and gate+up as one exl3_mgemm; "
                                      "reference_launch_list = the same token with q and k+v as two calls, the reference's Llama module code), "
                                      if tok.fanout and args.mode == "ops" else
                                      "(k+v and gate+up as one exl3_mgemm each: what the reference's model code issues through this library's "
                                      "ext shim, model/config.py:48-64), ") +
                                   f"m=1, mul1 codebook, "
                                   f"random-init trellis",
                       "parallelism": (f"tp{world}" if world > 1 else "single") + (f" (DRY RUN of tp{args.tp_shapes} rank-0 shapes, no collective: not a result)" if args.tp_shapes else ""),
                       "l2": "weights per step (%.2f GB/rank) exceed L2 (126 MB); no flush needed" % (tok.alg_bytes / 1e9),
                       "cuda_graph": graph is not None,
                       "row_parallel_sum": ("fused into the GEMM epilogue over NVLink peer memory" if tok.fused_reduce else
                                            ("NCCL all-reduce per row-parallel output" if world > 1 else "none (single GPU)"))},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "kernel": "gemm_tc_i8_kernel (tcgen05 kind::i8 decode-GEMM)",
                         "note": "achieved = algorithmic bytes of the step / step time = average over the step's launches of the "
                                 "dominant kernel (it is 100 % of the launches, profiles/r02_launches.md); traffic = bytes per average "
                                 "launch scaled from this round's ncu --set full capture of the kernel on the gate shape "
                                 "(profiles/r02_ncu_gate.csv: 29.486 MB read for 29.46 MB algorithmic, ratio 1.001; q and lm_head "
                                 "captures beside it)"},
            "cpu_baseline": cpu_baseline,
            "e2e": {"value": 1000.0 / e2e_ms, "unit": "tok/s", "h2d_bytes_per_step": hx.numel() * 2,
                    "d2h_bytes_per_step": hlogits.numel() * hlogits.element_size(),
                    "eager_value": (1000.0 / e2e_eager_ms) if e2e_eager_ms else None,
                    "note": "value: CUDA-graph replay of the token between the host copies; eager_value: the same with one "
                            "Python -> ctypes -> C-ABI call per launch (no graph), as the reference's eager module path issues them"},
            "reference_launch_list": ref_list,
            "gpu_launches": launches_per_step * args.steps,
            "clocks": clocks,
            "check": check,
            "qgemm": qgemm,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        # Tear-down order matters: a CUDA graph holding captured NCCL kernels must die before the communicator, and
        # destroy_process_group() has been seen to hang after graph-captured collectives -- leave without it.
        del graph
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400, help="timed tokens (default: >= 1 s of timed region)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="llama-3.1-8b", choices=list(MODELS))
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--mode", default="ops", choices=["ops", "blocks", "layer", "token"],
                    help="ops: one exl3_gemm / exl3_mgemm launch per projection group (the reference's eager operator granularity); "
                         "blocks / layer / token: GEMM chains (one persistent launch per block, per layer, per token)")
    ap.add_argument("--no-fanout", action="store_true", help="q, k+v as two operator calls like the reference's Llama attention module (no q+k+v fan-out exl3_mgemm)")
    ap.add_argument("--no-fuse", action="store_true", help="one launch per projection (no exl3_mgemm for k+v / gate+up)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-qgemm", action="store_true", help="skip the per-shape qgemm GB/s + prefill tensor-pipe section (N = 1 only)")
    ap.add_argument("--fused-allreduce", action="store_true", help="(default for N > 1 since round 2; kept for old command lines)")
    ap.add_argument("--nccl-allreduce", action="store_true",
                    help="N > 1: row-parallel outputs as exl3_gemm + NCCL all-reduce (what the reference issues) instead of the one-kernel "
                         "exl3_gemm_allreduce")
    ap.add_argument("--tp-shapes", type=int, default=0, help="debug: run rank 0's shard shapes of a TP-N token on one GPU without the all-reduce")
    ap.add_argument("--cpu-budget", type=float, default=0.0, help="seconds; 0 = the fixed sample (all of layer 0)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write rank 0's outputs of the last timed step to DIR/<projection>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = MODELS[args.model]
    if args.impl == "reference":
        run_reference_arm(args, cfg)
    else:
        run_gpu_arm(args, cfg)


if __name__ == "__main__":
    main()
