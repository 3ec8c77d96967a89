#!/usr/bin/env python
"""bench.py -- MAC reasoning steps/sec on synthetic CLEVR-shaped batches (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--prec bf16|fp32] [--impl ours|reference] [--dump-outputs DIR]

A bench "step" is one full pass of the hot path over one batch: the netLength-step unroll of the MAC cell
(model.py:447-458) on B=64 questions -- 12 reasoning steps at the headline configuration (BASELINE.json
configs[2]: B=64, S=40, 14x14 KB, d=512, netLength=12).  `value` = reasoning steps/s = K * netLength * N / t.

  value   inputs resident in HBM when the timed region starts; the K timed passes rotate over 8 resident
          batches (8 x 31 MB > 126 MB L2) so the knowledge base comes from HBM every pass.  `--dump-outputs DIR`
          writes what the last of them returned (final control and memory, both attention maps) as DIR/<name>.npy,
          float32; inputs and weights are seeded, so two builds run with the same arguments can be compared.
  e2e     the same metric through the public API with HOST (pinned) buffers: per pass the H2D copy of the batch
          (KB, words, question vector, lengths) and the D2H read of the final state + attention maps are inside the
          timed region (double-buffered against compute on a copy stream).
  roofline / roofline_kb_attend   per-kernel, measured live with CUDA events around single launches (cold L2).
  cpu_baseline   the oracle's fp32 PyTorch-CPU port (oracle/mac_torch_cpu.py) timed on this box's host cores.

`--impl reference` times that CPU port alone (TensorFlow-1 cannot be installed offline; see DESIGN.md).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from mac_network_b200.config import MACConfig  # noqa: E402
from mac_network_b200.params import init_params, perturb_biases  # noqa: E402
from mac_network_b200.synthetic import SHAPES, make_inputs  # noqa: E402

def workload_string(shape):
    B, S, N, d, L = shape
    return ("BASELINE.json configs[2]: args.txt cell, B=%d/GPU, S=%d, KB=14x14 (N=%d), d=%d, netLength=%d, inference "
            "(dropouts=1.0)" % (B, S, N, d, L))


def timed_blocks(run_block, K, barrier, dist, min_total_s=0.5, max_blocks=400):
    """Time EXACTLY K steps per block (barrier + synchronize on both sides, CUDA events, max over ranks) and repeat the
    block until >= min_total_s of timed work has accumulated; returns (median block seconds, all block seconds).  Every
    rank takes the same number of blocks (the decision uses the all-reduced maximum)."""
    times, total = [], 0.0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    while True:
        barrier()
        e0.record()
        run_block(K)
        e1.record()
        barrier()
        t = e0.elapsed_time(e1) * 1e-3
        if dist is not None:
            tt = torch.tensor([t], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t = float(tt[0])
        times.append(t)
        total += t
        if total >= min_total_s or len(times) >= max_blocks:
            break
    return float(np.median(times)), times


METRIC = "mac_reasoning_steps_per_sec"
UNIT = "reasoning-steps/s"
WORKLOAD = "headline"            # BASELINE.json configs[2]
NSLOTS = 8


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm": p["hbm_gbs"], "tensor_burst": p["bf16_tflops"], "tensor_sustained": p["bf16_tflops_sustained"],
                "src": "measured (MEASURED_PEAKS.json)"}
    return {"hbm": 6650.0, "tensor_burst": 1590.0, "tensor_sustained": 1400.0, "src": "fallback (B200_PROFILING.md)"}


def local_device():
    """This rank's CUDA device: LOCAL_RANK, re-ordered so that a job of fewer ranks than GPUs spreads over the sockets
    (serving.device_for_rank: GPUs 0-3 hang off NUMA node 0 and 4-7 off node 1 on the 8-GPU boxes)."""
    from mac_network_b200.serving import device_for_rank
    lr = int(os.environ.get("LOCAL_RANK", "0"))
    return device_for_rank(lr, int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1"))))


class ClockSampler(object):
    """nvidia-smi sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        try:        # address the GPU by PCI bus id: the CUDA index is not nvidia-smi's when devices are masked / re-ordered
            prop = torch.cuda.get_device_properties(index)
            bus = "%08x:%02x:%02x.0" % (getattr(prop, "pci_domain_id", 0), prop.pci_bus_id, prop.pci_device_id)
            out = subprocess.run(["nvidia-smi", "-i", bus, "--query-gpu=index", "--format=csv,noheader"],
                                 capture_output=True, text=True, timeout=20)
            if out.returncode == 0 and out.stdout.strip().isdigit():
                self.index = int(out.stdout.strip())
        except Exception:
            pass

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU reference arm
def host_threads():
    """All the host threads the process can really use: min(affinity, cgroup quota), then the fastest of a few
    candidates on a proxy of the workload (a 128-thread pool on a quota-limited container only thrashes)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p) + 0.5)))
    except Exception:
        pass
    cands = sorted({c for c in (4, 8, 16, 32, 64, n) if c <= n})
    x = torch.randn(12544, 1024)
    w = torch.randn(1024, 512)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        torch.nn.functional.elu(x @ w)
        t0 = time.perf_counter()
        for _ in range(3):
            torch.nn.functional.elu(x @ w)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best, n


def cpu_reference(cfg, shape, params_np, budget_s=15.0, max_forwards=8):
    """The oracle's op-by-op fp32 CPU port on all host threads.  Returns reasoning-steps/s and a description."""
    from oracle.mac_torch_cpu import TorchCPUCell
    B, S, N, d, L = shape
    nthr, navail = host_threads()
    inp = make_inputs(B, S, N, d, seed=1234)
    cell = TorchCPUCell(cfg, params_np, L)
    args = (torch.from_numpy(inp["vecQuestions"]), torch.from_numpy(inp["questionCntxWords"]),
            torch.from_numpy(inp["questionLengths"]).long(), torch.from_numpy(inp["knowledgeBase"]))
    t0 = time.perf_counter()
    cell.forward(*args)                                 # warm-up (also sizes the sample)
    t1 = time.perf_counter() - t0
    n = int(max(1, min(max_forwards, budget_s / max(t1, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(n):
        cell.forward(*args)
    dt = (time.perf_counter() - t0) / n
    return {"value": L / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": "%d full forward passes (B=%d, netLength=%d) of the fp32 PyTorch-CPU port after 1 warm-up; "
                      "%.3f s per pass; %d threads (fastest of the candidates <= %d usable host threads)"
                      % (n, B, L, dt, nthr, navail)}, dt


# ------------------------------------------------------------------------------------------------ our arm
class Slot(object):
    """One resident batch + its cell + the captured CUDA graph of the netLength unroll."""

    def __init__(self, cfg, params, shape, seed, prec, use_graph, host_inputs=None, fold_y=None, small_tc=None):
        from mac_network_b200.mac_cell import MACCell, mac_network
        B, S, N, d, L = shape
        inp = host_inputs if host_inputs is not None else make_inputs(B, S, N, d, seed=seed)
        self.x = {k: torch.from_numpy(v).cuda() for k, v in inp.items()}
        x = self.x
        self.cell = MACCell(x["vecQuestions"], x["questionWords"], x["questionCntxWords"], x["questionLengths"],
                            x["knowledgeBase"], 1.0, 1.0, 1.0, B, False, config=cfg, params=params, prec=prec, fold_y=fold_y,
                            small_tc=small_tc)
        self.L = L
        self.graph = None
        self._net = mac_network
        self.run()                                        # warm-up: fills caches (packed weights, scalars, attrs)
        torch.cuda.synchronize()
        from mac_network_b200 import _lib
        n0 = _lib.load().mac_b200_launch_count()
        self.run()                                        # steady-state pass: count the kernels it launches
        torch.cuda.synchronize()
        self.launches = _lib.load().mac_b200_launch_count() - n0
        if use_graph:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._net(self.cell, self.L)
            self.graph = g

    def run(self):
        if self.graph is not None:
            self.graph.replay()
        else:
            self._net(self.cell, self.L)

    def outputs(self):
        """What a caller of the pass receives, under the names serving.HostPipeline returns them by."""
        c = self.cell
        return {"control": c._hc[self.L], "memory": c._hm[self.L], "att_kb": c._att_kb, "att_question": c._att_q}


def dump_outputs(outdir, outputs):
    os.makedirs(outdir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(outdir, name + ".npy"), t.float().cpu().numpy())


def ncu_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[key]["dram_bytes_per_launch"]
    except Exception:
        return None


def time_kernel(fns, iters=24, flush=None):
    """Average device time (s) per launch.  `fns` is a list of closures launching the SAME kernel on DIFFERENT
    buffers whose total footprint exceeds the 126 MB L2 (so every launch reads HBM); the launches are issued back
    to back and bracketed by one pair of CUDA events on the launching stream.  With `flush` given, each launch is
    instead timed alone after a cold-L2 flush (a 256 MB write)."""
    for f in fns:
        f()
    torch.cuda.synchronize()
    if flush is not None:
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
        for i, (a, b) in enumerate(ev):
            flush.zero_()
            a.record()
            fns[i % len(fns)]()
            b.record()
        torch.cuda.synchronize()
        return float(np.mean([a.elapsed_time(b) for a, b in ev])) * 1e-3
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        fns[i % len(fns)]()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e-3 / iters


def kernel_rooflines(shape, prec, pk):
    """Per-kernel rooflines measured live: K3 (KB attention, HBM-bound) and the dominant projection GEMM."""
    import ctypes
    from mac_network_b200 import _lib as L
    lib = L.load()
    B, S, N, d, _ = shape
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    out = {}
    NB = 12        # rotating input sets: 12 x 25.7 MB (fp32) / 12 x 12.8 MB (bf16) > 126 MB L2
    # ---- K3: softmax over the KB + weighted sum.  Algorithmic bytes (SURVEY 8(d)): KB once + logits in + att out + info out
    for name, bf16 in (("fp32_kb", 0), ("bf16_kb", 1)):
        kbs = [torch.randn(B, N, d, device="cuda") for _ in range(NB)]
        if bf16:
            kbs = [k.to(torch.bfloat16) for k in kbs]
        parts = torch.randn(B, N, 4, device="cuda")
        att = torch.empty(B, N, device="cuda")
        info = torch.empty(B, d, device="cuda")

        def mk(kbx):
            def k3():
                L.check(lib.mac_kb_attend_fwd(L.ptr(parts), 4, 0.0, L.ptr(kbx), bf16, L.ptr(att), L.ptr(info), B, N, d,
                                              L.stream_ptr()))
            return k3
        fns = [mk(k) for k in kbs]
        t = time_kernel(fns, iters=48)
        t_cold = time_kernel(fns, iters=12, flush=flush)
        nbytes = B * N * d * (2 if bf16 else 4) + B * N * 4 * 4 + B * N * 4 + B * d * 4
        out["kb_attend_" + name] = {"bound": "hbm", "achieved": nbytes / t / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                                    "frac": nbytes / t / 1e9 / pk["hbm"], "traffic": ncu_traffic("kb_attend_" + name),
                                    "us": t * 1e6,
                                    "algorithmic_bytes": nbytes,
                                    "l2": "launches rotate over %d knowledge bases (%.0f MB > 126 MB L2), back to back"
                                          % (NB, NB * B * N * d * (2 if bf16 else 4) / 1e6),
                                    "us_single_launch_after_256MB_write_flush": t_cold * 1e6}
        if not bf16:
            # context for the fraction: what plain streaming kernels of the SAME size reach when timed the same way
            # (MEASURED_PEAKS' denominator is a 2 GiB copy; a 26 MB launch pays launch + first-byte latency on ~4 us)
            srcs = [k.view(-1) for k in kbs]
            dst = torch.empty(srcs[0].numel() // 2, device="cuda")
            t_copy = time_kernel([(lambda s_=s_: dst.copy_(s_[:dst.numel()])) for s_ in srcs], iters=48)
            t_sum = time_kernel([(lambda s_=s_: torch.sum(s_)) for s_ in srcs], iters=48)
            out["kb_attend_" + name]["same_size_context"] = {
                "torch_copy_13MB_read_13MB_write_us": t_copy * 1e6, "torch_copy_frac_of_peak": nbytes / t_copy / 1e9 / pk["hbm"],
                "torch_sum_26MB_read_us": t_sum * 1e6, "torch_sum_frac_of_peak": nbytes / t_sum / 1e9 / pk["hbm"]}
        del kbs
    # ---- the same kernel with six requests' knowledge bases in ONE launch (B = 384, 78 MB bf16): informational -- separates
    #      "latency-bound at 13 MB per launch" from "inefficient kernel" (the headline K3 entry stays the B = 64 one above)
    try:
        Bb = 6 * B
        kbs6 = [torch.randn(Bb, N, d, device="cuda").to(torch.bfloat16) for _ in range(3)]          # 3 x 77 MB > L2
        parts6 = torch.randn(Bb, N, 4, device="cuda")
        att6, info6 = torch.empty(Bb, N, device="cuda"), torch.empty(Bb, d, device="cuda")
        fns6 = [(lambda k_=k_: L.check(lib.mac_kb_attend_fwd(L.ptr(parts6), 4, 0.0, L.ptr(k_), 1, L.ptr(att6), L.ptr(info6), Bb,
                                                              N, d, L.stream_ptr()))) for k_ in kbs6]
        t6 = time_kernel(fns6, iters=24)
        nb6 = Bb * N * d * 2 + Bb * N * 4 * 4 + Bb * N * 4 + Bb * d * 4
        out["kb_attend_bf16_kb_x6_rows"] = {"bound": "hbm", "achieved": nb6 / t6 / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                                            "frac": nb6 / t6 / 1e9 / pk["hbm"], "traffic": None, "us": t6 * 1e6,
                                            "algorithmic_bytes": nb6,
                                            "note": "informational: B = %d rows per launch (six B = 64 requests), same kernel" % Bb}
        del kbs6
    except Exception as exc:
        out["kb_attend_bf16_kb_x6_rows"] = {"error": repr(exc)[:200]}
    # ---- dominant projection GEMM: memKbProj, [B*N, 2d] x [2d, d] (49.6 % of the step's FLOPs)
    M, K = B * N, 2 * d
    xs = [torch.randn(M, K, device="cuda") for _ in range(3)]
    W = torch.randn(K, d, device="cuda") / K ** 0.5
    bias = torch.zeros(d, device="cuda")
    y = torch.empty(M, d, device="cuda")
    arr_k = (ctypes.c_int * 1)(K)

    def mkg(x):
        arr_p = (ctypes.c_void_p * 1)(x.data_ptr())

        def gemm():
            L.check(lib.mac_linear_fwd(arr_p, arr_k, arr_k, 1, L.ptr(W), L.ptr(bias), 0.0, 3, L.ptr(y), d, M, d, None,
                                       0, L.stream_ptr()))
        return gemm
    t = time_kernel([mkg(x) for x in xs], iters=9)
    flops = 2.0 * M * K * d
    out["memKbProj_gemm_fp32"] = {"bound": "tensor", "achieved": flops / t / 1e12, "peak": pk["tensor_burst"],
                                  "unit": "TFLOP/s", "frac": flops / t / 1e12 / pk["tensor_burst"], "traffic": None,
                                  "us": t * 1e6, "note": "fp32 FMA-pipe kernel (parity path) against the bf16 tensor peak"}
    del xs
    # ---- the same projection on tensor cores (tcgen05.mma, bf16 operands, fp32 accumulate in TMEM)
    xb = [torch.randn(M, K, device="cuda").to(torch.bfloat16) for _ in range(6)]      # 6 x 25.7 MB > L2
    Wt = torch.empty(d, K, dtype=torch.bfloat16, device="cuda")
    L.check(lib.mac_pack_weight_bf16(L.ptr(W), L.ptr(Wt), K, d, L.stream_ptr()))

    yb = torch.empty(M, d, device="cuda", dtype=torch.bfloat16)

    def mkt(x):
        def gemm():   # the form the read unit uses: ELU epilogue, bf16 output
            L.check(lib.mac_linear_tc_fwd(L.ptr(x), L.ptr(Wt), L.ptr(bias), 3, L.ptr(yb), 1, M, K, d, L.stream_ptr()))
        return gemm
    t = time_kernel([mkt(x) for x in xb], iters=30)
    out["memKbProj_gemm_tc"] = {"bound": "tensor", "achieved": flops / t / 1e12, "peak": pk["tensor_burst"],
                                "unit": "TFLOP/s", "frac": flops / t / 1e12 / pk["tensor_burst"],
                                "traffic": ncu_traffic("tc_gemm_memKbProj"), "us": t * 1e6, "algorithmic_flops": flops,
                                "note": "tcgen05 UMMA, H = ELU([12544,1024] @ [1024,512] + b) bf16 in / bf16 out, "
                                        "fp32 accumulate in TMEM; A rotates over 6 buffers (154 MB > L2); burst peak"}
    # ---- the per-step form of the same projection in inference: P and Q = P @ Wm[d:2d] + bm are hoisted out of the
    #      netLength loop (mac_read_invariant), each step runs H = ELU((P*y) @ Wm[0:d] + Q): K = d.  With bf16 in/out this
    #      GEMM is below the ridge point (AI = 2MKN / 2(MK + 2MN) = K/3 ... 171 FLOP/B < peak_tensor / peak_hbm), i.e.
    #      HBM-bound on the roofline; both views are reported.
    Kh = d
    xh = [x[:, :Kh].contiguous() for x in xb]                                            # 6 x 12.8 MB
    Wth = Wt[:, :Kh].contiguous()
    t = time_kernel([(lambda x=x: L.check(lib.mac_linear_tc_fwd(L.ptr(x), L.ptr(Wth), L.ptr(bias), 3, L.ptr(yb), 1, M, Kh,
                                                                 d, L.stream_ptr()))) for x in xh], iters=30)
    hflops = 2.0 * M * Kh * d
    hbytes = 2.0 * (M * Kh + 2 * M * d + Kh * d)          # A in, addend Q in, H out, weights (bf16)
    t_hbm, t_tc = hbytes / (pk["hbm"] * 1e9), hflops / (pk["tensor_burst"] * 1e12)
    out["memKbProj_step_gemm_tc"] = {
        "bound": "hbm" if t_hbm >= t_tc else "tensor",
        "achieved": hbytes / t / 1e9 if t_hbm >= t_tc else hflops / t / 1e12,
        "peak": pk["hbm"] if t_hbm >= t_tc else pk["tensor_burst"], "unit": "GB/s" if t_hbm >= t_tc else "TFLOP/s",
        "frac": max(t_hbm, t_tc) / t, "traffic": ncu_traffic("tc_gemm_memKbProj_step"), "us": t * 1e6,
        "algorithmic_bytes": hbytes, "algorithmic_flops": hflops, "tflops": hflops / t / 1e12,
        "note": "tcgen05 UMMA, ELU([12544,512] @ [512,512] (+ Q)) bf16 in / bf16 out; timed through mac_linear_tc_fwd "
                "(same kernel template, bias instead of the Q addend); A rotates over 6 buffers"}
    del xb, xh
    # ---- the inference read step as ONE kernel (csrc/read_step.cuh): scale + both projections + logits + softmax + KB
    #      weighted sum.  The REAL kernel, on rotating inputs: NR sets of (P, Q, KB) bf16 = NR x 38.5 MB > L2, and rotating
    #      y / control / outputs.  Algorithmic work per launch (SURVEY 8(d), hoisted inference form): 4*B*N*d^2 flops
    #      (two [B*N,d]x[d,d] products); bytes = P + Q + KB (bf16) + both weights + y, control in + att, info out.
    try:
        if lib.mac_read_step_fused_supported(B, N, d):
            NR = 6
            g = torch.Generator(device="cuda").manual_seed(5)
            Wr = {k: (torch.randn(*shp, device="cuda", generator=g) * sc).contiguous() for k, shp, sc in (
                ("Wx", (d, d), d ** -0.5), ("bx", (d,), 0.1), ("Wy", (d, d), d ** -0.5), ("by", (d,), 0.1),
                ("Wm", (2 * d, d), (2 * d) ** -0.5), ("bm", (d,), 0.1), ("Wm2", (d, d), d ** -0.5), ("bm2", (d,), 0.1),
                ("wr", (d,), 4 * d ** -0.5))}
            W16 = []
            for k in ("Wx", "Wm", "Wm2"):
                o = torch.empty((Wr[k].shape[1], Wr[k].shape[0]), dtype=torch.bfloat16, device="cuda")
                L.check(lib.mac_pack_weight_bf16(L.ptr(Wr[k]), L.ptr(o), Wr[k].shape[0], Wr[k].shape[1], L.stream_ptr()))
                W16.append(o)
            rw = L.ReadWeights(Wr["Wx"].data_ptr(), Wr["bx"].data_ptr(), Wr["Wy"].data_ptr(), Wr["by"].data_ptr(),
                               Wr["Wm"].data_ptr(), Wr["bm"].data_ptr(), Wr["Wm2"].data_ptr(), Wr["bm2"].data_ptr(),
                               Wr["wr"].data_ptr(), 0.1, W16[0].data_ptr(), W16[1].data_ptr(), W16[2].data_ptr())
            sets = []
            nbi = lib.mac_read_invariant_bytes(B, N, d, 1)
            for _ in range(NR):
                kbx = torch.nn.functional.elu(torch.randn(B, N, d, device="cuda", generator=g)).to(torch.bfloat16).contiguous()
                inv = torch.empty(nbi, dtype=torch.uint8, device="cuda")
                L.check(lib.mac_read_invariant(None, L.ptr(kbx), ctypes.byref(rw), 1, L.ptr(inv), nbi, B, N, d, L.stream_ptr()))
                sets.append((kbx, inv, torch.randn(B, d, device="cuda", generator=g), torch.randn(B, d, device="cuda", generator=g),
                             torch.empty(B, d, device="cuda"), torch.empty(B, N, device="cuda")))

            def mkr(sx):
                kbx, inv, yy, cc, info_o, att_o = sx

                def rs():
                    L.check(lib.mac_read_step_fused(L.ptr(inv), L.ptr(kbx), L.ptr(yy), L.ptr(cc), ctypes.byref(rw),
                                                    L.ptr(info_o), L.ptr(att_o), B, N, d, L.stream_ptr()))
                return rs
            fns = [mkr(sx) for sx in sets]
            # the dominant kernel alone: profiling flag 8 skips the ~2 us combine launch that follows it in the packed form
            # (its outputs are then unmerged partials; nothing reads them here); the pair is timed too and reported beside it
            raw_lib = ctypes.CDLL(L.LIB_PATH)
            t_pair = time_kernel(fns, iters=60)
            raw_lib.mac_dbg_read_step_flags(8)
            try:
                t = time_kernel(fns, iters=60)
                t_cold = time_kernel(fns, iters=12, flush=flush)
            finally:
                raw_lib.mac_dbg_read_step_flags(0)
            Mr = B * N
            rflops = 4.0 * Mr * d * d
            rbytes = 3.0 * Mr * d * 2 + 2.0 * d * d * 2 + 2.0 * B * d * 4 + B * N * 4 + B * d * 4
            t_hbm, t_tc = rbytes / (pk["hbm"] * 1e9), rflops / (pk["tensor_burst"] * 1e12)
            out["read_step_fused"] = {
                "bound": "tensor" if t_tc >= t_hbm else "hbm",
                "achieved": rflops / t / 1e12 if t_tc >= t_hbm else rbytes / t / 1e9,
                "peak": pk["tensor_burst"] if t_tc >= t_hbm else pk["hbm"], "unit": "TFLOP/s" if t_tc >= t_hbm else "GB/s",
                "frac": max(t_hbm, t_tc) / t, "traffic": ncu_traffic("read_step_fused"), "us": t * 1e6,
                "us_single_launch_after_256MB_write_flush": t_cold * 1e6,
                "us_with_combine_kernel": t_pair * 1e6, "ctas": (Mr + 127) // 128 if N > 128 else None,
                # the packed kernel launches ceil(B*N/128) CTAs (1 per SM) and leaves the other SMs to the next pass's kernels:
                # the same fraction against the roof of the SMs it occupies (informational; `frac` is against the whole GPU)
                "frac_of_occupied_sms": (max(t_hbm, t_tc) / t) * (148.0 / max(1, min(148, (Mr + 127) // 128))) if N > 128 else None,
                "algorithmic_flops": rflops, "algorithmic_bytes": rbytes, "hbm_gbs": rbytes / t / 1e9,
                "hbm_frac": rbytes / t / 1e9 / pk["hbm"], "tflops": rflops / t / 1e12,
                "l2": "launches rotate over %d input sets (%.0f MB of bf16 P, Q, KB > 126 MB L2), back to back" % (NR, NR * 3 * Mr * d * 2 / 1e6),
                "note": "ONE launch per reasoning step: (P*y) @ Wm[0:d] + Q -> ELU -> @ Wm2 -> logits -> softmax -> sum att*KB; "
                        "tcgen05 cta_group::2 pairs over PACKED 128-row tiles (ceil(B*N/128) CTAs, no padded rows for N > 128), "
                        "fp32 accumulators fill TMEM (128 x 512), H stays in shared memory, per-sample softmax partials merged by "
                        "a B-CTA combine kernel (inside the timed launch pair); flops are the ALGORITHMIC 4*B*N*d^2"}
            del sets
    except Exception as exc:
        out["read_step_fused"] = {"error": repr(exc)[:300]}
    # ---- "next" row: the image stem that produces the knowledge base (2 x conv3x3 as im2col + tcgen05 GEMM)
    try:
        from mac_network_b200.stem import Stem, stem_specs, init_stem_params
        sp = {k: torch.from_numpy(v).cuda() for k, v in init_stem_params(stem_specs(1024, d), seed=3).items()}
        stem = Stem(sp, relu="ELU", prec="bf16")
        imgs = [torch.relu(torch.randn(B, 14, 14, 1024, device="cuda")) for _ in range(3)]     # 3 x 51 MB
        t = time_kernel([(lambda im=im: stem.forward(im)) for im in imgs], iters=6)
        sflops = 2.0 * B * 196 * 9 * (1024 * d + d * d)
        out["stem_forward_tc"] = {"bound": "tensor", "achieved": sflops / t / 1e12, "peak": pk["tensor_burst"],
                                  "unit": "TFLOP/s", "frac": sflops / t / 1e12 / pk["tensor_burst"], "traffic": None,
                                  "us": t * 1e6, "algorithmic_flops": sflops,
                                  "note": "stem (model.py:165-204): 2 x [fused im2col -> tcgen05 GEMM + ELU], bf16 operands"}
    except Exception as exc:                      # the stem is a 'next' row: never let it break the headline line
        out["stem_forward_tc"] = {"error": repr(exc)[:200]}
    return out


def h2d_probe_gbs(mb=128):
    """Pinned-host -> device copy bandwidth of this rank with nothing else running (after NUMA binding): what the end-to-end
    line's H2D of the batches can get at best."""
    try:
        src = torch.empty(mb << 20, dtype=torch.uint8).pin_memory()
        dst = torch.empty(mb << 20, dtype=torch.uint8, device="cuda")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(4):
            dst.copy_(src, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        return round(4 * (mb << 20) / (e0.elapsed_time(e1) * 1e-3) / 1e9, 1)
    except Exception:          # noqa: BLE001 -- informational
        return None


def cast_threads_for(world, numa):
    """Host-cast pool size of one rank: its share of the CPUs it may run on.  After NUMA binding the affinity mask is one
    socket, shared by the ranks whose GPUs hang off it (half of the ranks on a 2-socket box); a cgroup quota caps the total."""
    from mac_network_b200.serving import usable_cpus
    n = usable_cpus()
    sharing = max(1, (world + 1) // 2) if numa.get("bound") and world > 1 else max(1, world)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, int(float(q) / float(per)) // max(1, world) * sharing)
    except Exception:
        pass
    return max(1, min(12, (n - sharing) // sharing))


def run_ours(args):
    from mac_network_b200 import _lib
    from mac_network_b200.mac_cell import MACParams
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = local_device()
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = _lib.load()
    # one process per GPU: stay on the GPU's NUMA node before any host thread / pinned buffer exists.  Single-rank runs too: a
    # process that happens to start on the other socket stages every batch across the socket interconnect (H2D measured at
    # 39 GB/s instead of the link's ~52: the end-to-end line of one rank was copy-bound, not kernel-bound)
    numa = {"bound": False, "why": "MAC_NO_NUMA_BIND=1"}
    if os.environ.get("MAC_NO_NUMA_BIND", "0") != "1":
        from mac_network_b200.serving import bind_to_gpu_numa
        numa = bind_to_gpu_numa(local)
    # how many ranks stage their batches through this rank's socket (they share its memory bandwidth)
    ranks_on_node = 1
    if dist is not None:
        nodes = [None] * world
        dist.all_gather_object(nodes, numa.get("numa_node", -1))
        ranks_on_node = max(1, sum(1 for x in nodes if x == numa.get("numa_node", -1)))
    numa["ranks_on_node"] = ranks_on_node
    numa["cuda_device"] = local
    numa["h2d_gbs_alone"] = h2d_probe_gbs()
    shape = SHAPES[WORKLOAD]
    B, S, N, d, L = shape
    cfg = MACConfig.args("args", netLength=L)
    pv = perturb_biases(init_params(cfg, L, seed=100), seed=101)
    params = MACParams(cfg, L, values=pv)
    pk = peaks()
    use_graph = not args.no_graph

    # ---- resident-input arm
    nstreams = max(1, args.streams)
    fold_y = (nstreams < 4) if args.fold_y < 0 else bool(args.fold_y)     # see MACCell.__init__: latency vs throughput form
    small_tc = nstreams >= 2        # several passes in flight: tensor-core form of the batch-sized projections (MACCell.__init__)
    nslots = max(NSLOTS, nstreams)   # a resident batch (and its captured graph) is replayed by ONE stream at a time
    slots = [Slot(cfg, params, shape, 1234 + 1000 * rank + s, args.prec, use_graph, fold_y=fold_y, small_tc=small_tc)
             for s in range(nslots)]
    launches_per_pass = slots[0].launches

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # `--streams S`: S independent passes (different resident batches) in flight at once, each on its own stream.
    # A pass is one serial dependency chain whose small kernels leave most SMs idle; a second chain fills them.
    side = [torch.cuda.Stream() for _ in range(nstreams - 1)]
    main_stream = torch.cuda.current_stream()

    def run_passes(n):
        if nstreams == 1:
            for k in range(n):
                slots[k % nslots].run()
            return
        fork = torch.cuda.Event()
        fork.record(main_stream)
        for st in side:
            st.wait_event(fork)
        for k in range(n):
            j = k % nstreams
            if j == 0:
                slots[k % nslots].run()
            else:
                with torch.cuda.stream(side[j - 1]):
                    slots[k % nslots].run()
        for st in side:
            ev = torch.cuda.Event()
            ev.record(st)
            main_stream.wait_event(ev)

    run_passes(max(args.warmup, nstreams))
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # K = --steps passes per block, blocks repeated until >= --min-time s of device time (default: one block): the reported
    # time is the MEDIAN block
    t_dev, dev_blocks = timed_blocks(run_passes, args.steps, barrier, dist, min_total_s=args.min_time)
    # the sampler stops HERE: polling nvidia-smi through the host-driven end-to-end region below costs it ~15 % (19.8k vs
    # 23.5k reasoning-steps/s on the B200 box, profiles/r1/NOTES.md) -- the queries contend with the copy / launch calls
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:       # every block runs passes 0..K-1, so pass K-1 used slot (K-1) % nslots last
        dump_outputs(args.dump_outputs, slots[(args.steps - 1) % nslots].outputs())

    # ---- end-to-end arm: host (pinned) buffers; every pass does H2D of its batch, the netLength unroll, and D2H of the
    #      final state + attention maps.  ND device slots, each on its own stream, so the copies of one pass overlap the
    #      compute of the others (the public-API pattern for streaming batches).
    ND = max(2, nstreams)
    from mac_network_b200.serving import HostPipeline, usable_cpus
    host = []
    for s in range(4):
        inp = make_inputs(B, S, N, d, seed=777 + 1000 * rank + s)
        host.append({k: torch.from_numpy(v).pin_memory() for k, v in inp.items() if k != "questionWords"})
    del slots
    torch.cuda.empty_cache()
    pipe = HostPipeline(cfg, params, shape, prec=args.prec, slots=ND, use_graph=use_graph, fold_y=fold_y,
                        cast_threads=cast_threads_for(world, numa),
                        # host bf16 cast while at most two ranks stage through one socket (its staging ring stays in the
                        # last-level cache: 43.4k vs 40.0k without the cast at 2 ranks / socket); with more, fp32 over PCIe
                        host_cast=None if (ranks_on_node <= 2 or os.environ.get("MAC_FORCE_HOST_CAST", "0") == "1")
                        else False, stage_ring=3 if ranks_on_node <= 1 else 2)
    h2d_bytes, d2h_bytes = pipe.h2d_bytes, pipe.d2h_bytes
    e2e_host_cast, e2e_cast_threads, pipe_cast_ms = pipe.host_kb_bf16, pipe.cast_threads, pipe.cast_ms

    def e2e_passes(n):
        pipe.after(main_stream)
        for k in range(n):
            pipe.submit(host[k % len(host)], next_batch=host[(k + 1) % len(host)])
        pipe.wait_streams(main_stream)

    e2e_passes(max(args.warmup, ND))
    t_e2e, e2e_blocks = timed_blocks(e2e_passes, args.steps, barrier, dist, min_total_s=args.min_time)

    # ---- data-parallel training arm (all ranks take part: it contains the path's one collective)
    train = train_full = train_tc = batched = sub_lines = None
    if not args.skip_train:
        del pipe
        torch.cuda.empty_cache()
        train = train_arm(min(args.steps, 4), 2, rank, world, dist)
        if world == 1:                       # whole-model arm at N=1 only (like the CPU baseline): a rank-local failure of a
            try:                             # 'next' row inside a collective must never cost the N>1 headline lines
                train_full = train_full_arm(min(args.steps, 3), 2, rank, world, dist)
            except Exception as exc:
                train_full = {"error": repr(exc)[:300]}
        else:
            train_full = {"skipped": "measured at N=1 only; the N>1 lines carry the cell's DP-training arm (`train`)"}
        if world == 1:
            # sub-lines (VERDICT r1 'missing' #1, #6): the two paths inside the 1e-4 parity bar at the headline shape -- tc32 =
            # split-bf16 products on tcgen05 (6e-7 measured), fp32 = the SIMT FMA path (7e-7) -- and the GQA-shaped variant
            # (BASELINE configs[4]: 7x7 grid, self-attention + gate, netLength 6), resident inputs, measured in child processes
            sub_lines = {"tc32_headline": child_measure(["--mode", "quick", "--prec", "tc32", "--streams", "4", "--steps", "12",
                                                         "--warmup", "3"], timeout_s=120),
                         "fp32_headline": child_measure(["--mode", "quick", "--prec", "fp32", "--streams", "4", "--steps", "8",
                                                         "--warmup", "3"], timeout_s=120),
                         "bf16_gqa": child_measure(["--mode", "quick", "--workload", "gqa", "--streams", "12", "--steps", "24",
                                                    "--warmup", "6"], timeout_s=120),
                         "fp32_gqa": child_measure(["--mode", "quick", "--workload", "gqa", "--prec", "fp32", "--streams", "4",
                                                    "--steps", "12", "--warmup", "3"], timeout_s=120)}
            train_tc = {"note": "since round 2 the `train` entry above IS the tensor-core form (bf16 forward, tcgen05 backward products); "
                                "MAC_TRAIN_FP32=1 measures the all-fp32 SIMT form (38.8 ms per step: forward 12.3 + backward 26.5)"}
            # informational (NOT the headline configuration): six B=64 requests concatenated into one B=384 pass -- what
            # dynamic batching across requests would buy over independent passes in flight; measured in a child process
            batched = {"requests_x6_one_stream": child_measure(["--mode", "quick", "--batch-mult", "6", "--streams", "1",
                                                                 "--steps", "12", "--warmup", "3"]),
                       "requests_x6_two_streams": child_measure(["--mode", "quick", "--batch-mult", "6", "--streams", "2",
                                                                  "--steps", "12", "--warmup", "4"])}

    if rank == 0:
        roofs = kernel_rooflines(shape, args.prec, pk)
        if args.skip_cpu or world > 1:      # the CPU baseline is timed at N=1 only (rank 0)
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port",
                   "sample": "skipped (--skip-cpu)" if args.skip_cpu else "timed at N=1 only"}
        else:
            cpu, _ = cpu_reference(cfg, shape, pv)
        value = args.steps * L * world / t_dev
        dom = "memKbProj_gemm_fp32" if args.prec == "fp32" else (
            "read_step_fused" if "frac" in roofs.get("read_step_fused", {}) else "memKbProj_step_gemm_tc")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32" if args.prec == "fp32" else "bf16",
            "data": "synthetic",
            "config": {"workload": workload_string(shape),
                       "step": "one netLength-step unroll over one batch (%d reasoning steps)" % L,
                       "timing": "blocks of exactly --steps passes (barrier + synchronize on both sides, CUDA events, max over "
                                 "ranks), repeated until >= %.2f s (0: one block); ms_per_step / value are the MEDIAN block"
                                 % args.min_time,
                       "l2": "timed passes rotate over %d resident batches (%.0f MB > 126 MB L2)"
                             % (nslots, nslots * (B * N * d + B * S * d) * 4 / 1e6),
                       "cuda_graph": use_graph, "projections": args.prec, "concurrent_passes": nstreams,
                       "write_unit_folded_with_next_projY": bool(fold_y or small_tc),
                       "batch_sized_projections": "tcgen05, 3-pass split bf16 (fp32-class accuracy)" if small_tc else "fp32 cluster kernel",
                       "read_step": "one fused launch per reasoning step (csrc/read_step.cuh)", "parallelism": "dp%d (replicas, no "
                       "data-path collective in inference)" % world},
            "sample_steps_per_sec": value * B,
            "timed_blocks": {"resident": {"blocks": len(dev_blocks), "total_s": float(np.sum(dev_blocks)),
                                          "block_ms_min_median_max": [min(dev_blocks) * 1e3, t_dev * 1e3, max(dev_blocks) * 1e3]},
                             "e2e": {"blocks": len(e2e_blocks), "total_s": float(np.sum(e2e_blocks)),
                                     "block_ms_min_median_max": [min(e2e_blocks) * 1e3, t_e2e * 1e3, max(e2e_blocks) * 1e3]}},
            "e2e": {"value": args.steps * L * world / t_e2e, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": d2h_bytes, "ms_per_step": t_e2e / args.steps * 1e3,
                    "api": "mac_network_b200.serving.HostPipeline.submit (pinned host fp32 in, pinned host out)",
                    "numa": numa,
                    "host_cast": ("knowledge base fp32 -> bf16 on %d host threads inside the timed region (%.2f ms "
                                  "per batch when timed alone); H2D moves 2 B per KB element"
                                  % (e2e_cast_threads, pipe_cast_ms or 0.0)) if e2e_host_cast
                                 else "off (fp32 knowledge base over PCIe; host cast alone took %s ms on %d threads)"
                                      % (pipe_cast_ms, e2e_cast_threads)},
            "gpu_launches": int(launches_per_pass) * args.steps,
            "clocks": clocks,
            "roofline": roofs.get(dom, roofs["memKbProj_gemm_fp32"]),
            "roofline_kb_attend": dict(roofs["kb_attend_bf16_kb" if args.prec == "bf16" else "kb_attend_fp32_kb"],
                                       status=("standalone K3 kernel (training / fp32 / unsupported shapes); in the bf16 inference "
                                               "form its work is the tail of read_step_fused, whose roofline line carries the KB bytes")),
            "rooflines_all": roofs,
            "peaks": pk,
            "cpu_baseline": cpu,
            "train": train,
            "train_full": train_full,
            "train_tc": train_tc,
            "info_batched_requests": batched,
            "sub_lines": sub_lines,
        }
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def train_arm(steps, warmup, rank, world, dist):
    """Short DP-training measurement used inside the default (inference) bench line: returns a dict or None."""
    from mac_network_b200.dp import DPTrainer
    shape = SHAPES[WORKLOAD]
    B, S, N, d, L = shape
    cfg = MACConfig.args("args", netLength=L)
    pv = perturb_biases(init_params(cfg, L, seed=100), seed=101)
    # read unit's forward and backward products on tcgen05 tensor cores (bf16 operands, fp32 accumulation / master weights /
    # optimizer state): the DP default since round 2 (gated by tests/test_zzz_tensor_core_training.py); MAC_TRAIN_FP32=1
    # measures the all-fp32 SIMT form instead (38.9 ms per step in round 1)
    tc = os.environ.get("MAC_TRAIN_FP32", "0") != "1"
    tr = DPTrainer(cfg, L, param_values=pv, seed=7, rank=rank, world=world, classifier=(28, [512]),   # CLEVR: 28 answers
                   prec="bf16" if tc else "fp32", bwd_tc=tc)
    inp = make_inputs(B, S, N, d, seed=4321 + 1000 * rank)
    batch = {k: torch.from_numpy(v).cuda() for k, v in inp.items()}
    answers = torch.from_numpy(np.random.RandomState(5 + rank).randint(0, 28, size=(B,)).astype(np.int32)).cuda()
    for _ in range(warmup):
        tr.train_step_answers(0, batch, answers, B * world)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        tr.train_step_answers(0, batch, answers, B * world)
    e1.record()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) * 1e-3
    sync = True
    if dist is not None:
        tt = torch.tensor([t], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t = float(tt[0])
        chk = torch.stack([tr.params.flat.double().sum(), tr.params.flat.double().abs().sum()])
        allc = [torch.zeros_like(chk) for _ in range(world)]
        dist.all_gather(allc, chk)
        sync = all(bool(torch.equal(allc[0], c)) for c in allc)
    out = {"value": steps * L * world / t, "unit": UNIT, "ms_per_step": t / steps * 1e3, "steps": steps,
           "what": "DP training step: train-mode cell forward + output unit + mean softmax-CE over the global batch + hand-written "
                   "backward + all-reduce of the flat gradient bucket (%.1f MB, NCCL) + fused clip/Adam/EMA; B=%d per GPU, %s"
                   % (tr.params.numel * 4 / 1e6, B, "read-unit forward + backward products on tcgen05 (bf16 operands, fp32 "
                      "accumulate, fp32 master weights)" if tc else "fp32 path"),
           "replicas_in_sync": sync}
    del tr
    torch.cuda.empty_cache()
    return out


def train_tc_arm(timeout_s=90):
    """Mixed-precision training of the cell (bf16 tensor-core forward AND backward GEMMs; DESIGN.md section 9) measured in a
    CHILD process: the composition was written after the round's GPU budget was spent, so a failure of it must not be able
    to touch this process's CUDA context or its JSON line."""
    cmd = [sys.executable, os.path.abspath(__file__), "--mode", "train", "--train-prec", "bf16", "--bwd-tc", "1",
           "--steps", "4", "--warmup", "3"]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s, cwd=ROOT)
        if out.returncode != 0:
            return {"error": "exit %d: %s" % (out.returncode, out.stderr.strip()[-300:])}
        line = json.loads(out.stdout.strip().splitlines()[-1])
        return {"value": line["value"], "unit": line["unit"], "ms_per_step": line["ms_per_step"], "steps": line["steps"],
                "gpu_launches": line["gpu_launches"], "replicas_in_sync": line["config"]["replicas_in_sync_after_run"],
                "what": "bench.py --mode train --train-prec bf16 --bwd-tc 1 in a child process: DP training step of the cell with "
                        "the read unit's forward and backward products on tcgen05 tensor cores (linear-probe loss)"}
    except Exception as exc:
        return {"error": repr(exc)[:300]}


def train_full_arm(steps, warmup, rank, world, dist):
    """DP-training step of the WHOLE reference model (SURVEY section 8(f) rows 1-3 around the cell): embeddings + bi-LSTM
    question encoder -> 2 x conv3x3 stem on [B,14,14,1024] features -> 12 MAC steps -> output unit -> classifier -> loss,
    hand-written backward of each, ONE all-reduce of the flat bucket, fused clip/Adam/EMA.  fp32 path."""
    from mac_network_b200.dp import DPTrainer
    shape = SHAPES[WORKLOAD]
    B, S, N, d, L = shape
    V, E, A, C = 90, 300, 28, 1024                     # CLEVR: ~90 question words, 300-d embeddings, 28 answers, ResNet-101 conv4
    cfg = MACConfig.args("args", netLength=L)
    tr = DPTrainer(cfg, L, seed=7, rank=rank, world=world, classifier=(A, [512]), encoder=(V, E), stem=(C, 2))
    rng = np.random.RandomState(31 + rank)
    lengths = rng.randint(S // 2, S + 1, size=(B,)).astype(np.int32)
    lengths[0] = S
    q = rng.randint(1, V + 1, size=(B, S)).astype(np.int32)
    q[np.arange(S)[None, :] >= lengths[:, None]] = 0
    data = {"questions": torch.from_numpy(q).cuda(), "questionLengths": torch.from_numpy(lengths).cuda(),
            "images": torch.relu(torch.randn(B, 14, 14, C, device="cuda")),
            "answers": torch.from_numpy(rng.randint(0, A, size=(B,)).astype(np.int32)).cuda()}
    from mac_network_b200 import _lib
    for _ in range(warmup):
        tr.train_step_full(0, data, B * world)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    n0 = _lib.load().mac_b200_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        _, losses = tr.train_step_full(0, data, B * world)
    e1.record()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) * 1e-3
    launches = _lib.load().mac_b200_launch_count() - n0
    if dist is not None:
        tt = torch.tensor([t], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t = float(tt[0])
    out = {"value": steps * L * world / t, "unit": UNIT, "ms_per_step": t / steps * 1e3, "steps": steps,
           "loss_last": float(losses.mean().item()), "gpu_launches": int(launches),
           "what": "whole-model DP training step: embedding + bi-LSTM encoder (S=%d, 2x256) + stem (2 x conv3x3, 1024->512->512 on "
                   "14x14) + %d MAC steps + output unit/classifier/softmax-CE, hand-written backward, all-reduce of %.1f MB, fused "
                   "clip/Adam/EMA; B=%d per GPU, fp32 path, reference training dropouts" % (S, L, tr.params.numel * 4 / 1e6, B)}
    del tr
    torch.cuda.empty_cache()
    return out


def run_train(args):
    """Data-parallel TRAINING step of the cell (BASELINE.json configs[3]): forward with train-mode dropouts + hand-written
    backward + NCCL all-reduce of the flat gradient bucket + fused clip/Adam/EMA, B=64 per GPU (weak scaling), fp32 path."""
    from mac_network_b200 import _lib
    from mac_network_b200.dp import DPTrainer
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = local_device()
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = _lib.load()
    shape = SHAPES[WORKLOAD]
    B, S, N, d, L = shape
    cfg = MACConfig.args("args", netLength=L)
    pv = perturb_biases(init_params(cfg, L, seed=100), seed=101)
    tr = DPTrainer(cfg, L, param_values=pv, seed=7, rank=rank, world=world, prec=args.train_prec, bwd_tc=bool(args.bwd_tc))
    nslots = 4
    batches, probes = [], []
    for s_ in range(nslots):
        inp = make_inputs(B, S, N, d, seed=1234 + 1000 * rank + s_)
        batches.append({k: torch.from_numpy(v).cuda() for k, v in inp.items()})
        g = torch.Generator(device="cuda").manual_seed(99 + 17 * rank + s_)
        probes.append((torch.randn(B, d, device="cuda", generator=g), torch.randn(B, d, device="cuda", generator=g)))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def one(k):
        sl = k % nslots
        tr.train_step(sl, batches[sl], probes[sl][0], probes[sl][1], B * world)

    for w in range(args.warmup):
        one(w)
    barrier()
    n0 = lib.mac_b200_launch_count()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(args.steps):
        one(k)
    e1.record()
    barrier()
    t_dev = e0.elapsed_time(e1) * 1e-3
    launches = lib.mac_b200_launch_count() - n0
    clocks = sampler.stop() if rank == 0 else None
    in_sync = True
    if dist is not None:
        tt = torch.tensor([t_dev], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_dev = float(tt[0])
        # replicas must stay bit-identical: every rank applied the same all-reduced gradient
        chk = torch.stack([tr.params.flat.double().sum(), tr.params.flat.double().abs().sum()])
        allc = [torch.zeros_like(chk) for _ in range(world)]
        dist.all_gather(allc, chk)
        in_sync = all(bool(torch.equal(allc[0], c)) for c in allc)
    if rank == 0:
        value = args.steps * L * world / t_dev
        nparam = tr.params.numel
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32" if (args.train_prec == "fp32" and not args.bwd_tc) else "bf16", "data": "synthetic",
                "config": {"workload": "BASELINE.json configs[3]: DP training of the args.txt cell, B=%d per GPU (global %d), "
                                       "S=%d, N=%d, d=%d, netLength=%d; dropouts memory/read/write = %s"
                                       % (B, B * world, S, N, d, L, str(tr.dropouts)),
                           "step": "forward + hand-written backward + all-reduce(%d fp32 = %.1f MB) + clip/Adam/EMA; "
                                   "%d reasoning steps" % (nparam, nparam * 4 / 1e6, L),
                           "l2": "timed steps rotate over %d resident batches per rank; activations saved for backward "
                                 "(%.0f MB per step) exceed L2" % (nslots, L * 3 * B * N * d * 4 / 1e6),
                           "cuda_graph": False, "projections": "forward %s, backward %s" % (
                               args.train_prec, "bf16 tensor cores" if args.bwd_tc else "fp32"), "parallelism": "dp%d, NCCL all-reduce per step" % world,
                           "replicas_in_sync_after_run": in_sync},
                "sample_steps_per_sec": value * B, "gpu_launches": int(launches), "clocks": clocks,
                "e2e": None, "roofline": None, "cpu_baseline": None}
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def run_quick(args):
    """Resident-input throughput only (no e2e / rooflines / CPU / training arms): used in child processes for informational
    side measurements, e.g. `--batch-mult 6 --streams 1` = six B=64 requests concatenated into one B=384 pass."""
    from mac_network_b200.mac_cell import MACParams
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    B, S, N, d, L = SHAPES[args.workload]
    mult = max(1, args.batch_mult)
    shape = (B * mult, S, N, d, L)
    cfg = MACConfig.args("gqa" if args.workload == "gqa" else "args", netLength=L)
    params = MACParams(cfg, L, values=perturb_biases(init_params(cfg, L, seed=100), seed=101))
    nstreams = max(1, args.streams)
    fold_y = (nstreams < 4) if args.fold_y < 0 else bool(args.fold_y)
    nslots = max(2, min(NSLOTS, 2 * nstreams)) if mult > 1 else max(NSLOTS, nstreams)   # keep > 126 MB of inputs in rotation
    slots = [Slot(cfg, params, shape, 1234 + s, args.prec, not args.no_graph, fold_y=fold_y, small_tc=(nstreams >= 2))
             for s in range(nslots)]
    side = [torch.cuda.Stream() for _ in range(nstreams - 1)]
    main_stream = torch.cuda.current_stream()

    def run(n):
        fork = torch.cuda.Event()
        fork.record(main_stream)
        for st in side:
            st.wait_event(fork)
        for k in range(n):
            j = k % nstreams
            if j == 0:
                slots[k % nslots].run()
            else:
                with torch.cuda.stream(side[j - 1]):
                    slots[k % nslots].run()
        for st in side:
            ev = torch.cuda.Event()
            ev.record(st)
            main_stream.wait_event(ev)
    run(max(args.warmup, nstreams))
    t, _ = timed_blocks(run, args.steps, torch.cuda.synchronize, None, min_total_s=args.min_time)
    print(json.dumps({"metric": METRIC, "value": args.steps * L * mult / t, "unit": UNIT, "workload": args.workload,
                      "shape_B_S_N_d_L": list(shape), "prec": args.prec, "batch_rows_per_pass": B * mult,
                      "requests_of_64_per_pass": mult, "concurrent_passes": nstreams, "ms_per_pass": t / args.steps * 1e3,
                      "launches_per_pass": int(slots[0].launches), "resident_slots": nslots}))


def child_measure(extra, timeout_s=60):
    """Run `bench.py <extra>` in a child process and return its last JSON line (or an error record).  The side
    measurements take few passes, so their block is repeated until 0.5 s is timed."""
    try:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--min-time", "0.5"] + extra, capture_output=True,
                             text=True, timeout=timeout_s, cwd=ROOT)
        if out.returncode != 0:
            return {"error": "exit %d: %s" % (out.returncode, out.stderr.strip()[-300:])}
        return json.loads(out.stdout.strip().splitlines()[-1])
    except Exception as exc:
        return {"error": repr(exc)[:300]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    shape = SHAPES[WORKLOAD]
    B, S, N, d, L = shape
    cfg = MACConfig.args("args", netLength=L)
    pv = perturb_biases(init_params(cfg, L, seed=100), seed=101)
    from oracle.mac_torch_cpu import TorchCPUCell
    host_threads()
    inp = make_inputs(B, S, N, d, seed=1234)
    cell = TorchCPUCell(cfg, pv, L)
    a = (torch.from_numpy(inp["vecQuestions"]), torch.from_numpy(inp["questionCntxWords"]),
         torch.from_numpy(inp["questionLengths"]).long(), torch.from_numpy(inp["knowledgeBase"]))
    # the SAME --steps / --warmup as the driver passes to our arm (a CPU pass is ~0.3-0.4 s; bounded at 60 / 5 so the run
    # ends within a few minutes whatever the flags)
    steps = max(1, min(args.steps, 60))
    warm = max(1, min(args.warmup, 5))
    for _ in range(warm):
        cell.forward(*a)
    t0 = time.perf_counter()
    for _ in range(steps):
        cell.forward(*a)
    dt = time.perf_counter() - t0
    v = steps * L / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
            "steps": steps, "warmup": warm, "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(shape),
                       "note": "TensorFlow-1 is not installable offline: this is the oracle's fp32 PyTorch-CPU port at "
                               "TF-op granularity on all host threads (rank 0 only)"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                             "sample": "%d full forward passes (B=%d, netLength=%d), %.3f s each" % (steps, B, L, dt / steps)},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--prec", default="bf16", choices=["fp32", "bf16", "tc32"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-train", action="store_true", help="skip the short DP-training arm of the default run")
    ap.add_argument("--mode", default="infer", choices=["infer", "train", "quick"])
    ap.add_argument("--batch-mult", type=int, default=1, help="--mode quick: requests of B=64 concatenated per pass")
    ap.add_argument("--streams", type=int, default=12, help="independent passes in flight (each on its own stream); "
                    "measured on the B200 (packed read step): 1: 19.9k, 4: 32.4k, 8: 34.4k, 12: 35.1k, 16: 35.1k reasoning-steps/s")
    ap.add_argument("--fold-y", type=int, default=-1, help="write unit folded with the next step's projY: 1/0, -1 = by --streams")
    ap.add_argument("--rooflines-only", action="store_true", help="only the per-kernel measurements (for ncu)")
    ap.add_argument("--min-time", type=float, default=0.0, help="repeat the --steps block until this many seconds are timed "
                    "(default: one block, so exactly --steps passes are timed)")
    ap.add_argument("--workload", default="headline", choices=["headline", "gqa", "cpu_ref"], help="--mode quick: shape + flag file")
    ap.add_argument("--train-prec", default="fp32", choices=["fp32", "bf16"], help="--mode train: read-unit forward GEMMs")
    ap.add_argument("--bwd-tc", type=int, default=0, help="--mode train: read-unit backward GEMMs on tensor cores (1/0)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed pass of the resident-input arm returned "
                    "(rank 0) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.rooflines_only or args.impl != "ours" or args.mode != "infer"):
        ap.error("--dump-outputs applies to the default inference run only")
    args.warmup = max(args.warmup, 3)
    if args.rooflines_only:
        torch.cuda.set_device(0)
        print(json.dumps(kernel_rooflines(SHAPES[WORKLOAD], args.prec, peaks())))
    elif args.impl == "reference":
        run_reference(args)
    elif args.mode == "train":
        run_train(args)
    elif args.mode == "quick":
        run_quick(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
