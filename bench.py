"""bench.py -- Sycamore n53 m20 sliced-contraction throughput (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--dtype complex128] [--impl reference]
                    [--config m20|peps8x8|m10|m10s|m12] [--scaling weak|strong]
                    [--dump-outputs DIR]

Default workload (config.workload): the reference's own benchmark structure
``examples/benchmarks/sycamore_n53_m20_s0_e0_pABCDCDAB.json`` (381 tensors, 754
indices) with the SURVEY.md Appendix-B contraction tree: W = 2^30 elements per
slice, 36 sliced indices (2^36 slices), 4.449e11 scalar MACs per slice -- shipped
as ``tests/golden/sycamore_m20.json``.  Synthetic seeded operands.

A *step* contracts ``--slices-per-gpu`` slices on every GPU (slice ids taken
round-robin over ranks exactly like ``ContractionTree.contract_mpi``,
cotengra/core.py:4070), accumulates them on the device, and (N > 1) sums the
partial outputs with one NCCL all-reduce.  Throughput = 8 * C_slice real flops per
slice of the REFERENCE's tree (complex multiply-add = 8 flops, docs convention;
BASELINE.md section 1; the executor's stem fusion changes what is executed, not what is
counted) times slices, divided by device time (CUDA events, max over ranks).  The
whole job has 2^36 slices, so -- exactly as ``tree.benchmark()`` (core.py:4143-4158)
-- the number is measured on a slice sample and the total is an extrapolation
(``config.est_total_hours``).

The same JSON line also carries, at N = 1: the complex64 run of the same workload
(``secondary``; BASELINE config 5 "complex64 vs complex128"), the GPU-library baseline
SURVEY 2.3 asks for -- the reference's own dispatch for torch inputs, ``torch.tensordot``
+ ``permute`` on the same B200 (``gpu_library_baseline``) --, a parity check of one slice
against the CPU oracle's golden value at this very width (``parity``) and the CPU baseline.

The reference arm (``--impl reference``) times the CPU restatement of the
reference's numpy path (``oracle/``) on the host cores, on slices of the same
network sliced further until a step fits host memory/time.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRICS = {
    "m20": "sycamore_n53_m20_sliced_contract_tflops",
    "peps8x8": "peps8x8_bond6_contract_tflops",
    "m10": "sycamore_n53_m10_amplitude_tflops",
    "m10s": "sycamore_n53_m10_rank_simplified_amplitude_tflops",
    "m12": "sycamore_n53_m12_256slices_tflops",
}
UNIT = "TFLOP/s"
SEED, SCALE = 0, 0.65
DUMP_BYTES = 60 * 10**6  # --dump-outputs: arrays plus .npy headers stay under 64 MB


# ---------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------


def load_spec():
    import cotengra_b200 as cb
    from tests.helpers import decode_sliced, load_json

    rec = next(r for r in load_json("sycamore_m20.json") if r["name"] == "sycamore_m20_appxB")
    spec = cb.TreeSpec(rec["inputs"], rec["output"], rec["size_dict"], rec["path"],
                       decode_sliced(rec["sliced"]))
    return spec, rec


def load_workload(config, dtype):
    """(spec, arrays, description) of a BASELINE.json configuration."""
    import cotengra_b200 as cb
    from tests.helpers import GOLDEN_DIR, load_json, load_npz, make_arrays

    if config == "m20":
        spec, _rec = load_spec()
        arrays = make_arrays(spec.shapes(), dtype, seed=SEED, scale=SCALE)
        return spec, arrays, ("sycamore_n53_m20 amplitude (examples/benchmarks/sycamore_n53_m20_s0_e0_pABCDCDAB.json), "
                              "SURVEY Appendix-B tree: W=2^30, 36 sliced indices (2^36 slices)")
    if config == "peps8x8":
        rec = next(r for r in load_json("trees.json") if r["name"] == "peps8x8_d2")
        size_dict = {ix: 6 for ix in rec["size_dict"]}
        spec = cb.TreeSpec(rec["inputs"], rec["output"], size_dict, rec["path"])
        arrays = make_arrays(spec.shapes(), dtype, seed=11, scale=0.35)
        return spec, arrays, "8x8 PEPS amplitude, bond 6 (lattice_equation([8,8], d_min=6)), greedy tree, unsliced"
    with open(os.path.join(GOLDEN_DIR, "circuits.json")) as f:
        rec = json.load(f)[config]
    flat = load_npz("circuits_arrays.npz")[f"{config}_arrays_flat"]
    spec = cb.TreeSpec.from_dict(rec["spec"])
    arrays, off = [], 0
    for shape in spec.shapes():
        n = int(np.prod(shape))
        arrays.append(np.ascontiguousarray(flat[off:off + n].reshape(shape)).astype(dtype))
        off += n
    desc = (f"Sycamore circuit_n53_{config} amplitude from the reference's .qsim file (real gate tensors), "
            f"{spec.N} tensors, {spec.nslices} slice(s)")
    return spec, arrays, desc


def golden_big_slice():
    """Slice 0 of the m20 Appendix-B tree at W = 2^30 from the CPU oracle (tests/golden/big_slices.json,
    scripts/gen_big_goldens.py); None if the fixture is absent."""
    gpath = os.path.join(ROOT, "tests", "golden", "big_slices.json")
    if not os.path.exists(gpath):
        return None
    with open(gpath) as f:
        g = json.load(f).get("appxB_w30_slice0")
    return None if g is None else complex(g["re"], g["im"])


def measured_bf16():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        if "bf16_tflops" in d:
            return float(d["bf16_tflops"]), "MEASURED_PEAKS.json dense bf16 (cuBLAS, burst)"
    return 2250.0, "nominal 2.25 PFLOP/s dense bf16 (MEASURED_PEAKS.json absent)"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "MEASURED_PEAKS.json (driver-measured copy bandwidth)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md; MEASURED_PEAKS.json absent)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(
                    ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                     "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.samples.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        self.stop_flag = True
        sm = sorted(float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples if len(s) >= 7
                          for n, v in zip(names, s[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]),
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle on the host cores
# ---------------------------------------------------------------------------


def _blas_threads(n):
    """Pin the BLAS pool explicitly (torchrun exports OMP_NUM_THREADS=1) and report what the
    pools really have."""
    try:
        import threadpoolctl

        ctl = threadpoolctl.threadpool_limits(limits=n)
        got = sorted({int(p["num_threads"]) for p in threadpoolctl.threadpool_info()})
        return ctl, got
    except Exception:
        return None, None


class CpuSample:
    """One slice of the m20 network sliced further to W = 2^width_log2, through the oracle
    (port of the reference's numpy path)."""

    def __init__(self, dtype, width_log2):
        from oracle import ctg_oracle as orc
        from tests.helpers import make_arrays
        from tests.slicing_util import slice_to_width

        spec, _ = load_spec()
        self.orc = orc
        self.small = slice_to_width(spec, 2 ** width_log2)
        self.ir = self.small.contractions()
        self.inputs = [tuple(t) for t in self.small.inputs]
        self.arrays = make_arrays(self.small.shapes(), dtype, seed=SEED, scale=SCALE)
        self.macs, _el = orc.contraction_cost(self.ir, self.small.sliced_shapes())
        self.width_log2 = width_log2

    def run(self, i):
        t0 = time.perf_counter()
        self.last = self.orc.run_contractions(self.ir, self.orc.slice_arrays(self.inputs, self.small.sliced,
                                                                              self.arrays, i))
        return time.perf_counter() - t0


def cpu_baseline(dtype, width_log2=24, reps=3):
    """Oracle on a bounded sample: warm-up slice (as tree.benchmark, core.py:4143-4144), then
    ``reps`` timed slices, median.  Returns (tflops, seconds_per_slice, info)."""
    cores = os.cpu_count()
    ctl, pools = _blas_threads(cores)
    s = CpuSample(dtype, width_log2)
    s.run(0)
    times = sorted(s.run(i + 1) for i in range(reps))
    dt = times[len(times) // 2]
    tflops = 8 * s.macs / dt / 1e12
    info = {
        "value": tflops, "unit": UNIT, "cores": cores, "kind": "port",
        "blas_threads": pools, "reps": reps, "seconds_per_slice": [round(t, 3) for t in times],
        "sample": (f"median of {reps} slices (after 1 warm-up) of the same m20 network sliced to "
                   f"W=2^{width_log2} ({s.macs:.3g} MACs/slice, {dt:.2f} s/slice), oracle/ctg_oracle.py "
                   f"(numpy {np.__version__}; BLAS pool set to {cores} threads with threadpoolctl, pools report "
                   f"{pools}; OMP_NUM_THREADS={os.environ.get('OMP_NUM_THREADS', 'unset')})"),
    }
    del ctl
    return tflops, dt, info


def run_reference(args):
    """The reference arm: exactly ``warmup`` untimed + ``steps`` timed steps, a step = one slice
    of the m20 network at a width chosen so that the whole run stays within ~2 minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count()
    ctl, pools = _blas_threads(cores)
    budget_s = 120.0
    probe = CpuSample(args.dtype, 20)
    probe.run(0)
    t20 = probe.run(1)
    width = 20
    for w in (22, 24):
        # per-slice cost grows about linearly with the width
        if (args.steps + args.warmup) * t20 * 2 ** (w - 20) * 1.3 <= budget_s:
            width = w
    s = probe if width == 20 else CpuSample(args.dtype, width)
    for i in range(args.warmup):
        s.run(i)
    times = [s.run(args.warmup + i) for i in range(args.steps)]
    total = sum(times)
    value = 8 * s.macs * len(times) / total / 1e12
    info = {
        "value": value, "unit": UNIT, "cores": cores, "kind": "port", "blas_threads": pools,
        "sample": (f"{args.steps} timed slices (+{args.warmup} warm-up) of the m20 Appendix-B network sliced "
                   f"further to W=2^{width} ({s.macs:.3g} MACs/slice), oracle/ctg_oracle.py "
                   f"(numpy {np.__version__}; BLAS pool {pools}; OMP_NUM_THREADS="
                   f"{os.environ.get('OMP_NUM_THREADS', 'unset')})"),
    }
    line = {
        "impl": "reference", "metric": METRICS["m20"], "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / max(1, len(times)),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype_tag(args.dtype),
        "data": "synthetic",
        "config": {"workload": "sycamore_n53_m20 amplitude, SURVEY Appendix-B tree (the GPU arm's network and "
                               f"operands); CPU step = one slice of it at W=2^{width} instead of 2^30 "
                               "(host memory/time bound)",
                   "same_slice_width_as_gpu_arm": False,
                   "note": "reference = the repo's CPU restatement (oracle/) of cotengra's numpy path, pinned to "
                           "the unmodified reference by golden vectors; cotengra itself is pure Python and needs "
                           "autoray, absent on the box"},
        "cpu_baseline": info,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    del ctl
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"out": s.last})
    print(json.dumps(line))


def dump_outputs(dirname, outputs):
    """``--dump-outputs``: each array of the timed path's last step as ``DIR/<name>.npy``, complex
    values as (real, imag) pairs on a trailing axis in the precision they were computed in.  An
    output larger than its share of ``DUMP_BYTES`` is replaced by a fixed seeded sample of its flattened
    elements (ascending positions), so that two builds can be compared value for value."""
    os.makedirs(dirname, exist_ok=True)
    budget = DUMP_BYTES // max(1, len(outputs))
    for name, a in outputs.items():
        a = np.asarray(a)
        real = np.dtype(np.float64 if a.dtype in (np.complex128, np.float64) else np.float32)
        per = real.itemsize * (2 if a.dtype.kind == "c" else 1)
        if a.size * per > budget:
            keep = np.random.default_rng(SEED).choice(a.size, budget // per, replace=False)
            a = a.reshape(-1)[np.sort(keep)]
        if a.dtype.kind == "c":
            a = np.stack([a.real, a.imag], axis=-1)
        np.save(os.path.join(dirname, f"{name}.npy"), a.astype(real))


def dtype_tag(dtype):
    return {"complex128": "c128 (f64 arithmetic)", "complex64": "c64 (f32 arithmetic)"}.get(dtype, dtype)


# ---------------------------------------------------------------------------
# GPU-library baseline: what the reference itself does with torch inputs
# ---------------------------------------------------------------------------


def torch_run_contractions(ir, tensors):
    """The reference's node loop (contract.py:791-832) with the array ops it dispatches to for
    torch inputs (contract.py:752-773): ``torch.tensordot`` (+ ``permute``) / ``torch.einsum``.
    None of this repo's kernels are involved."""
    import torch

    live = dict(enumerate(tensors))
    out = None
    for p, l, r, tdot, arg, perm in ir:
        if r is None:
            if l is None:
                live[p] = torch.einsum(arg, live[p])
                continue
            return torch.einsum(arg, live[l])
        x, y = live.pop(l), live.pop(r)
        if tdot:
            out = torch.tensordot(x, y, dims=(list(arg[0]), list(arg[1])))
            if perm:
                out = out.permute(perm)
        else:
            out = torch.einsum(arg, x, y)
        del x, y
        live[p] = out
    return out


def torch_slice_arrays(spec, tensors, i):
    key = spec.slice_key(i)
    out = list(tensors)
    for c, term in enumerate(spec.inputs):
        if any(ix in key for ix in term):
            out[c] = tensors[c][tuple(key.get(ix, slice(None)) for ix in term)]
    return out


def gpu_library_baseline(spec, tensors, flops_slice, reps=2, first_slice=0):
    import torch

    try:
        ir = spec.contractions()
        bad = [a for _p, _l, r, tdot, a, _q in ir if not tdot and any(ord(ch) > 122 for ch in a if ch not in ",->")]
        if bad:
            return {"unavailable": "torch.einsum only takes [a-zA-Z] index symbols; this tree has einsum nodes beyond them"}
        torch.cuda.synchronize()
        val = torch_run_contractions(ir, torch_slice_arrays(spec, tensors, first_slice))  # warm-up
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(reps):
            torch_run_contractions(ir, torch_slice_arrays(spec, tensors, first_slice + 1 + k))
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        peak = torch.cuda.max_memory_allocated() / 2**30
        return {
            "value": flops_slice / (ms * 1e-3) / 1e12, "unit": UNIT, "ms_per_slice": ms, "reps": reps,
            "impl": ("the reference's own dispatch for torch inputs (cotengra/contract.py:752-773): torch.tensordot + "
                     "permute per node on the same B200 (cuBLAS GEMM behind permute/reshape copies); no kernel of "
                     f"this repo involved (torch {torch.__version__})"),
            "peak_gib": peak,
            "_slice_value": complex(val.reshape(-1)[0].item()) if val.numel() == 1 else None,
        }
    except Exception as exc:  # out of memory, > 64 dims, ...
        return {"unavailable": f"{type(exc).__name__}: {str(exc)[:200]}"}
    finally:
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------
# the GPU arm
# ---------------------------------------------------------------------------


def timed_run(ex, tensors, args, world, rank, dev, S, slice_ids=None):
    """warmup + exactly ``steps`` timed steps on the device; returns a dict of measurements."""
    import torch
    import torch.distributed as dist

    from cotengra_b200 import _lib

    plan = ex.plan
    tdt = getattr(torch, ex.dtype)
    out = torch.zeros(plan.out_shape, dtype=tdt, device=dev)
    nsl = ex.nslices

    def step(i):
        # slices base, base+1, ... shared round-robin between the ranks (core.py:4070)
        base = (i * S * world) % max(1, nsl - S * world + 1) if nsl > S * world else 0
        out.zero_()
        ex.contract_device(tensors, begin=base + rank, step=world, count=S, out=out)
        if world > 1:
            dist.all_reduce(torch.view_as_real(out) if out.is_complex() else out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    sampler = ClockSampler(dev.index)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        step(args.warmup + i)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = _lib.launch_count() - launches0
    clocks = sampler.summary() if rank == 0 else None
    # per-node CUDA events (two records per node) cost ~2 % when they sit inside the timed region:
    # one more step, outside it, feeds the roofline of the dominant kernel
    plan.profile(True)
    ex.contract_device(tensors, begin=rank, step=world, count=1, out=torch.zeros_like(out))
    torch.cuda.synchronize()
    node_ms = plan.profile_read()
    plan.profile(False)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        lt = torch.tensor([launches], device=dev, dtype=torch.int64)
        dist.all_reduce(lt)
        launches = int(lt.item())
    return {"ms": ms, "launches": launches, "node_ms": node_ms, "clocks": clocks, "out": out, "barrier": barrier}


def roofline_of(plan, node_ms, dtype, peaks):
    """Binding roofline of the dominant node of the last timed slice."""
    hbm_peak, hbm_src = measured_peaks()
    pair_nodes = [(nd, t) for nd, t in zip(plan.nodes, node_ms) if nd["kind"] == 0 and t > 0]
    nd, t_ms = max(pair_nodes, key=lambda x: x[1])
    Bn, M, N, K = nd["sizes"]
    el = sum(int(np.prod(x.shape)) for x in (nd["a"], nd["b"], nd["c"]))
    node_flops = 8.0 * Bn * M * N * K
    node_bytes = el * plan.esize
    traffic, traffic_src = None, None
    for name in ("r02_top_kernel.json", "r01_top_kernel.json"):
        tp = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tp):
            with open(tp) as f:
                rec = json.load(f).get(dtype, {})
            # (only for the node the capture was taken on: other configurations have no capture)
            if rec.get("dram_bytes_per_launch") and abs(rec.get("algorithmic_bytes", 0) - node_bytes) <= 1e-3 * node_bytes:
                traffic = rec["dram_bytes_per_launch"]
                traffic_src = (f"static: dram__bytes_read.sum + dram__bytes_write.sum of this node from the "
                               f"ncu --set full capture recorded in profiles/{name} (not measured in this run)")
                break
    fp64 = dtype in ("complex128", "float64")
    achieved_tf = node_flops / (t_ms * 1e-3) / 1e12
    achieved_gbs = node_bytes / (t_ms * 1e-3) / 1e9
    if fp64:
        tensor_peak = peaks["dmma_tflops"]
        tensor_src = ("fp64 DMMA microbenchmark run in this process (ctgb_probe_fp64_peaks); "
                      "MEASURED_PEAKS.json holds no fp64 figure")
    else:
        # complex64 runs as three kind::tf32 passes over the real embedding (8C real flops each):
        # effective peak = dense TF32 peak / 3, dense TF32 = half the measured dense bf16 figure
        bf16, bf16_src = measured_bf16()
        tensor_peak = bf16 / 2.0 / 3.0
        tensor_src = f"{bf16_src} / 2 (tf32) / 3 (3xTF32 passes)"
    frac_tensor, frac_hbm = achieved_tf / tensor_peak, achieved_gbs / hbm_peak
    tensor_bound = frac_tensor >= frac_hbm
    roofline = {
        # the binding roofline of the dominant node: whichever of the two it sits closer to
        "bound": "tensor" if tensor_bound else "hbm",
        "kernel": f"node M={M} N={N} K={K} (variant {int(nd['plan'].variant)})",
        "achieved": achieved_tf if tensor_bound else achieved_gbs,
        "peak": tensor_peak if tensor_bound else hbm_peak,
        "unit": "TFLOP/s" if tensor_bound else "GB/s",
        "peak_source": tensor_src if tensor_bound else hbm_src,
        "frac_tensor": frac_tensor, "frac_hbm": frac_hbm,
        "launch_ms": t_ms,
        "share_of_slice": t_ms / sum(t for _n, t in pair_nodes),
        "algorithmic_bytes": node_bytes,
        "algorithmic_flops": node_flops,
        "traffic": traffic, "traffic_source": traffic_src,
    }
    roofline["frac"] = roofline["achieved"] / roofline["peak"]
    # per-node roofline sum of the executed plan: how close the kernels are to what per-node
    # kernels can reach on this tree (each node at max(flops/peak, bytes/bw))
    floor_ms = sum(max(8.0 * np.prod(n_["sizes"], dtype=float) / (tensor_peak * 1e12),
                       sum(int(np.prod(x.shape)) for x in (n_["a"], n_["b"], n_["c"])) * plan.esize / (hbm_peak * 1e9))
                   for n_, _t in pair_nodes) * 1e3
    return roofline, floor_ms, sum(t for _n, t in pair_nodes)


def run_gpu(args):
    import torch
    import torch.distributed as dist

    import cotengra_b200 as cb
    from cotengra_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    spec, arrays, workload = load_workload(args.config, args.dtype)
    ex = cb.TreeExecutor(spec, dtype=args.dtype, device=local, fuse=not args.no_fuse)
    plan = ex.plan
    strong = args.scaling == "strong"
    if strong:
        # the whole (finite) job shared by the ranks: a step = every slice once
        if spec.nslices % world:
            raise SystemExit(f"--scaling strong needs the {spec.nslices} slices to divide over {world} ranks")
        S = spec.nslices // world
    else:
        S = min(args.slices_per_gpu, max(1, spec.nslices // world))
    tensors = [torch.from_numpy(a).to(dev) for a in arrays]
    tdt = getattr(torch, args.dtype)
    ex.workspace(host_staging=True)  # allocate once, outside the timed region

    r = timed_run(ex, tensors, args, world, rank, dev, S)
    ms, launches, node_ms, clocks, out, barrier = (r[k] for k in ("ms", "launches", "node_ms", "clocks", "out", "barrier"))
    dumped = {"out": out.cpu().numpy()}
    macs_ref, _macs_inv, elems_ref = ex.reference_work
    flops_slice = 8 * macs_ref
    total_slices = S * world * args.steps
    value = flops_slice * total_slices / (ms * 1e-3) / 1e12
    finite = bool(torch.isfinite(torch.view_as_real(out) if out.is_complex() else out).all().item())

    # ---- end to end through the C-ABI host call (rank-local, then max over ranks):
    # pinned host inputs -> H2D -> slices -> D2H of the result, every step
    pinned = []
    for a in arrays:
        t = torch.empty(a.shape, dtype=tdt).pin_memory()
        t.copy_(torch.from_numpy(a))
        pinned.append(t.numpy())
    h2d = int(sum(a.nbytes for a in pinned))
    d2h = int(plan.out_elements * plan.esize)
    ex.contract_host(pinned, begin=rank, step=world, count=1)  # warm
    barrier()
    t0 = time.perf_counter()
    e2e_steps = args.steps if not strong else 1
    for i in range(e2e_steps):
        base = 0 if strong or spec.nslices <= S * world else (args.warmup + args.steps + i) * S * world
        res = ex.contract_host(pinned, begin=base + rank, step=world, count=S)
        if world > 1:
            rr = torch.from_numpy(np.asarray(res)).to(dev)
            dist.all_reduce(torch.view_as_real(rr) if rr.is_complex() else rr)
            res = rr.cpu()
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = flops_slice * S * world * e2e_steps / e2e_s / 1e12

    # ---- complex64 on the same workload, same protocol (BASELINE config 5: "complex64 vs complex128")
    secondary = None
    if args.config == "m20" and args.dtype == "complex128" and not args.no_secondary:
        peaks64 = None
        ex64 = cb.TreeExecutor(spec, dtype="complex64", device=local, fuse=not args.no_fuse)
        t64 = [t.to(torch.complex64) for t in tensors]
        r64 = timed_run(ex64, t64, args, world, rank, dev, S)
        dumped["out_complex64"] = r64["out"].cpu().numpy()
        m64, _i64, _e64 = ex64.reference_work
        v64 = 8 * m64 * total_slices / (r64["ms"] * 1e-3) / 1e12
        if rank == 0:
            peaks64 = _lib.probe_fp64_peaks()
            roof64, floor64, sum64 = roofline_of(ex64.plan, r64["node_ms"], "complex64", peaks64)
            par64 = {"checked": False}
            g64 = golden_big_slice()
            if g64 is not None:
                chk = torch.zeros(ex64.plan.out_shape, dtype=torch.complex64, device=dev)
                ex64.contract_device(t64, begin=0, step=1, count=1, out=chk)
                got64 = complex(chk.reshape(-1)[0].item())
                # one slice amplitude is a cancelling sum over 2^30-element tensors: fp32 arithmetic
                # cannot hold north_star's 1e-5 on it whatever the kernel (numpy's complex64 runs of the
                # small configs sit at 3e-6..3e-5, tests/test_gpu_round2.py bounds the kernels by those);
                # the complex128 leg of this line is the 1e-10 check
                par64 = {"checked": True, "slice_id": 0, "gpu_value": [got64.real, got64.imag],
                         "rel_err": abs(got64 - g64) / abs(g64), "tolerance": 5e-5,
                         "tolerance_note": "fp32 arithmetic on a cancelling 2^30-term sum; complex128 leg holds 1e-10"}
                par64["ok"] = par64["rel_err"] <= par64["tolerance"]
            secondary = {
                "dtype": dtype_tag("complex64"), "value": v64, "unit": UNIT,
                "ms_per_step": r64["ms"] / args.steps, "slice_ms": r64["ms"] / (S * args.steps),
                "gpu_launches": r64["launches"], "clocks": r64["clocks"], "roofline": roof64,
                "per_node_roofline_floor_ms": floor64, "node_ms_sum": sum64,
                "result_finite": bool(torch.isfinite(torch.view_as_real(r64["out"])).all().item()),
                "speedup_vs_complex128": v64 / value, "parity": par64,
            }
        del ex64, t64, r64
        torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = _lib.probe_fp64_peaks()
    roofline, floor_ms, node_sum_ms = roofline_of(plan, node_ms, args.dtype, peaks)
    hbm_peak, hbm_src = measured_peaks()
    fp64 = args.dtype in ("complex128", "float64")
    slice_ms = ms / (S * args.steps)
    tf = flops_slice / (slice_ms * 1e-3) / 1e12
    whole = {
        "slice_ms": slice_ms,
        "tflops": tf,
        "frac_of_fp64_tensor_peak": tf / peaks["dmma_tflops"] if fp64 else None,
        "hbm_achieved_gbs": plan.elements_per_slice * plan.esize / (slice_ms * 1e-3) / 1e9,
        "hbm_peak_gbs": hbm_peak, "hbm_peak_source": hbm_src,
        "hbm_frac": plan.elements_per_slice * plan.esize / (slice_ms * 1e-3) / 1e9 / hbm_peak,
        "fp64_peaks_measured": peaks,
        "per_node_roofline_floor_ms": floor_ms, "node_ms_sum": node_sum_ms,
        "stem_fusion": {
            "enabled": not args.no_fuse, "changed": bool(ex.fusion.get("changed")),
            "bytes_executed_over_reference_tree": plan.elements_per_slice / max(1, elems_ref),
            "macs_executed_over_reference_tree": plan.macs_per_slice / max(1, macs_ref),
            "root_peel": ex.fusion.get("root_peel"), "nodes_removed": ex.fusion.get("nodes_removed"),
        },
    }

    # ---- parity at the benchmarked width: one slice against the CPU oracle's golden value
    parity = {"checked": False}
    gpu_lib = None
    if args.config == "m20":
        check = torch.zeros(plan.out_shape, dtype=tdt, device=dev)
        ex.contract_device(tensors, begin=0, step=1, count=1, out=check)
        got = complex(check.reshape(-1)[0].item())
        parity = {"checked": False, "slice_id": 0, "gpu_value": [got.real, got.imag]}
        want = golden_big_slice()
        if want is not None:
            parity.update(checked=True, oracle_value=[want.real, want.imag],
                          rel_err=abs(got - want) / abs(want),
                          tolerance=1e-10 if fp64 else 5e-5,  # (fp32 on a cancelling 2^30-term sum, see the c64 leg)
                          source="tests/golden/big_slices.json (oracle/ctg_oracle.py on host cores, scripts/gen_big_goldens.py)")
            parity["ok"] = parity["rel_err"] <= parity["tolerance"]
        if world == 1 and not args.no_gpu_lib:
            ex._ws = None
            torch.cuda.empty_cache()
            gpu_lib = gpu_library_baseline(spec, tensors, flops_slice)
            tv = gpu_lib.pop("_slice_value", None)
            if tv is not None:
                parity["vs_torch_rel_err"] = abs(got - tv) / abs(tv)
            if "value" in gpu_lib:
                gpu_lib["b200_speedup"] = value / gpu_lib["value"]

    cpu = None
    if world == 1 and not args.no_cpu and args.config == "m20":
        _v, _dt, cpu = cpu_baseline(args.dtype)

    nslices = spec.nslices
    line = {
        "metric": METRICS[args.config], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": dtype_tag(args.dtype), "data": "synthetic",
        "config": {
            "workload": f"{workload}; {macs_ref:.4g} MACs/slice"
                        + ("; sample of the slice stream" if not strong and nslices > S * world else ""),
            "slices_per_step": S * world, "slices_per_gpu_per_step": S,
            "parallelism": f"slices round-robin over {world} GPU(s), one NCCL all-reduce per step",
            "l2": "inputs larger than L2 (per-slice intermediates of 2-16 GiB stream through HBM)",
            "flop_convention": "8*C real flops per complex MAC of the reference's tree (4*C figure = value/2)",
            "est_total_hours": slice_ms * 1e-3 * nslices / world / 3600.0,
            "hoisted_invariant_nodes": sum(1 for n_ in plan.nodes if n_["invariant"]),
            "workspace_gib": plan.total_bytes / 2**30,
        },
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps,
                "api": "TreeExecutor.contract_host -> ctgb_plan_execute_host (pinned host inputs)"},
        "gpu_launches": launches,
        "result_finite": finite,
        "clocks": clocks,
        "roofline": roofline,
        "whole_slice": whole,
        "parity": parity,
        "secondary": secondary,
        "gpu_library_baseline": gpu_lib,
        "cpu_baseline": cpu,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dumped)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dtype", default="complex128", choices=["complex128", "complex64"])
    ap.add_argument("--config", default="m20", choices=sorted(METRICS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="strong: a step contracts EVERY slice of the (finite) job once, shared by the ranks")
    ap.add_argument("--slices-per-gpu", type=int, default=2)
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--no-secondary", action="store_true", help="skip the complex64 leg")
    ap.add_argument("--no-gpu-lib", action="store_true", help="skip the torch.tensordot GPU-library baseline")
    ap.add_argument("--no-fuse", action="store_true", help="execute the reference's node sequence one to one")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32/float64)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
