#!/usr/bin/env python
"""bench.py -- headline benchmark of BASELINE.json: coded bits/s of LDPC5G BP decoding, n=8448 (k=4224), 20
iterations, batch 4096 per GPU (weak scaling over 1/2/4/8 B200; one process per GPU, NCCL all-reduce of the four
int64 error counters per step, as sim_ber's replicas do: /root/reference/src/sionna/phy/utils/misc.py:614-655).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload ldpc|qpsk_awgn|ofdm_siso|mimo_ofdm|pusch]
                  [--cn-update boxplus-phi|minsum|...] [--impl reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Default workload `ldpc` = configs[1] (the configuration BASELINE.json's metric is quoted on): a "step" = one
LDPC5GDecoder call on a [4096, 8448] fp32 logit tensor resident in HBM + error counting (+ the counter all-reduce for
N > 1). The other workloads are the receive chains of configs[0], [2], [3], [4] (tools/bench_links.py). Prints ONE JSON
line (rank 0). The default line also carries, inside keys the driver keeps, the boxplus-phi kernel at 0 dB (nothing
converges: no saturation shortcut applies), the min-sum rule, and a short measurement of every other workload
(`config.other_workloads`). See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K_INFO, N_CODE, BATCH, NUM_ITER = 4224, 8448, 4096, 20
EBNO_DB = 2.0
# SURVEY.md 8(d) / BASELINE.md: algorithmic bytes per codeword for flooding BP, one fp32 message per edge read +
# written once per iteration, one channel LLR read per VN per iteration, plus compulsory I/O.
E_EDGES, N_VNS = 40320, 8832
ALG_BYTES_PER_CW = NUM_ITER * (8 * E_EDGES + 4 * N_VNS) + 4 * N_CODE + 4 * K_INFO      # 7 208 448
DUMP_BYTES = 60 << 20        # --dump-outputs: array data of all files together (< 64 MB with the .npy headers)


def host_cores():
    """Threads this process may really use: CPU affinity capped by the cgroup CPU quota (os.cpu_count() reports the
    machine, not the container). Returns (usable, detail dict)."""
    try:
        aff = len(os.sched_getaffinity(0))
    except AttributeError:
        aff = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                 # cgroup v2: "<quota|max> <period>"
            q, p = f.read().split()[:2]
            if q != "max":
                quota = float(q) / float(p)
    except (OSError, ValueError):
        try:                                                      # cgroup v1
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                p = float(f.read())
            if q > 0:
                quota = q / p
        except (OSError, ValueError):
            pass
    usable = aff if quota is None else max(1, min(aff, int(math.ceil(quota))))
    return usable, {"os_cpu_count": os.cpu_count(), "sched_affinity": aff, "cgroup_cpu_quota": quota}


def committed_traffic(cn_update):
    """DRAM bytes per launch of the decode kernel from the committed `ncu --set full` capture (profiles/traffic.json)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        if cn_update in d:
            return d[cn_update]["traffic_bytes_per_launch"], d[cn_update].get("source", "profiles/traffic.json")
    return None, None


def live_traffic(cn_update, ebno_db, timeout=240):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the decode kernel, measured now by running this
    script's `--traffic-probe` leg under `ncu` (two metrics, one pass). Returns None if ncu cannot run here."""
    ncu = "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "-k",
           "regex:ldpc_bp", "-s", "2", "-c", "1", "--csv", sys.executable, os.path.abspath(__file__), "--traffic-probe",
           "--cn-update", cn_update, "--ebno-db", str(ebno_db)]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=dict(os.environ, RANK="0", WORLD_SIZE="1")).stdout
    except Exception:
        return None
    total, seen = 0.0, 0
    for ln in out.splitlines():
        f = [v.strip('"') for v in ln.split('","')]
        if len(f) > 3 and f[-3] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            try:
                v = float(f[-1].replace(",", ""))
            except ValueError:
                continue
            unit = f[-2].lower()
            v *= {"byte": 1.0, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(unit, 1.0)
            total += v
            seen += 1
    return total if seen == 2 else None


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons while the timed region runs: NVML (`pynvml`, ~20 ms period) when it is
    importable, else `nvidia-smi` polling (the recipe's clocks line, ~5 samples/s)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self._halt = index, [], threading.Event()   # samples: (sm_mhz, max_mhz, set(reasons))

    def _run_nvml(self):
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        masks = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self._halt.is_set():
            sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            self.samples.append((int(sm), int(mx), {n for n, m in masks.items() if bits & m}))
            self._halt.wait(0.02)
        nv.nvmlShutdown()

    def _run_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                f = [v.strip() for v in out.split(",")]
                if len(f) >= 6 and f[0].isdigit() and f[1].isdigit():
                    self.samples.append((int(f[0]), int(f[1]),
                                         {n for n, v in zip(names, f[2:6]) if v.lower().startswith("active")}))
            except Exception:
                pass
            self._halt.wait(0.2)

    def run(self):
        try:
            self._run_nvml()
        except Exception:
            self._run_smi()

    def stop(self):
        self._halt.set()
        self.join(timeout=5)
        sm = sorted(s[0] for s in self.samples)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": max((s[1] for s in self.samples), default=None),
                "reasons": sorted(set().union(*[s[2] for s in self.samples])) if self.samples else [],
                "samples": len(sm)}


def make_inputs(seed, batch, ebno_db=EBNO_DB):
    """Seeded synthetic channel logits for the all-zero codeword (a valid codeword of the linear code) sent with
    the reference's BPSK-equivalent mapping over AWGN: logit = log p(1)/p(0) = 4 y / no with y = -1 + w."""
    import numpy as np
    rng = np.random.default_rng(seed)
    no = 1.0 / (10 ** (ebno_db / 10) * (K_INFO / N_CODE))
    y = -1.0 + rng.standard_normal((batch, N_CODE), dtype=np.float32) * np.float32(np.sqrt(no / 2))
    return (np.float32(4.0 / no) * y).astype(np.float32)


def run_reference(args):
    """--impl reference: the reference's algorithm on the host cores. TensorFlow (the reference's backend) is not
    installable offline, so this times the CPU restatement (oracle/, libm math, all usable host threads) on a bounded
    sample of the same workload: SAMPLE codewords of the [4096, 8448] batch per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    from oracle import ldpc as O
    cores, core_info = host_cores()
    sample = max(cores * 2, 32)
    enc = O.LDPC5GEncoderRef(K_INFO, N_CODE)
    dec = O.LDPC5GDecoderRef(enc, cn_update=args.cn_update, num_iter=NUM_ITER)
    llr = make_inputs(1234, sample, args.ebno_db)
    for _ in range(args.warmup):
        dec(llr[:cores], num_threads=cores)
    t0 = time.perf_counter()
    errs = 0
    for _ in range(args.steps):
        u_hat = dec(llr, num_threads=cores)
        errs += int(u_hat.sum())
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        import torch
        dump_outputs(args.dump_outputs, {"u_hat": torch.from_numpy(np.asarray(u_hat))})
    val = sample * N_CODE * args.steps / dt
    line = {"metric": "coded bits/s, LDPC5G n=8448 k=4224 BP-20 decode", "value": val, "unit": "coded bits/s",
            "impl": "reference", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"LDPC5GDecoder(LDPC5GEncoder(4224,8448)) {args.cn_update} 20 it, "
                                   f"{sample}-codeword sample of the batch-4096 workload per step"},
            "cpu_baseline": {"value": val, "unit": "coded bits/s", "cores": cores, "core_detail": core_info, "kind": "port",
                             "sample": f"{sample} codewords/step x {args.steps} steps, oracle/ldpc_bp_ref.c libm mode, "
                                       f"OpenMP {cores} threads (TensorFlow reference not installable offline)"},
            "e2e": {"value": val, "unit": "coded bits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


_RESULT_FD = None


def emit(line):
    """Writes the ONE result line to the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def dump_outputs(out_dir, arrays):
    """--dump-outputs: writes what the timed path returned in its last step as out_dir/<name>.npy, so that two builds of
    the project can be compared output for output (the inputs are seeded: the same arguments give the same inputs).
    float64 and int64 arrays are stored as float64, all others as float32, complex ones as trailing (real, imag) pairs.
    An array larger than its share of DUMP_BYTES keeps a fixed, seeded sample of its rows, the same rows in every run."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    items = []
    for name, t in arrays.items():
        t = t.detach()
        if t.is_complex():
            t = torch.view_as_real(t)
        t = t.to(torch.float64 if t.dtype in (torch.float64, torch.int64) else torch.float32)
        items.append((name, t.cpu().numpy()))
    budget = DUMP_BYTES
    for j, (name, a) in enumerate(sorted(items, key=lambda it: it[1].nbytes)):
        share = budget // (len(items) - j)
        if a.ndim and a.nbytes > share:
            rows = np.random.default_rng(0).choice(a.shape[0], share // (a.nbytes // a.shape[0]), replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(out_dir, name + ".npy"), a)
        budget -= a.nbytes


def time_calls(fn, reps, warm=2):
    """Mean device milliseconds of `fn()` over `reps` back-to-back calls (CUDA events on the current stream)."""
    import torch
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def dist_setup(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep NCCL's banner / debug lines off stdout
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, "--gpus must match the torchrun world size"
    from sionna_b200.phy import config as sb_config
    sb_config.device = dev
    return rank, world, local, dev


# =====================================================================================================================
# configs[0], [2], [3], [4]: receive chains (tools/bench_links.py)
# =====================================================================================================================
def measure_link(wl, steps, warmup, world, dev, e2e_steps=None, stage_reps=5, dump_dir=None):
    """Times `steps` passes of the workload's hot path (device time, max over ranks), its per-stage roofline table and
    the end-to-end leg with host buffers. Returns a dict of results (used by run_link and by the default line's
    `config.other_workloads`). With `dump_dir`, the last timed pass's output is written there (dump_outputs)."""
    import torch
    import torch.distributed as dist
    from sionna_b200 import _lib
    for i in range(warmup):
        wl.run(i)
    if hasattr(wl, "counter"):
        wl.counter.reset()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reduced = torch.zeros(4, dtype=torch.int64, device=dev)
    l0 = _lib.lib().sb_launch_count()
    t0.record()
    for i in range(steps):
        out = wl.run(i)
        if world > 1 and hasattr(wl, "counter"):
            dist.all_reduce(reduced.copy_(wl.counter.counters), op=dist.ReduceOp.SUM)
    t1.record()
    launches = _lib.lib().sb_launch_count() - l0
    torch.cuda.synchronize()
    if dump_dir:
        dump_outputs(dump_dir, {"output": out, **({"error_counters": wl.counter.counters} if hasattr(wl, "counter") else {})})
    if world > 1:
        dist.barrier()
    t = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    res = {"ms_per_step": ms_total / steps, "value": world * wl.units_per_step * steps / (ms_total * 1e-3),
           "gpu_launches": launches}
    if hasattr(wl, "counter"):
        c = wl.counter.counters
        if world > 1:
            dist.all_reduce(reduced.copy_(c), op=dist.ReduceOp.SUM)
            c = reduced
        c = c.cpu().tolist()
        res["ber"] = {"bit_errors": c[0], "block_errors": c[1], "bits": c[2], "blocks": c[3]}
    # ---- per-stage table: each block call alone, CUDA events, inputs of the alternating sets (> L2 or rotated) ------
    peak, peak_src = measured_peak_gbs()
    table = []
    for name, fn, alg, note in wl.stages(0):
        ms = time_calls(fn, stage_reps)
        gbs = alg / ms * 1e-6
        table.append({"stage": name, "ms": ms, "alg_bytes": alg, "achieved_gbs": gbs, "frac": gbs / peak, "note": note})
    res["stages"] = table
    res["peak"], res["peak_source"] = peak, peak_src
    # ---- end to end: received samples from pinned host memory, result back to pinned host memory, 2 streams -----------
    wl.host_buffers()
    streams = [torch.cuda.Stream(device=dev) for _ in range(2)]
    n_e2e = e2e_steps or max(4, min(steps, 10))

    def e2e_step(i):
        with torch.cuda.stream(streams[i & 1]):
            x = wl.host_in[i & 1].to(dev, non_blocking=True)
            wl.host_out[i & 1].copy_(wl.run(i, x), non_blocking=True)

    for i in range(2):
        e2e_step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s_ in streams:
        s_.wait_event(e0)
    for i in range(n_e2e):
        e2e_step(i)
    for s_ in streams:
        torch.cuda.current_stream().wait_stream(s_)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    res["e2e"] = {"value": world * wl.units_per_step * n_e2e / (float(t.item()) * 1e-3), "unit": wl.unit,
                  "h2d_bytes_per_step": wl.h2d_bytes, "d2h_bytes_per_step": wl.d2h_bytes, "steps": n_e2e,
                  "pipeline": "2 CUDA streams, double-buffered pinned host buffers"}
    return res


def run_link(args):
    import torch
    import torch.distributed as dist
    from tools.bench_links import WORKLOADS
    rank, world, local, dev = dist_setup(args)
    from sionna_b200.phy import config as sb_config
    sb_config.seed = 300 + 1000 * rank
    wl = WORKLOADS[args.workload](dev, rank, world, args.batch)
    wl.build()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    res = measure_link(wl, args.steps, max(args.warmup, 3), world, dev,
                       dump_dir=args.dump_outputs if rank == 0 else None)
    clocks = sampler.stop() if sampler else None
    link = None
    if hasattr(wl, "link_step"):                                  # PUSCH: the whole Monte-Carlo step incl. tx + channel
        ms = time_calls(wl.link_step, max(3, args.steps // 2))
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        link = {"ms_per_step": float(t.item()), "transport_blocks_per_s": world * wl.batch / (float(t.item()) * 1e-3),
                "what": "PUSCHTransmitter + TDL generation + channel + PUSCHReceiver + error counting per step"}
    if rank == 0:
        on_path = [s for s in res["stages"] if not s["stage"].startswith("[separate]")]
        dom = max(on_path, key=lambda s: s["ms"]) if on_path else None
        line = {"metric": wl.metric, "value": res["value"], "unit": wl.unit, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": res["ms_per_step"], "higher_is_better": True,
                "scaling": wl.scaling, "vs_baseline": None, "dtype": wl.dtype, "data": "synthetic",
                "config": {"workload": wl.desc, "batch_per_gpu": wl.batch, "parallelism": f"{'shards' if wl.scaling == 'strong' else 'replicas'} x{world}",
                           "l2": "alternating / rotating input sets larger than L2"},
                "gpu_launches": res["gpu_launches"], "clocks": clocks, "e2e": res["e2e"]}
        if dom:
            line["roofline"] = {"bound": "hbm", "achieved": dom["achieved_gbs"], "peak": res["peak"], "unit": "GB/s",
                                "frac": dom["frac"], "traffic": None, "peak_source": res["peak_source"],
                                "kernel": dom["stage"], "kernel_ms": dom["ms"], "alg_bytes_per_launch": dom["alg_bytes"],
                                "stages": res["stages"]}
        if "ber" in res:
            line["config"]["ber"] = res["ber"]
        if link:
            line["config"]["monte_carlo_link"] = link
        if not args.no_cpu_baseline and world == 1:
            cores, core_info = host_cores()
            n = args.cpu_sample or {"qpsk_awgn": 256, "ofdm_siso": 32, "mimo_ofdm": 8}.get(wl.name, 0)
            cb = wl.cpu_chain(n) if n else None
            if cb:
                line["cpu_baseline"] = {"value": cb.pop("units") / cb["seconds"], "unit": wl.unit, "cores": cores,
                                        "core_detail": core_info, "kind": "port", "sample": cb.pop("what"), **cb}
            else:
                line["cpu_baseline"] = {"value": None, "unit": wl.unit, "cores": cores, "kind": "port",
                                        "sample": "no CPU restatement of this whole chain (its blocks are checked one by "
                                                  "one against oracle/ in tests/)"}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


# =====================================================================================================================
# configs[1]: LDPC5G BP decoding (headline)
# =====================================================================================================================
def traffic_probe(args):
    """Three decode launches on the bench's inputs; bench.py runs this leg under ncu to measure DRAM traffic."""
    import torch
    from sionna_b200.phy import config as sb_config
    from sionna_b200.phy.fec.ldpc import LDPC5GEncoder, LDPC5GDecoder
    torch.cuda.set_device(0)
    sb_config.device = torch.device("cuda", 0)
    dec = LDPC5GDecoder(LDPC5GEncoder(K_INFO, N_CODE), cn_update=args.cn_update, num_iter=NUM_ITER)
    x = [torch.from_numpy(make_inputs(s, BATCH, args.ebno_db)).cuda() for s in (1, 2)]
    for i in range(3):
        dec(x[i & 1])
    torch.cuda.synchronize()


def run_ldpc(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from sionna_b200 import _lib
    from sionna_b200.phy.fec.ldpc import LDPC5GEncoder, LDPC5GDecoder
    rank, world, local, dev = dist_setup(args)

    from sionna_b200.phy import config as sb_config
    from sionna_b200.phy.mapping import BinarySource, Mapper, Demapper
    from sionna_b200.phy.channel import AWGN
    from sionna_b200.phy.utils import ebnodb2no, ErrorCounter

    enc = LDPC5GEncoder(K_INFO, N_CODE)
    dec = LDPC5GDecoder(enc, cn_update=args.cn_update, num_iter=NUM_ITER, hard_out=True, return_infobits=True)
    assert dec.on_chip and dec.num_edges == E_EDGES and dec.num_vns == N_VNS

    # Synthetic inputs, generated once on the device by the package's own transmit chain (per-rank Philox stream):
    # BinarySource -> LDPC5GEncoder -> QPSK Mapper -> AWGN(Eb/N0 = 2 dB) -> Demapper("app"). Two distinct input sets
    # (2 x 138 MB > 126 MB L2) are alternated between steps: nothing the decoder reads can be an L2 hit left over
    # from the previous step.
    sb_config.seed = 100 + 1000 * rank
    src, mapper, demapper, awgn = BinarySource(), Mapper("qam", 2), Demapper("app", "qam", 2), AWGN()

    def synth(ebno_db):
        no = ebnodb2no(ebno_db, 2, K_INFO / N_CODE)
        us, xs = [], []
        for _ in range(2):
            u = src([BATCH, K_INFO])
            us.append(u)
            xs.append(demapper(awgn(mapper(enc(u)), no), no))
        return us, xs

    d_u, d_in = synth(args.ebno_db)
    h_in = [t.cpu().pin_memory() for t in d_in]
    counter = ErrorCounter(dev)                                   # device int64[4]: bit errors, block errors, bits, blocks
    reduced = torch.zeros(4, dtype=torch.int64, device=dev)

    def step(i):
        u_hat = dec(d_in[i & 1])
        counter.update(d_u[i & 1], u_hat)                         # sb_count_errors
        if world > 1:
            dist.all_reduce(reduced.copy_(counter.counters), op=dist.ReduceOp.SUM)
        return u_hat

    for i in range(args.warmup):
        step(i)
    counter.reset()
    torch.cuda.synchronize()

    # ---- timed region: K steps; CUDA events on the launching stream around every decode call for the roofline --------
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_start, t_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = _lib.lib().sb_launch_count()
    t_start.record()
    for i in range(args.steps):
        ev[i][0].record()
        u_hat = dec(d_in[i & 1])
        ev[i][1].record()
        counter.update(d_u[i & 1], u_hat)
        if world > 1:
            dist.all_reduce(reduced.copy_(counter.counters), op=dist.ReduceOp.SUM)
    t_stop.record()
    launches = _lib.lib().sb_launch_count() - launches0
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms_total = t_start.elapsed_time(t_stop)
    kern_ms = sum(a.elapsed_time(b) for a, b in ev) / args.steps
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = world * BATCH * N_CODE * args.steps / (ms_total * 1e-3)
    if world > 1:
        dist.all_reduce(reduced.copy_(counter.counters), op=dist.ReduceOp.SUM)
        totals = reduced.cpu().tolist()
    else:
        totals = counter.counters.cpu().tolist()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"u_hat": u_hat, "error_counters": counter.counters})

    # ---- end to end through the public API with HOST buffers: every step copies its logits from pinned host memory to
    # the device, decodes, and copies the decoded bits back to pinned host memory. Two streams are used round-robin so the
    # copies of one step overlap the kernel of the other (a double-buffered serving loop).
    h_out = [torch.empty((BATCH, K_INFO), dtype=torch.float32).pin_memory() for _ in range(2)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(2)]
    e2e_steps = max(4, min(args.steps, 10))

    def e2e_step(i):
        with torch.cuda.stream(streams[i & 1]):
            x = h_in[i & 1].to(dev, non_blocking=True)
            h_out[i & 1].copy_(dec(x), non_blocking=True)

    for i in range(2):
        e2e_step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s_ in streams:
        s_.wait_event(e0)
    for i in range(e2e_steps):
        e2e_step(i)
    for s_ in streams:
        torch.cuda.current_stream().wait_stream(s_)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_val = world * BATCH * N_CODE * e2e_steps / (float(t.item()) * 1e-3)

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        alg = ALG_BYTES_PER_CW * BATCH
        achieved = alg / (kern_ms * 1e-3) / 1e9
        c = totals
        traffic, traffic_src = None, None
        if world == 1 and not args.no_traffic:
            traffic = live_traffic(args.cn_update, args.ebno_db)
            traffic_src = "measured in this run: ncu dram__bytes_read.sum + dram__bytes_write.sum of one decode launch"
        if traffic is None:
            traffic, traffic_src = committed_traffic(args.cn_update)
            if traffic_src:
                traffic_src = "committed capture, not re-measured in this run: " + traffic_src
        line = {
            "metric": "coded bits/s, LDPC5G n=8448 k=4224 BP-20 decode", "value": value, "unit": "coded bits/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"configs[1]: LDPC5GDecoder(LDPC5GEncoder(4224,8448)), cn_update={args.cn_update}, "
                                   f"20 BP iterations, batch 4096 per GPU, QPSK/AWGN Eb/N0 {args.ebno_db:g} dB",
                       "cn_update": args.cn_update, "batch_per_gpu": BATCH, "parallelism": f"replicas x{world}", "ebno_db": args.ebno_db,
                       "l2": "2 alternating input sets of 138 MB each (> 126 MB L2)",
                       "ber": {"bit_errors": c[0], "block_errors": c[1], "bits": c[2], "blocks": c[3]}},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernel": "ldpc_bp_qc_kernel",
                         "kernel_ms": kern_ms, "alg_bytes_per_launch": alg},
            "e2e": {"value": e2e_val, "unit": "coded bits/s", "h2d_bytes_per_step": BATCH * N_CODE * 4,
                    "d2h_bytes_per_step": BATCH * K_INFO * 4, "steps": e2e_steps,
                    "pipeline": "2 CUDA streams, double-buffered pinned host buffers"},
            "gpu_launches": launches, "clocks": clocks,
        }
        # ---- the same kernel where its data-dependent shortcuts do not apply (0 dB: nothing converges) and the
        # north-star's min-sum rule, on this GPU, inside a key the driver keeps --------------------------------------
        if not args.no_variants:
            variants = {}
            if args.cn_update == "boxplus-phi" and args.ebno_db != 0.0:
                _, x0 = synth(0.0)
                ms = time_calls(lambda it=[0]: (dec(x0[it[0] & 1]), it.__setitem__(0, it[0] + 1)), 6)
                variants["boxplus-phi @ 0 dB"] = {"kernel_ms": ms, "value": BATCH * N_CODE / (ms * 1e-3),
                                                  "frac": alg / (ms * 1e-3) / 1e9 / peak}
                del x0
            if args.cn_update != "minsum":
                dec_ms = LDPC5GDecoder(enc, cn_update="minsum", num_iter=NUM_ITER, hard_out=True, return_infobits=True)
                ms = time_calls(lambda it=[0]: (dec_ms(d_in[it[0] & 1]), it.__setitem__(0, it[0] + 1)), 10, warm=3)
                variants["minsum"] = {"kernel_ms": ms, "value": BATCH * N_CODE / (ms * 1e-3),
                                      "frac": alg / (ms * 1e-3) / 1e9 / peak}
            try:                                              # opt-in early termination (NOT the reference's semantics)
                dec_et = LDPC5GDecoder(enc, cn_update=args.cn_update, num_iter=NUM_ITER, hard_out=True, return_infobits=True,
                                       early_stop=True)
                ms = time_calls(lambda it=[0]: (dec_et(d_in[it[0] & 1]), it.__setitem__(0, it[0] + 1)), 10, warm=3)
                variants[f"{args.cn_update} early_stop (opt-in; the reference always runs 20 iterations)"] = {
                    "kernel_ms": ms, "value": BATCH * N_CODE / (ms * 1e-3),
                    "mean_iterations": float(dec_et.num_iter_run.float().mean())}
            except Exception as e:
                variants["early_stop"] = {"error": repr(e)[:160]}
            line["roofline"]["variants"] = variants
        if not args.no_cpu_baseline and world == 1:           # reported baseline: rank 0 at N = 1 only
            from oracle import ldpc as O
            cores, core_info = host_cores()
            sample = min(BATCH, args.cpu_sample or max(32 * cores, 1024))   # ~10 s of CPU work on 128 threads
            ref = O.LDPC5GDecoderRef(O.LDPC5GEncoderRef(K_INFO, N_CODE), cn_update=args.cn_update, num_iter=NUM_ITER)
            x = h_in[0][:sample].numpy()
            ref(x[:cores], num_threads=cores)
            t0 = time.perf_counter()
            u_ref = ref(x, num_threads=cores)
            dt = time.perf_counter() - t0
            u_gpu = dec(d_in[0][:sample].contiguous()).cpu().numpy()
            line["cpu_baseline"] = {"value": sample * N_CODE / dt, "unit": "coded bits/s", "cores": cores,
                                    "core_detail": core_info, "kind": "port",
                                    "sample": f"first {sample} codewords of the step-0 batch, oracle/ldpc_bp_ref.c libm "
                                              f"mode, {cores} OpenMP threads",
                                    "bit_mismatch_vs_gpu": int((u_ref != u_gpu).sum())}
        # ---- the rest of the path (configs[0], [2], [3], [4]) in short form, so that the driver's record carries it ------
        if world == 1 and not args.no_links:
            del d_in, d_u, h_in, h_out
            torch.cuda.empty_cache()
            from tools.bench_links import WORKLOADS
            others = {}
            for name in ("qpsk_awgn", "ofdm_siso", "mimo_ofdm", "pusch"):
                try:
                    wl = WORKLOADS[name](dev, 0, 1, None)
                    wl.build()
                    r = measure_link(wl, 4, 3, 1, dev, e2e_steps=4, stage_reps=3)
                    on_path = [s for s in r["stages"] if not s["stage"].startswith("[separate]")]
                    dom = max(on_path, key=lambda s: s["ms"]) if on_path else {}
                    others[name] = {"value": r["value"], "unit": wl.unit, "ms_per_step": r["ms_per_step"],
                                    "e2e": r["e2e"]["value"], "dominant_stage": dom.get("stage"),
                                    "dominant_frac": dom.get("frac"),
                                    "stages": {s["stage"]: [round(s["ms"], 4), round(s["frac"], 3)] for s in r["stages"]}}
                    del wl
                    torch.cuda.empty_cache()
                except Exception as e:                             # a secondary workload must never cost the headline line
                    others[name] = {"error": repr(e)[:200]}
            line["config"]["other_workloads"] = others
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    # stdout carries exactly one JSON line: everything else that might write to fd 1 (NCCL's version banner, library
    # printf, build logs) is routed to stderr for the lifetime of the process
    global _RESULT_FD
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ldpc", choices=["ldpc", "qpsk_awgn", "ofdm_siso", "mimo_ofdm", "pusch"])
    ap.add_argument("--batch", type=int, default=0, help="override the workload's batch (link workloads only)")
    ap.add_argument("--cn-update", default="boxplus-phi",
                    choices=["boxplus-phi", "boxplus", "minsum", "offset-minsum"])
    ap.add_argument("--cpu-sample", type=int, default=0, help="codewords / frames for the cpu_baseline leg (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-variants", action="store_true", help="skip the 0 dB and min-sum side measurements")
    ap.add_argument("--no-links", action="store_true", help="skip the short measurement of configs[0], [2], [3], [4]")
    ap.add_argument("--no-traffic", action="store_true", help="do not re-measure DRAM traffic with ncu")
    ap.add_argument("--traffic-probe", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs to DIR/<name>.npy (float32 / float64, <= 64 MB in all)")
    ap.add_argument("--ebno-db", type=float, default=EBNO_DB,
                    help="Eb/N0 of the synthetic inputs (default 2 dB, SURVEY.md section 8d). The boxplus-phi kernel skips "
                         "provably-zero phi terms of saturated messages, so its speed depends on how early codewords converge")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.traffic_probe:
        return traffic_probe(args)
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "ldpc":
        return run_ldpc(args)
    return run_link(args)


if __name__ == "__main__":
    main()
