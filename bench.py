"""Headline benchmark: fwd+bwd TFLOP/s of causal cosine-sim attention at (B,H,N,D) = (4,8,4096,64),
bf16 - BASELINE.json's metric - on N GPUs of one node (one process per GPU; each rank runs the
same workload: batch x heads shards with no data-path collective, so scaling is "weak").

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this library
    python bench.py --impl reference [--steps K] [--warmup W]      # the reference's CPU path
    python bench.py ... --dump-outputs DIR                         # + what the last timed step computed

--steps K is the number of timed steps of every timed pass.  --dump-outputs writes o, dq, dk, dv of the last
headline step (rank 0) as DIR/{o,dq,dk,dv}.npy, float32 of shape (4, 8, 1024, 64): every (batch, head) at the
same 1024 sequence positions, drawn with a fixed seed (DUMP_ROWS).  The inputs are seeded too, so two builds
run with the same arguments can be compared output for output.  o, dk and dv repeat bit for bit from run to run;
dq is summed over key tiles by fp32 reduce-adds from many CTAs in no fixed order, so its final bf16 rounding can
land one step apart (4.9e-4 at most, on values up to 2.6, between two runs on a B200 at 1000 W).

One JSON line on stdout (rank 0).  Keys follow the driver contract; in short:
  value        whole-job TFLOP/s, inputs resident in HBM, timed with CUDA events per step
               (an L2 flush runs between steps, outside the events)
  e2e          the same metric through the public API starting from pinned HOST buffers:
               H2D of q,k,v,d_out and D2H of o,dq,dk,dv of every step inside the timed region
               (upload / compute / download on three streams, double-buffered across steps)
  roofline     the dominant kernel (the tcgen05 backward kernel), timed live with events recorded
               around exactly that launch, against the measured bf16 peak (MEASURED_PEAKS.json)
  cpu_baseline the reference's own naive path (plain_cosine_sim_attention, loaded unmodified by path when
               a copy is present, else the oracle's port of it) on the host cores
  c5           BASELINE config 5, (8,16,16384,128) bf16 causal, split over the N ranks by
               flash_cosine_sim_attention_b200.sharding (batch first: 8/N batch elements per GPU), fwd+bwd,
               plus - separately timed - the one NCCL all-gather of `o` a caller may ask for
"""
import argparse
import contextlib
import importlib.util
import io
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B, H, N, D = 4, 8, 4096, 64
SCALE, GROUPS = 8.0, 1
FWD_FLOPS = 4 * B * H * N * N * D / 2            # causal: half the score matrix (SURVEY.md par. 8d)
BWD_FLOPS = 2.5 * FWD_FLOPS                      # 5 GEMMs vs 2
STEP_FLOPS = FWD_FLOPS + BWD_FLOPS               # 2.405e11
METRIC = "fwd+bwd TFLOP/s at (4,8,4096,64) bf16 causal"
C5 = (8, 16, 16384, 128)
C5_FLOPS = 3.5 * 4 * C5[0] * C5[1] * C5[2] * C5[2] * C5[3] / 2      # 3.079e13
DUMP_ROWS = 1024                                 # sequence positions kept by --dump-outputs (32 MiB in all)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(bf16=p.get("bf16_tflops", 1590.0), bf16_sustained=p.get("bf16_tflops_sustained", 1400.0),
                    hbm=p.get("hbm_gbs", 6650.0), source="measured (MEASURED_PEAKS.json)")
    return dict(bf16=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons of ONE GPU, sampled by one background process (rank 0 only:
    eight pollers at 10 ms were part of the host-side contention seen at N = 8 in round 1).  It runs from
    before the warm-up to after the last timed pass; rows are time-stamped on arrival and only those that
    fall inside a marked window (the timed regions) are summarised."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.windows = index, [], None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    @contextlib.contextmanager
    def window(self):
        t0 = time.perf_counter()
        yield
        self.windows.append((t0, time.perf_counter()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.05)
        self.proc.terminate()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def summarise(rows):
            sm, mx, reasons = [], None, set()
            for _, r in rows:
                if len(r) < 6:
                    continue
                try:
                    sm.append(float(r[0]))
                    mx = float(r[1])
                except ValueError:
                    continue
                for nm, val in zip(names, r[2:6]):
                    if val.lower().startswith("active"):
                        reasons.add(nm)
            sm.sort()
            return sm, mx, reasons
        inside = [row for row in self.rows if any(a - 0.02 <= row[0] <= b + 0.02 for a, b in self.windows)]
        sm, mx, reasons = summarise(inside)
        scope = "timed regions"
        if not sm:          # the timed regions are a few ms long: fall back to everything sampled under load
            sm, mx, reasons = summarise(self.rows)
            scope = "whole run (warm-up to last pass)"
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "scope": scope}


# ---------------------------------------------------------------------------------------------------
# the reference arm: the reference's own CPU path on the host cores
# ---------------------------------------------------------------------------------------------------
REF_CANDIDATES = (os.path.join(ROOT, "baseline", "_ref", "flash_cosine_sim_attention", "flash_cosine_sim_attention.py"),)


def load_reference_plain():
    """The reference's plain_cosine_sim_attention, loaded UNMODIFIED by path (the package import itself
    fails without its compiled extension).  (fn, "reference") or (oracle port, "port")."""
    for path in REF_CANDIDATES:
        if os.path.exists(path):
            spec = importlib.util.spec_from_file_location("ref_fcsa_for_bench", path)
            mod = importlib.util.module_from_spec(spec)
            with contextlib.redirect_stdout(io.StringIO()):     # it prints a "not compiled" hint
                spec.loader.exec_module(mod)
            return mod.plain_cosine_sim_attention, "reference", path
    from oracle import cosine_sim_attention_oracle as oracle

    def port(q, k, v, scale=8, groups=1, causal=False):
        return oracle.torch_cpu_forward_backward(q, k, v, scale=scale, groups=groups, causal=causal, backward=False)
    return port, "port", "oracle/cosine_sim_attention_oracle.py"


def cpu_reference_sample(torch, fn, heads):
    """One bounded sample of the workload on the host: (1, heads, 4096, 64) f32 causal fwd+bwd through the
    reference's naive path.  Returns (seconds, flops)."""
    g = torch.Generator().manual_seed(0)
    q, k, v = (torch.randn(1, heads, N, D, generator=g).requires_grad_() for _ in range(3))
    t0 = time.perf_counter()
    out = fn(q, k, v, scale=SCALE, groups=GROUPS, causal=True)
    out.sum().backward()
    dt = time.perf_counter() - t0
    return dt, STEP_FLOPS * heads / (B * H)


def host_threads(torch, fn=None):
    """Thread count for the CPU arm, also under torchrun (which exports OMP_NUM_THREADS=1).  All allowed cores are
    offered; when `fn` is given the candidates {all, 64, 32, 16} are each timed on one bounded sample and the fastest
    is kept (on a 128-thread host the naive path of a 2-head sample runs 3-4x faster on 32 threads than on 128)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    n = max(1, n)
    if fn is None:
        torch.set_num_threads(n)
        return torch.get_num_threads()
    best, best_t = n, None
    for cand in sorted({n, min(n, 64), min(n, 32), min(n, 16)}, reverse=True):
        torch.set_num_threads(cand)
        t, _ = cpu_reference_sample(torch, fn, 2)
        if best_t is None or t < best_t:
            best, best_t = cand, t
    torch.set_num_threads(best)
    return torch.get_num_threads()


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path (naive PyTorch ops on the
    host cores).  Rank 0 alone runs it; the other ranks exit."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    fn, kind, src = load_reference_plain()
    cores = host_threads(torch, fn)
    heads = 2                                    # bounded sample: 1/16 of the workload per step
    for _ in range(max(args.warmup, 1)):
        cpu_reference_sample(torch, fn, heads)
    tot_t, tot_f = 0.0, 0.0
    for _ in range(args.steps):
        dt, fl = cpu_reference_sample(torch, fn, heads)
        tot_t += dt
        tot_f += fl
    val = tot_f / tot_t / 1e12
    sample = (f"(1,{heads},4096,64) f32 causal fwd+bwd per step = {heads}/{B*H} of the workload, {src}; "
              f"{os.cpu_count()} logical cpus, thread count calibrated over {{all, 64, 32, 16}}")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "TFLOP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": tot_t / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "causal self-attn (4,8,4096,64) fwd+bwd, cosine-sim, scale 8", "sample": sample,
                   "note": "ms_per_step is the time of ONE bounded sample; value = sample FLOPs / sample time"},
        "cpu_baseline": {"value": val, "unit": "TFLOP/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa_node(torch, index):
    """Pin this rank's host threads (and therefore its pinned staging buffers: first touch) to the NUMA node the
    GPU hangs off.  Host<->device copies through the other socket ran at half the bandwidth on some boxes, and
    eight ranks enqueueing from arbitrary cores was part of the N = 8 slowdown of round 1.  Best effort."""
    try:
        bus = torch.cuda.get_device_properties(index).pci_bus_id
        dom = torch.cuda.get_device_properties(index).pci_domain_id
        dev = torch.cuda.get_device_properties(index).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return {"node": None, "note": "kernel reports no NUMA affinity for the GPU"}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return {"node": node, "note": "no allowed cpu on that node"}
        os.sched_setaffinity(0, allowed)
        return {"node": node, "cpus": len(allowed)}
    except Exception as e:      # noqa: BLE001
        return {"node": None, "note": f"not bound ({type(e).__name__})"}


def dump_outputs(out_dir, outs):
    """Write o, dq, dk, dv of one step as float32 DIR/<name>.npy: every (batch, head) at DUMP_ROWS sequence positions
    drawn with a fixed seed (the full tensors would be 128 MiB).  Returns a description for the JSON line."""
    import numpy as np
    import torch
    rows = np.sort(np.random.default_rng(0).choice(N, DUMP_ROWS, replace=False))
    idx = torch.from_numpy(rows).to(outs[0].device)
    names = ("o", "dq", "dk", "dv")
    for name, t in zip(names, outs):
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().index_select(2, idx).float().cpu().numpy())
    return {"dir": out_dir, "files": [n + ".npy" for n in names], "dtype": "float32",
            "shape": [B, H, DUMP_ROWS, D], "sample": f"{DUMP_ROWS} of {N} sequence positions, numpy seed 0"}


# ---------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c5", action="store_true", help="skip the config-5 (8,16,16384,128) sharded measurement")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a seeded sample of o, dq, dk, dv of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to --impl b200")
        return run_reference_arm(args)
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    saved_stdout_fd = None
    if world > 1:
        # NCCL's INFO lines (version banner, "nranks N", NVLS/ring choice) must be visible so the run can be
        # checked for a real N-rank communicator, but NCCL writes them to STDOUT and stdout has to stay one JSON
        # line: file descriptor 1 points at stderr for the whole run (every rank); rank 0 restores it for the
        # very last thing it does, printing the line.
        os.environ.setdefault("NCCL_DEBUG", "INFO")
        sys.stdout.flush()
        saved_stdout_fd = os.dup(1)
        os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    from flash_cosine_sim_attention_b200 import _abi, debug, flash_cosine_sim_attention
    from flash_cosine_sim_attention_b200.sharding import shard_range, sharded_flash_cosine_sim_attention

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(torch, local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        probe = torch.ones(1, device=dev)
        dist.all_reduce(probe)                   # creates the communicator now; every rank contributes 1
        if rank == 0:
            print(f"[bench] NCCL communicator up: nranks {world} (all_reduce of ones = {int(probe.item())}), "
                  f"NCCL {'.'.join(map(str, torch.cuda.nccl.version()))}, one process per GPU", file=sys.stderr, flush=True)
    lib = _abi.load()
    W = max(args.warmup, 3)
    K = args.steps
    dt = torch.bfloat16

    g = torch.Generator().manual_seed(rank)
    host = [torch.randn(B, H, N, D, generator=g).to(dt).pin_memory() for _ in range(4)]   # q, k, v, d_out
    q, k, v, do = (t.to(dev) for t in host)
    q.requires_grad_(), k.requires_grad_(), v.requires_grad_()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)                 # > 126 MB L2

    def step(qq, kk, vv, dd):
        o = flash_cosine_sim_attention(qq, kk, vv, causal=True, scale=SCALE, groups=GROUPS)
        return (o,) + torch.autograd.grad(o, (qq, kk, vv), dd)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    for _ in range(W):
        step(q, k, v, do)
    barrier()

    # ---- device-resident timing -------------------------------------------------------------
    NEV = 5                                      # l2norm(q,k), forward, preprocess, backward, dq conversion
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    kev = [[torch.cuda.Event(enable_timing=True) for _ in range(2 * NEV)] for _ in range(K)]
    for row in kev:                                                                       # materialise handles
        for e in row:
            e.record()
    launches0 = debug()
    barrier()
    # pass 1 - the headline: exactly K steps of the public API, nothing else on the stream between the
    # kernels of a step (an event recorded between two launches would turn their programmatic dependent
    # launch back into a full serialisation).  A ~1 ms spin kernel in front of the loop (outside every event
    # pair) plus two untimed steps let the launch queue fill and the clocks ramp after the barrier.
    with (sampler.window() if sampler else contextlib.nullcontext()):
        torch.cuda._sleep(2_000_000)
        for _ in range(2):
            flush.zero_()
            step(q, k, v, do)
        host_t0 = time.perf_counter()
        for i in range(K):
            flush.zero_()
            ev[i][0].record()
            outs = step(q, k, v, do)
            ev[i][1].record()
            if i < K - 1:
                # freed at once, as in the warm-up: outputs held into the next step would make the caching
                # allocator grow (cudaMalloc) inside the timed region
                del outs
        host_enqueue_us = (time.perf_counter() - host_t0) / K * 1e6      # host time to ENQUEUE one step (no sync inside)
        barrier()
    dumped = dump_outputs(args.dump_outputs, outs) if args.dump_outputs and rank == 0 else None
    del outs
    launches_per_step = (debug() - launches0) // (K + 2)
    launches = launches_per_step * K
    step_ms = [a.elapsed_time(b) for a, b in ev]
    # pass 2 - attribution: the same K steps again with events recorded around each kernel of the step
    # (library hook); not part of `value`
    which = {"l2norm_qk": 2, "forward": 0, "preprocess": 3, "backward": 1, "dq_finish": 4}
    with (sampler.window() if sampler else contextlib.nullcontext()):
        torch.cuda._sleep(2_000_000)
        for i in range(K):
            flush.zero_()
            for slot, w in enumerate(which.values()):
                lib.fcsa_set_kernel_events(w, kev[i][2 * slot].cuda_event, kev[i][2 * slot + 1].cuda_event)
            step(q, k, v, do)
        barrier()
    for w in range(5):
        lib.fcsa_set_kernel_events(w, None, None)
    # the poller stops here: NVML queries during the end-to-end pass below were seen to stall the PCIe copies
    # (30 ms per step instead of 1.5 ms with a 20 ms poll period)
    clocks = sampler.stop() if sampler else None
    parts = {name: sum(r[2 * slot].elapsed_time(r[2 * slot + 1]) for r in kev) / K for slot, name in enumerate(which)}
    fwd_avg, bwd_avg = parts["forward"], parts["backward"]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)

    # ---- end to end from pinned host buffers ---------------------------------------------------
    # Every step copies its four inputs host->device and its four results device->host; the copies
    # are inside the timed region.  Three streams (upload, compute, download) and two sets of device
    # buffers: the upload of step i+1 and the download of step i-1 run under the compute of step i,
    # the way an input pipeline feeds a training loop.  The compute is the public API call.
    houts = [[torch.empty(B, H, N, D, dtype=dt).pin_memory() for _ in range(4)] for _ in range(2)]
    dins = [[torch.empty(B, H, N, D, dtype=dt, device=dev) for _ in range(4)] for _ in range(2)]
    for bufs in dins:
        for t in bufs[:3]:
            t.requires_grad_()
    s_up, s_cmp, s_dn = torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    ev_up = [torch.cuda.Event() for _ in range(2)]      # inputs of buffer set b are on the device
    ev_cmp = [torch.cuda.Event() for _ in range(2)]     # results of buffer set b are computed (inputs consumed)
    ev_dn = [torch.cuda.Event() for _ in range(2)]      # results of buffer set b are on the host

    def e2e_run(n):
        keep = [None, None]
        for i in range(n):
            bsel = i & 1
            with torch.cuda.stream(s_up):
                s_up.wait_event(ev_cmp[bsel])               # step i-2 has consumed this buffer set
                with torch.no_grad():
                    for dst, src in zip(dins[bsel], host):
                        dst.copy_(src, non_blocking=True)
                ev_up[bsel].record(s_up)
            with torch.cuda.stream(s_cmp):
                s_cmp.wait_event(ev_up[bsel])
                outs = step(*dins[bsel])
                ev_cmp[bsel].record(s_cmp)
            with torch.cuda.stream(s_dn):
                s_dn.wait_event(ev_cmp[bsel])
                s_dn.wait_event(ev_dn[bsel])                # host buffers of step i-2 are written
                for dst, src in zip(houts[bsel], outs):
                    src.record_stream(s_dn)
                    dst.copy_(src.detach(), non_blocking=True)
                ev_dn[bsel].record(s_dn)
            keep[bsel] = outs
        for st in (s_up, s_cmp, s_dn):
            torch.cuda.current_stream().wait_stream(st)

    e2e_run(2)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with contextlib.nullcontext():
        e0.record()
        for st in (s_up, s_cmp, s_dn):
            st.wait_stream(torch.cuda.current_stream())
        e2e_run(K)
        e1.record()
        barrier()
    e2e_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    del houts, dins, host

    # ---- config 5: (8,16,16384,128) bf16 causal split over the ranks (SURVEY par. 8e) -------------------
    c5 = None
    if not args.no_c5:
        Bc, Hc, Nc, Dc = C5
        # every rank owns its batch elements (8 / world of the 8): generated per global batch index, so the
        # union over ranks is the same problem at every N
        lo, hi = shard_range(Bc, rank, world)

        def gen(seed):
            parts_ = []
            for bi in range(lo, hi):
                gc = torch.Generator(device=dev).manual_seed(1000 * seed + bi)
                parts_.append(torch.randn(1, Hc, Nc, Dc, generator=gc, device=dev, dtype=dt))
            return torch.cat(parts_, 0)
        qc, kc, vc, dc = gen(1), gen(2), gen(3), gen(4)
        qc.requires_grad_(), kc.requires_grad_(), vc.requires_grad_()

        def c5_step():
            o = sharded_flash_cosine_sim_attention(qc, kc, vc, causal=True, scale=SCALE, presharded=True)
            grads = torch.autograd.grad(o, (qc, kc, vc), dc)
            return o, grads
        for _ in range(2):
            c5_step()
        barrier()
        KC = K
        cev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(KC)]
        for i in range(KC):
            cev[i][0].record()
            o5, _ = c5_step()
            cev[i][1].record()
        barrier()
        c5_ms = torch.tensor([sum(a.elapsed_time(b) for a, b in cev) / KC], dtype=torch.float64, device=dev)
        gather_ms, gather_ok = None, None
        if world > 1:
            # the one collective of the path, only when the caller wants the whole-batch output: an NCCL
            # all-gather of o over NVLink, timed on its own and checked against the local shard
            full = torch.empty(Bc, Hc, Nc, Dc, dtype=dt, device=dev)
            o5c = o5.contiguous()
            dist.all_gather_into_tensor(full, o5c)
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(3):
                dist.all_gather_into_tensor(full, o5c)
            g1.record()
            barrier()
            gm = torch.tensor([g0.elapsed_time(g1) / 3], dtype=torch.float64, device=dev)
            dist.all_reduce(gm, op=dist.ReduceOp.MAX)
            dist.all_reduce(c5_ms, op=dist.ReduceOp.MAX)
            gather_ms = float(gm.item())
            ok = torch.tensor([int(torch.equal(full[lo:hi], o5c) and bool(torch.isfinite(full.float()).all())
                                   and bool((full.float().abs().amax(dim=(1, 2, 3)) > 0).all()))], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            gather_ok = bool(ok.item())
            del full
        c5_ms_f = float(c5_ms.item())
        c5 = {"workload": f"(8,16,16384,128) bf16 causal fwd+bwd, batch split {Bc // world if Bc % world == 0 else '~' + str(Bc / world)} "
                          f"per GPU x {world} (sharding.py, no data-path collective)",
              "ms_per_step": c5_ms_f, "tflops": C5_FLOPS / (c5_ms_f * 1e-3) / 1e12, "steps": KC, "scaling": "strong",
              "all_gather_o_ms": gather_ms, "all_gather_o_bytes": Bc * Hc * Nc * Dc * 2 if world > 1 else 0,
              "all_gather_o_gbs_per_rank": (Bc * Hc * Nc * Dc * 2 * (world - 1) / world / (gather_ms * 1e-3) / 1e9)
                                           if gather_ms else None,
              "gathered_output_matches_local_shard": gather_ok}
        del qc, kc, vc, dc, o5

    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
        he = torch.tensor([host_enqueue_us], dtype=torch.float64, device=dev)
        dist.all_reduce(he, op=dist.ReduceOp.MAX)
        host_enqueue_us = float(he.item())
    total_ms, e2e_ms = float(total_ms.item()), float(e2e_ms.item())

    if rank == 0:
        peaks = load_peaks()
        value = STEP_FLOPS * K * world / (total_ms * 1e-3) / 1e12
        e2e_val = STEP_FLOPS * K * world / (e2e_ms * 1e-3) / 1e12
        ach = BWD_FLOPS / (bwd_avg * 1e-3) / 1e12
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get("fcsa_bwd_kernel_dram_bytes_per_launch")
        aux = parts["l2norm_qk"] + parts["preprocess"] + parts["dq_finish"]
        line = {
            "metric": METRIC, "value": value, "unit": "TFLOP/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "causal self-attn (B,H,N,D)=(4,8,4096,64) per GPU, cosine-sim (l2norm of q,k inside the op), "
                                   "scale 8, fwd+bwd through flash_cosine_sim_attention()",
                       "global_batch": B * world, "seq_len": N, "heads": H, "head_dim": D,
                       "parallelism": f"batch-shard x{world} (no data-path collective)",
                       "l2": "256 MiB L2 flush between timed steps (outside the events)",
                       "timing": "W warm-up steps, barrier+sync, 2 more untimed steps (clock ramp, launch queue), K steps "
                                 "each between its own CUDA events, barrier+sync; max over ranks",
                       "flops_per_step_per_gpu": STEP_FLOPS},
            "frac_of_peak": value / world / peaks["bf16"], "peak_source": peaks["source"],
            "roofline": {"bound": "tensor", "kernel": "fcsa_bwd_kernel<bf16,64>",
                         "achieved": ach, "peak": peaks["bf16"], "unit": "TFLOP/s", "frac": ach / peaks["bf16"],
                         "traffic": traffic, "ms": bwd_avg, "flops_per_launch": BWD_FLOPS},
            "roofline_fwd": {"bound": "tensor", "kernel": "fcsa_fwd_kernel<bf16,64>",
                             "achieved": FWD_FLOPS / (fwd_avg * 1e-3) / 1e12, "peak": peaks["bf16"],
                             "unit": "TFLOP/s", "frac": FWD_FLOPS / (fwd_avg * 1e-3) / 1e12 / peaks["bf16"],
                             "ms": fwd_avg, "flops_per_launch": FWD_FLOPS},
            "e2e": {"value": e2e_val, "unit": "TFLOP/s", "h2d_bytes_per_step": 4 * B * H * N * D * 2 * world,
                    "d2h_bytes_per_step": 4 * B * H * N * D * 2 * world, "ms_per_step": e2e_ms / K},
            "step_breakdown_ms": {**parts, "aux_total": aux,
                                  "note": "instrumented second pass (events between the launches); the headline pass "
                                          "has none"},
            "gpu_launches": int(launches), "gpu_launches_per_step": int(launches_per_step),
            "host_enqueue_us_per_step": host_enqueue_us, "numa": numa, "clocks": clocks,
            "ms_per_step_min_median_max": [min(step_ms), sorted(step_ms)[len(step_ms) // 2], max(step_ms)],
            "slowest_step_index": int(max(range(len(step_ms)), key=lambda j: step_ms[j])),
        }
        if c5 is not None:
            line["c5"] = c5
        if dumped is not None:
            line["dumped_outputs"] = dumped
        if world == 1 and not args.no_cpu_baseline:
            fn, kind, src = load_reference_plain()
            cores = host_threads(torch, fn)                           # calibrates the thread count (also the warm-up)
            t, f = 0.0, 0.0
            for _ in range(3):
                a, b = cpu_reference_sample(torch, fn, 2)
                t, f = t + a, f + b
            line["cpu_baseline"] = {"value": f / t / 1e12, "unit": "TFLOP/s", "cores": cores, "kind": kind,
                                    "sample": "3 x (1,2,4096,64) f32 causal fwd+bwd (2/32 of the workload each), "
                                              f"naive path of {src}, {os.cpu_count()} logical cpus"}
        final_line = json.dumps(line)
    else:
        final_line = None
    if world > 1:
        dist.destroy_process_group()
    if final_line is not None:
        sys.stdout.flush()
        if saved_stdout_fd is not None:
            os.dup2(saved_stdout_fd, 1)
        print(final_line, flush=True)


if __name__ == "__main__":
    main()
