#!/usr/bin/env python
"""Evoformer trunk forward benchmark (BASELINE.json: residue-pairs/sec at N_res=256, depth=12; fwd ms/block).

    python bench.py --gpus 1 --steps 10 --warmup 3                      # B200 arm (this repo)
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1      # CPU arm: oracle port of the reference
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...    # one rank per GPU

A "step" is one forward of the C2 workload: Alphafold2(dim=256, depth=12, heads=8, dim_head=64),
N_res=256, MSA 128x256, batch 1, synthetic tokens, all-ones masks, random-init weights (zero-init
tensors randomised so no path is an identity).
  value = residue-pairs/s of the trunk (Evoformer.forward) with x / m already resident in HBM;
  e2e   = the same metric through the public API Alphafold2.forward(seq, msa, mask, msa_mask) with HOST
          (pinned) inputs: H2D of the token ids / masks and D2H of the distogram logits inside the timed region.
Timing: CUDA events per step on the launching stream, L2 flushed (256 MiB write) between steps outside the
event pairs, barrier + synchronize around the loop, max over ranks.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CFG = dict(dim=256, depth=12, heads=8, dim_head=64)
WORKLOADS = {"C2": (256, 128), "C3": (384, 512), "C4": (512, 1024)}      # BASELINE.json configs[1..3]: (N_res, MSA rows)
N_RES, N_SEQ = WORKLOADS["C2"]
WORKLOAD = "C2: Alphafold2(dim=256,depth=12,heads=8,dim_head=64) N_res=256 MSA=128x256 batch=1"


def set_workload(name):
    """The default (C2) is the configuration BASELINE.json quotes the metric on; C3 / C4 are its larger shapes."""
    global N_RES, N_SEQ, WORKLOAD
    N_RES, N_SEQ = WORKLOADS[name]
    WORKLOAD = f"{name}: Alphafold2(dim=256,depth=12,heads=8,dim_head=64) N_res={N_RES} MSA={N_SEQ}x{N_RES} batch=1"

METRIC = "evoformer_residue_pairs_per_sec"
UNIT = "residue-pairs/s"


def flops_per_block(N, S, d, H, dh):
    """Algorithmic matmul FLOPs of one EvoformerBlock (SURVEY.md §8d)."""
    I = H * dh
    Tm, Tx = S * N, N * N
    return float(10 * Tm * d * I + 2 * Tx * d * H + 4 * S * N * N * I + 10 * Tm * d * I + 4 * N * S * S * I +
                 24 * Tm * d * d + 4 * Tm * d * d + 2 * N * N * S * d + 2 * Tx * d * d +
                 2 * (12 * Tx * d * d + 2 * N ** 3 * d) + 2 * (10 * Tx * d * I + 2 * Tx * d * H + 4 * N ** 3 * I) +
                 24 * Tx * d * d)


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(tflops=float(p["bf16_tflops_sustained"]), tflops_burst=float(p["bf16_tflops"]),
                    hbm_gbs=float(p["hbm_gbs"]), source="MEASURED_PEAKS.json (measured)")
    except Exception:
        return dict(tflops=1400.0, tflops_burst=1590.0, hbm_gbs=6650.0, source="B200_PROFILING.md fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.proc, self.lines, self.index = None, [], index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [t.strip() for t in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


DUMP_ELEMS = 2 ** 22     # per array: the three dumped arrays stay under 64 MiB of float32 together


def output_sample(t, seed):
    """float32 host copy of `t`: the whole tensor when it has at most DUMP_ELEMS elements, else DUMP_ELEMS elements at
    seeded flat indices, so that runs with the same arguments dump the same elements."""
    flat = t.detach().reshape(-1)
    if flat.numel() <= DUMP_ELEMS:
        return t.detach().float().cpu().numpy()
    idx = torch.randint(flat.numel(), (DUMP_ELEMS,), generator=torch.Generator().manual_seed(seed))
    return flat[idx.to(flat.device)].float().cpu().numpy()


def write_outputs(out_dir, arrays):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def randomize_zero_init_(model, std=0.02, seed=1234):
    """Quirk Q8: zero-init projections / identity gates would make most of the trunk an identity."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if bool((p == 0).all()):
                p.copy_(torch.randn(p.shape, generator=g) * std)
            elif bool((p == 1).all()) and (".gating." in name or "_gate." in name):
                p.copy_(1.0 + torch.randn(p.shape, generator=g) * std)


# ------------------------------------------------------------------------------------------------------------------
# CPU arm: oracle port of the reference (the Python reference itself cannot travel to the GPU box)
# ------------------------------------------------------------------------------------------------------------------
def exchange_transport():
    """How the sharded schedule moved its row<->column re-layouts in this run (alphafold2_b200/parallel.py)."""
    from alphafold2_b200 import parallel as _p
    live = [ex for ex in _p._PEER_ARENAS.values() if ex is not None]
    if live:
        return {"all_to_all": "peer-store kernel over CUDA IPC mappings (af2_peer_exchange)", "exchanges": sum(ex.exchanges for ex in live),
                "barrier_timeouts": int(any(ex.error() for ex in live)), "all_gather": "NCCL"}
    return {"all_to_all": "NCCL all_to_all_single + pack/unpack copies", "all_gather": "NCCL"}


def host_threads():
    """All the host CORES the CPU arm can use.  torchrun exports OMP_NUM_THREADS=1 to its workers (round 1's N>1 CPU arm ran
    on one thread), so the count is set explicitly -- to the PHYSICAL cores: with one thread per hyper-thread (128 on the
    pool's 64-core hosts) MKL / OpenMP oversubscribe and the block takes 131 s instead of 6.9 s (measured, profiles/r02a)."""
    n = None
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
    except Exception:
        n = None
    if not n:
        n = max(1, (os.cpu_count() or 2) // 2)
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    torch.set_num_threads(int(n))
    return torch.get_num_threads()


def make_config(world):
    """One config dict for both arms (the driver compares them)."""
    return {"workload": WORKLOAD,
            "parallelism": "single GPU" if world == 1 else
            f"1 sequence axis-sharded over {world} GPUs (MSA-row / pair-row shards; per block 6 all-gathers + 6 all-to-alls over NCCL)",
            "l2": "flushed between timed steps (256 MiB write outside the event pairs)",
            "accumulate": "fp32", "residual_stream": "fp32"}


def cpu_block_sample(literal=False):
    """One Evoformer block of the C2 workload on the host cores (fp32); the forward is 12 identical blocks.
    literal=False: the oracle's einsum OuterMean (validated against the reference), several times FASTER on a CPU than the
    reference's literal (S,N,N,d) materialisation (alphafold2.py:341, 73 % of its block time, SURVEY.md 6) -- a conservative
    baseline.  literal=True follows alphafold2.py:341-349 line by line (needs ~18 GB of RSS at C2)."""
    from oracle import evoformer_oracle as O
    import alphafold2_b200 as A
    torch.manual_seed(0)
    d, H, dh = CFG["dim"], CFG["heads"], CFG["dim_head"]
    blk = A.EvoformerBlock(dim=d, seq_len=N_RES, heads=H, dim_head=dh, attn_dropout=0., ff_dropout=0.)   # parameter container only
    randomize_zero_init_(blk)
    w = {k: v.detach() for k, v in blk.state_dict().items()}
    x = torch.randn(1, N_RES, N_RES, d)
    m = torch.randn(1, N_SEQ, N_RES, d)
    mask = torch.ones(1, N_RES, N_RES, dtype=torch.bool)
    msa_mask = torch.ones(1, N_SEQ, N_RES, dtype=torch.bool)

    def step():
        t0 = time.perf_counter()
        with torch.no_grad():
            O.evoformer_block(w, "", x, m, H, mask, msa_mask, literal_outer=literal)
        return time.perf_counter() - t0
    return step


def literal_ok():
    try:
        import psutil
        return psutil.virtual_memory().available > 40 * 2 ** 30
    except Exception:
        return False


def cpu_baseline(max_seconds=30.0):
    """Bounded sample on the host cores (rank 0, N = 1 only): one block with the einsum OuterMean (the reported value) and,
    when the box has the memory, one block with the reference's literal OuterMean next to it."""
    cores = host_threads()
    step = cpu_block_sample(False)
    t = step()
    if t < max_seconds / 3:
        t = min(t, step())
    fwd = t * CFG["depth"]
    out = {"value": N_RES * N_RES / fwd, "unit": UNIT, "cores": cores, "kind": "port",
           "sample": f"1 of {CFG['depth']} Evoformer blocks of the C2 workload (fp32 torch CPU oracle port, einsum OuterMean), "
                     f"{t:.2f} s/block x {CFG['depth']}",
           "seconds_per_block": t}
    if literal_ok():
        try:
            tl = cpu_block_sample(True)()
            out["literal_outer_seconds_per_block"] = tl
            out["literal_outer_value"] = N_RES * N_RES / (tl * CFG["depth"])
            out["sample"] += f"; same block with the literal (S,N,N,d) OuterMean of alphafold2.py:341: {tl:.2f} s/block"
        except Exception as ex:  # noqa: BLE001
            out["literal_outer_error"] = repr(ex)[:200]
    return out


def run_reference(args, rank, world):
    """Reference arm: the reference's CPU path (oracle port; the Python reference cannot travel to the GPU box) on all host
    threads.  A step is a bounded sample of the C2 forward: ONE of its 12 identical Evoformer blocks; `ms_per_step` is the
    measured time of that sample, `value` the residue-pairs/s of the whole forward it implies (N^2 / (12 x block))."""
    if rank != 0:
        return
    cores = host_threads()
    step = cpu_block_sample(False)
    budget = float(os.environ.get("AF2_REF_BUDGET_S", "420"))
    t_start = time.perf_counter()
    warm = 0
    for _ in range(args.warmup):
        step()
        warm += 1
        if time.perf_counter() - t_start > budget * 0.3:
            break
    times = [step() for _ in range(args.steps)]
    t_blk = sum(times) / len(times)
    fwd = t_blk * CFG["depth"]
    val = N_RES * N_RES / fwd
    sample = f"each step = 1 of {CFG['depth']} Evoformer blocks of the C2 workload on {cores} host threads (fp32 oracle port, " \
             f"einsum OuterMean); forward = {CFG['depth']} x block; value = N_res^2 / forward"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
        "warmup": warm, "ms_per_step": t_blk * 1e3, "ms_per_block": t_blk * 1e3, "ms_per_forward": fwd * 1e3,
        "higher_is_better": True,
        "scaling": "weak" if world == 1 else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(world),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def gpu_torch_baseline(dev, x0, m0, x_mask, msa_mask, model):
    """Same-silicon yardstick (BASELINE.md 3.8), OUTSIDE every timed region of this repo's arm: the oracle port of the
    reference trunk run by stock PyTorch (ATen / cuBLAS) on this GPU in fp32 and under autocast-bf16."""
    from oracle import evoformer_oracle as O
    w = {k[len("net."):]: v.detach() for k, v in model.state_dict().items() if k.startswith("net.")}
    out = {}
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        for name, ctx in (("fp32", None), ("autocast_bf16", torch.autocast("cuda", dtype=torch.bfloat16))):
            def fwd():
                with torch.no_grad():
                    if ctx is None:
                        return O.evoformer(w, "", x0, m0, CFG["heads"], CFG["depth"], x_mask, msa_mask, chunk=64)
                    with ctx:
                        return O.evoformer(w, "", x0, m0, CFG["heads"], CFG["depth"], x_mask, msa_mask, chunk=64)
            fwd()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(3):
                fwd()
            b.record()
            b.synchronize()
            ms = a.elapsed_time(b) / 3
            out[name] = {"ms_per_step": ms, "value": N_RES * N_RES / (ms * 1e-3), "unit": UNIT}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    out["what"] = "oracle port of the reference trunk (einsum OuterMean) executed by stock PyTorch eager on the same B200; not part of any timed region"
    return out


# ------------------------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    import alphafold2_b200 as A
    from alphafold2_b200 import _lib
    import ctypes as C

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    torch.manual_seed(0)
    model = A.Alphafold2(**CFG)
    randomize_zero_init_(model)
    model = model.to(dev).eval()
    if world > 1:
        # one sequence, trunk sharded over the MSA-row / pair-row axes of all ranks (alphafold2_b200/parallel.py):
        # STRONG scaling -- total work is fixed, every rank gets the same replicated inputs and the full outputs
        from alphafold2_b200.parallel import shard_evoformer
        shard_evoformer(model)

    seq_h = torch.randint(0, 21, (1, N_RES)).pin_memory()
    msa_h = torch.randint(0, 21, (1, N_SEQ, N_RES)).pin_memory()
    mask_h = torch.ones(1, N_RES, dtype=torch.bool).pin_memory()
    msa_mask_h = torch.ones(1, N_SEQ, N_RES, dtype=torch.bool).pin_memory()
    out_h = torch.empty(1, N_RES, N_RES, 37, dtype=torch.float32).pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in (seq_h, msa_h, mask_h, msa_mask_h))
    d2h = out_h.numel() * out_h.element_size()

    # trunk inputs resident in HBM (built by the model's own glue, alphafold2.py:676-726)
    with torch.no_grad():
        seq, msa, mask, msa_mask = (t.to(dev) for t in (seq_h, msa_h, mask_h, msa_mask_h))
        e = model.token_emb(seq)
        m0 = model.token_emb(msa) + e[:, None]
        l, r = model.to_pairwise_repr(e).chunk(2, dim=-1)
        idx = torch.arange(N_RES, device=dev)
        rel = (idx[None, :, None] - idx[None, None, :]).clamp(-32, 32) + 32
        x0 = l[:, :, None, :] + r[:, None, :, :] + model.pos_emb(rel)
        x_mask = mask[:, :, None] & mask[:, None, :]
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)

    def trunk_step():
        return model.net(x0, m0, mask=x_mask, msa_mask=msa_mask)

    def e2e_step():
        s_, m_, k_, mk_ = (t.to(dev, non_blocking=True) for t in (seq_h, msa_h, mask_h, msa_mask_h))
        ret = model(s_, m_, mask=k_, msa_mask=mk_)
        out_h.copy_(ret.distance, non_blocking=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        total = 0.0
        barrier()
        for _ in range(steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            last = fn()
            b.record()
            b.synchronize()
            total += a.elapsed_time(b)
        barrier()
        if world > 1:
            t = torch.tensor([total], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total = t.item()
        return total, last   # ms over `steps` steps, max over ranks; what the last step returned

    for _ in range(max(args.warmup, 3)):
        trunk_step()
    e2e_step()
    torch.cuda.synchronize()

    clocks = ClockSampler(local_rank)
    clocks.start()
    l0 = lib.af2_launch_count()
    ms_total, (x_out, m_out) = timed(trunk_step, args.steps)
    launches = int(lib.af2_launch_count() - l0)
    graphed = getattr(model.net, "_af2_graph", None) if world > 1 else None
    if graphed is not None and graphed.graph is not None:
        launches = graphed.launches_per_replay * args.steps      # the sharded forward is replayed as a CUDA graph
    clk = clocks.stop()
    dumps = {}
    if args.dump_outputs and rank == 0:
        # copied before the e2e steps, which run the trunk again
        dumps = {"pair": output_sample(x_out, 1), "msa": output_sample(m_out, 2)}
    ms_e2e, _ = timed(e2e_step, args.steps)
    if args.dump_outputs and rank == 0:
        dumps["distogram"] = output_sample(out_h, 3)
        write_outputs(args.dump_outputs, dumps)

    # secondary, labelled number at N > 1 (SURVEY.md 8e fallback statement): N independent replicas, one unsharded sequence
    # per GPU, all ranks at the same time -- never the headline (`value` is the ONE sequence sharded over all ranks)
    replicas = None
    if world > 1:
        def rep_step():
            return A.Evoformer.forward(model.net, x0, m0, mask=x_mask, msa_mask=msa_mask)
        for _ in range(3):
            rep_step()
        rsteps = max(3, min(args.steps, 5))
        ms_rep = timed(rep_step, rsteps)[0] / rsteps
        replicas = {"value": world * N_RES * N_RES / (ms_rep * 1e-3), "unit": UNIT, "ms_per_step": ms_rep, "scaling": "weak",
                    "what": f"{world} independent sequences, one unsharded trunk forward per GPU, concurrently (secondary number)"}

    ms_step = ms_total / args.steps
    pairs = N_RES * N_RES
    value = pairs / (ms_step * 1e-3)                 # one sequence per step (sharded over all ranks when world > 1)
    e2e_value = pairs / (ms_e2e / args.steps * 1e-3)

    # per-kernel-class device time of 2 more steps (CUDA events around every launch; not part of `value`)
    names = ["gemm_linear(tcgen05)", "gemm_per_channel(tcgen05)", "axial_attention(tcgen05)", "layernorm",
             "channel_to_token", "misc"]
    lib.af2_profile_enable(1)
    prof_steps = 2
    if world > 1:
        import alphafold2_b200.parallel as _par
        _par.GRAPH_ENABLED = False                   # the per-launch event pairs need the eager schedule
    for _ in range(prof_steps):
        trunk_step()
    if world > 1:
        _par.GRAPH_ENABLED = True
    classes = []
    for c, nm in enumerate(names):
        ms, fl, by = C.c_double(), C.c_double(), C.c_double()
        n = lib.af2_profile_read(c, C.byref(ms), C.byref(fl), C.byref(by))
        classes.append(dict(name=nm, launches=int(n), ms=ms.value, flops=fl.value, bytes=by.value))
    lib.af2_profile_enable(0)
    peaks = measured_peaks()
    tot_ms = sum(c["ms"] for c in classes) or 1.0
    dom = max(classes, key=lambda c: c["ms"])
    # DRAM traffic per launch of the dominant class from the committed `ncu --set full` capture of one C2 block
    traffic, traffic_src = None, None
    try:
        import glob
        cand = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")))
        if cand:
            tj = json.load(open(cand[-1]))
            if dom["name"] in tj:
                traffic = tj[dom["name"]]["dram_bytes_per_launch"]
                traffic_src = os.path.relpath(cand[-1], ROOT)
    except Exception:
        pass
    # whole-block DRAM traffic of the committed `ncu --set full` capture of one C2 block, next to SURVEY.md 8(d)'s
    # ideal-fusion minimum (0.69 GB with bf16 activations; ~1.0 GB with the fp32 residual stream kept here)
    block_dram, block_src = None, None
    try:
        import csv
        import glob
        cand = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_block_C2_ncu_full_summary.csv")))
        if cand and N_RES == 256:
            rows = list(csv.DictReader(open(cand[-1])))
            rk = [k for k in rows[0] if k.startswith("dram_read_MB")][0]
            wk = [k for k in rows[0] if k.startswith("dram_write_MB")][0]
            block_dram = sum(float(r[rk]) + float(r[wk]) for r in rows) * 1e6
            block_src = os.path.relpath(cand[-1], ROOT)
    except Exception:
        pass
    if dom["flops"] > 0:
        ach = dom["flops"] / (dom["ms"] * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": dom["name"], "achieved": ach, "peak": peaks["tflops"], "unit": "TFLOP/s",
                "frac": ach / peaks["tflops"], "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": dom["bytes"] / max(dom["launches"], 1),
                "peak_source": peaks["source"] + ", sustained bf16",
                "share_of_step": dom["ms"] / tot_ms, "avg_launch_ms": dom["ms"] / max(dom["launches"], 1),
                "flops_per_launch": dom["flops"] / max(dom["launches"], 1)}
    else:
        ach = dom["bytes"] / (dom["ms"] * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": dom["name"], "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": ach / peaks["hbm_gbs"], "traffic": traffic, "traffic_source": traffic_src, "peak_source": peaks["source"],
                "share_of_step": dom["ms"] / tot_ms, "avg_launch_ms": dom["ms"] / max(dom["launches"], 1)}
    step_flops = flops_per_block(N_RES, N_SEQ, CFG["dim"], CFG["heads"], CFG["dim_head"]) * CFG["depth"]
    step_tf = step_flops / (ms_step * 1e-3) / 1e12

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_step, "ms_per_block": ms_step / CFG["depth"], "higher_is_better": True,
        "scaling": "weak" if world == 1 else "strong",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": make_config(world),
        "schedule": ("eager" if world == 1 else ("CUDA graph replay per rank" if (graphed is not None and graphed.graph is not None) else "eager")),
        "clocks": clk,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches,
        "replicas": replicas,
        "collectives_per_block": (None if world == 1 else {"all_gather_small_bias": 3, "all_gather_operand": 3, "all_to_all_msa": 2, "all_to_all_pair": 4}),
        "exchange": (None if world == 1 else exchange_transport()),
        "roofline": roof,
        "roofline_whole_step": {"bound": "tensor", "achieved": step_tf, "peak": peaks["tflops"], "unit": "TFLOP/s",
                                "frac": step_tf / peaks["tflops"], "frac_of_burst_peak": step_tf / peaks["tflops_burst"],
                                "flops_per_step": step_flops, "block_dram_bytes": block_dram,
                                "block_dram_bytes_source": block_src, "block_algorithmic_min_bytes": 0.69e9 if N_RES == 256 else None,
                                "block_dram_over_min": (block_dram / 0.69e9) if block_dram else None},
        "kernel_classes": [dict(name=c["name"], launches_per_step=c["launches"] // prof_steps,
                                ms_per_step=c["ms"] / prof_steps, share=c["ms"] / tot_ms,
                                tflops=(c["flops"] / (c["ms"] * 1e-3) / 1e12 if c["ms"] > 0 else 0.0),
                                gbs=(c["bytes"] / (c["ms"] * 1e-3) / 1e9 if c["ms"] > 0 else 0.0)) for c in classes],
    }
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            try:
                out["cpu_baseline"] = cpu_baseline()
            except Exception as ex:  # noqa
                out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                                       "sample": f"failed: {ex}"}
            try:
                out["gpu_torch_baseline"] = gpu_torch_baseline(dev, x0, m0, x_mask, msa_mask, model)
            except Exception as ex:  # noqa
                out["gpu_torch_baseline"] = {"error": repr(ex)[:300]}
        print(json.dumps(out), flush=True)
    if world > 1:
        from alphafold2_b200.parallel import release_graphs
        release_graphs(model)          # a live CUDA graph with NCCL nodes must not outlive the process group


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="C2", choices=list(WORKLOADS),
                    help="BASELINE.json config shape (default C2 = the configuration the metric is quoted on)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32): pair.npy and "
                         "msa.npy from the trunk, distogram.npy from Alphafold2.forward; an array of more than "
                         f"{DUMP_ELEMS} elements is replaced by that many of its elements at fixed seeded flat indices")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    set_workload(args.workload)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
