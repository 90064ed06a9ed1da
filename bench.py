#!/usr/bin/env python
"""bench.py -- atom-steps/s (energy + forces) of the NequIP hot path on B200.

  python bench.py --gpus N --steps K --warmup W            (own arm: sm_100a kernels)
  python bench.py --impl reference --gpus N --steps K ...  (reference arm: the e3nn-formulation
                                                            CPU path = oracle port, all host threads,
                                                            bounded sample of the same workload)

A "step" is one energy+forces evaluation (forward + autograd backward w.r.t. positions) of the
BASELINE.json configs[2] model -- NequIP l_max=2, 4 layers, 64 features, parity, radial MLP 1x128,
r_max 5 A -- on a synthetic ~10k-atom Li3PO4-like periodic box (10 648 atoms, ~589k edges).
`value`  : device-resident inputs, CUDA-event timed, max over ranks.
`e2e`    : the same step through NequIPEnergyModel.forward with HOST (pinned) inputs: H2D of
           pos/edge_index/shifts/types/cell and D2H of forces+energy inside the timed region.
`e2e_device_neighbor_list`: as `e2e`, but only positions travel and the neighbour list is built on the GPU.
`roofline`: every hot kernel class of every layer timed ALONE (CUDA events on the launching stream, step-sized
           inputs > L2); the class with the largest share of the step is the headline, the rest is under
           `roofline.by_kernel` (HBM fraction of the measured copy peak; for the tcgen05 GEMMs also the 3xTF32
           issue rate against half the measured bf16 cuBLAS rate, and the ncu tensor-pipe activity).
N > 1 (default): ONE frame partitioned by atoms into N bricks with halo (ghost) atoms -- the north_star
partition: per-layer NCCL halo exchange of ghost features, energy all-reduce, ghost-force reduction to the
owners; the whole sharded step is one CUDA-graph replay per rank.  `--scaling weak` (default) grows the frame
with N (the N-fold periodic supercell of the N = 1 frame along x: N x 10 648 atoms), `--scaling strong` splits the
10 648-atom frame.  `checks`: sum of all forces = 0, and in halo mode `partition_parity` = forces / energy of the
sharded frame against the UNSHARDED base frame evaluated on each rank (every atom is a periodic copy of a base atom).
`--decomp frames` keeps the round-1 mode (one independent frame per GPU, the reference's DDP axis).
`--dump-outputs DIR`: after the timed steps, the floating-point outputs of the last timed step (total_energy, forces;
the reference arm also atomic_energy) are written as DIR/<name>.npy (float32 / float64; `.rank<r>` before `.npy` when
N > 1).  Inputs and weights are seeded, so two builds run with the same arguments can be compared output for output.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # name: (structure kind, n_side, model kwargs)
    "li3po4_10k_l2_f64": ("li3po4", 22, dict(l_max=2, num_layers=4, num_features=64, radial_mlp_depth=1, radial_mlp_width=128)),
    "water_1k_l2_f32": ("water", 10, dict(l_max=2, num_layers=4, num_features=32, radial_mlp_depth=1, radial_mlp_width=128)),
    "asi_50k_l3_f32": ("asi", 37, dict(l_max=3, num_layers=5, num_features=32, radial_mlp_depth=1, radial_mlp_width=128)),
    "tiny": ("water", 5, dict(l_max=2, num_layers=3, num_features=8, radial_mlp_depth=1, radial_mlp_width=16)),
}
# CPU arms: the sample is a smaller box of the SAME structure kind, density, r_max and model (atom-steps/s is
# per atom, the neighbour count per atom is the same); its size is chosen from a measured per-atom cost so that
# the whole CPU run stays within CPU_BUDGET_S -- at least 1000 atoms whenever that fits.
CPU_SAMPLE_NSIDE_MAX = {"li3po4_10k_l2_f64": 10, "water_1k_l2_f32": 10, "asi_50k_l3_f32": 11, "tiny": 4}
CPU_SAMPLE_NSIDE_MIN = {"li3po4_10k_l2_f64": 6, "water_1k_l2_f32": 6, "asi_50k_l3_f32": 7, "tiny": 4}
CPU_BUDGET_S = 200.0      # cpu_baseline leg of the own arm (3 steps)
REF_ARM_BUDGET_S = 300.0  # --impl reference: all of its --steps + --warmup steps ("a few minutes")
R_MAX = 5.0


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": (sm[len(sm) // 2] if sm else None), "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def tp_algorithmic_bytes(sig, N, E, elem=4, backward=False):
    """SURVEY.md section 8(d): forward reads x, edge_attr, edge_weight, two int64 index arrays, writes out."""
    b = elem * (N * sig.d_in + E * sig.s_dim + E * sig.weight_numel + N * sig.d_out) + 16 * E
    if backward:
        b = elem * (N * sig.d_out + N * sig.d_in + E * sig.s_dim + 2 * E * sig.weight_numel + E * sig.s_dim
                    + N * sig.d_in) + 16 * E
    return b


def build_system(workload, seed, n_side=None):
    from nequip_b200 import data as D

    kind, ns, mk = WORKLOADS[workload]
    sysd = D.make_system(kind, n_side or ns, r_max=R_MAX, seed=seed)
    meta = sysd.pop("_meta")
    return sysd, meta, mk


def build_partitioned_frame(workload, world, scaling):
    """The ONE frame that ``world`` ranks share in halo mode, built from the N = 1 workload frame (seed 0):
    ``weak``  : its ``world``-fold periodic supercell along x (world x the atoms, box elongated along x);
    ``strong``: the frame itself.
    Either way every atom of the partitioned frame is a periodic copy of a base-frame atom, so the energies and forces
    of the sharded computation must equal those of the UNSHARDED base frame (tiled) -- checked on the hardware after
    the timed region (``checks.partition_parity``).  Returns (full frame, base frame, meta, model kwargs, copies)."""
    from nequip_b200 import data as D

    base, meta, mk = build_system(workload, seed=0)
    copies = world if scaling == "weak" else 1
    full = D.replicate_frame(base, copies, r_max=R_MAX, axis=0) if copies > 1 else dict(base)
    return full, base, meta, mk, copies


def pick_threads(workload):
    """Thread count for the CPU arm: torch's intra-op pool oversubscribes badly on many-core hosts (128
    threads were 12x slower than 8 on the first GPU box), so time one small step at a few counts and keep
    the fastest.  Returns (threads, {count: seconds})."""
    from nequip_b200.nn.model import NequIPEnergyModel
    from oracle import model as omodel

    cores = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores})
    sysd, meta, mk = build_system(workload, seed=0, n_side=5)
    model = NequIPEnergyModel(r_max=R_MAX, type_names=meta["type_names"], parity=True,
                              avg_num_neighbors=meta["avg_num_neighbors"], **mk)
    sd, cfg = model.state_dict(), model.config
    times = {}
    for c in cands:
        torch.set_num_threads(c)
        omodel.energy_and_forces(sd, cfg, sysd, torch.float32, tp_chunk=20000)
        t0 = time.perf_counter()
        omodel.energy_and_forces(sd, cfg, sysd, torch.float32, tp_chunk=20000)
        times[c] = time.perf_counter() - t0
    best = min(times, key=times.get)
    torch.set_num_threads(best)
    return best, times, times[best] / sysd["pos"].shape[0]


def pick_sample_nside(workload, sec_per_atom, nsteps, budget_s=None):
    """Largest box (n_side^3 atoms) whose ``nsteps`` CPU steps fit the budget at the measured per-atom cost."""
    budget_s = CPU_BUDGET_S if budget_s is None else budget_s
    lo, hi = CPU_SAMPLE_NSIDE_MIN[workload], CPU_SAMPLE_NSIDE_MAX[workload]
    ns = lo
    for n in range(lo, hi + 1):
        if nsteps * sec_per_atom * n ** 3 <= budget_s:
            ns = n
    return ns


def run_reference(args, rank, world):
    """Reference arm: the reference's own (e3nn-formulation) CPU implementation of the path -- the
    oracle port -- with all host threads, on a bounded sample of the workload."""
    if rank != 0:
        return
    from nequip_b200.nn.model import NequIPEnergyModel
    from oracle import model as omodel

    cores, _, spa = pick_threads(args.workload)
    ns = pick_sample_nside(args.workload, spa, args.steps + args.warmup, budget_s=REF_ARM_BUDGET_S)
    sysd, meta, mk = build_system(args.workload, seed=0, n_side=ns)
    model = NequIPEnergyModel(r_max=R_MAX, type_names=meta["type_names"], parity=True,
                              avg_num_neighbors=meta["avg_num_neighbors"], **mk)
    sd, cfg = model.state_dict(), model.config
    n_atoms = sysd["pos"].shape[0]
    chunk = 20000
    for _ in range(args.warmup):
        omodel.energy_and_forces(sd, cfg, sysd, torch.float32, tp_chunk=chunk)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e, ea, f = omodel.energy_and_forces(sd, cfg, sysd, torch.float32, tp_chunk=chunk)
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        dump_outputs(output_arrays({"total_energy": e, "atomic_energy": ea, "forces": f}), args.dump_outputs)
    val = n_atoms / dt
    sample = (f"{n_atoms}-atom {WORKLOADS[args.workload][0]} box, same model/density, E={sysd['edge_index'].shape[1]}, "
              f"edge chunk {chunk}, {cores} of {os.cpu_count()} host threads (fastest of a short sweep)")
    line = {
        "impl": "reference", "metric": "atom-steps/sec (energy+forces)", "value": val, "unit": "atom-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # the own arm's workload and model keys; what was actually evaluated per step is `cpu_baseline.sample`
        "config": {"workload": args.workload, "r_max": R_MAX, "parity": True, **mk,
                   "atoms_per_step_sample": n_atoms, "edges_per_step_sample": int(sysd["edge_index"].shape[1]),
                   "note": ("CPU e3nn-formulation path (oracle port) on a bounded sample of the workload: a smaller box of "
                            "the same structure kind, density, r_max and model (atom-steps/s is per atom)")},
        "cpu_baseline": {"value": val, "unit": "atom-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "atom-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def cpu_baseline(workload):
    from nequip_b200.nn.model import NequIPEnergyModel
    from oracle import model as omodel

    cores, _, spa = pick_threads(workload)
    ns = pick_sample_nside(workload, spa, 3)  # one warm-up + two timed steps
    sysd, meta, mk = build_system(workload, seed=0, n_side=ns)
    model = NequIPEnergyModel(r_max=R_MAX, type_names=meta["type_names"], parity=True,
                              avg_num_neighbors=meta["avg_num_neighbors"], **mk)
    sd, cfg = model.state_dict(), model.config
    n_atoms = sysd["pos"].shape[0]
    omodel.energy_and_forces(sd, cfg, sysd, torch.float32, tp_chunk=20000)
    t0 = time.perf_counter()
    reps = 0
    while reps < 2:
        omodel.energy_and_forces(sd, cfg, sysd, torch.float32, tp_chunk=20000)
        reps += 1
    dt = (time.perf_counter() - t0) / reps
    return {"value": n_atoms / dt, "unit": "atom-steps/s", "cores": cores, "kind": "port",
            "sample": (f"{n_atoms}-atom {WORKLOADS[workload][0]} box (same model, density, r_max), {reps} steps, "
                       f"E={sysd['edge_index'].shape[1]}, {cores} of {os.cpu_count()} host threads (fastest of a short sweep)")}


def ncu_summary(kernel, field):
    """A per-launch metric of ``kernel`` from the committed ``ncu --set full`` summaries of this round
    (profiles/r02_ncu_full_summary.json; falls back to round 1's), or None."""
    for name in ("r02_ncu_full_summary.json", "r01_ncu_full_summary.json"):
        try:
            rows = json.load(open(os.path.join(ROOT, "profiles", name)))[kernel]
            r = max(rows, key=lambda x: x["ms"])
            if field == "traffic":
                return int(round((r["dram_read_GB"] + r["dram_write_GB"]) * 1e9))
            return r.get(field)
        except Exception:
            continue
    return None


def force_sum_vector(forces):
    """[sum Fx, sum Fy, sum Fz, sum |F|, 1] (float64) of one rank's forces -- summed over the ranks this is the
    size-independent parity property of the step: the forces of a periodic frame add up to zero (Newton's third law),
    and under the halo partition they only do if every ghost contribution reached its owner."""
    f = forces.detach().double().reshape(-1, 3)
    v = torch.zeros(5, dtype=torch.float64, device=f.device)
    v[:3] = f.sum(0)
    v[3] = f.abs().sum()
    v[4] = 1.0
    return v


def parity_checks(step, unsharded_model, base_frame, copies, owned_ids, halo_mode, world, rank, dev):
    """Parity properties of the step that was timed, evaluated on the hardware and at the size of the run.

    ``step()`` is the timed step (in halo mode it contains collectives: it is called unconditionally by every rank);
    everything inside the try blocks is rank-local, so a failure there is reported on stderr but can never
    desynchronise the ranks, and every collective below is entered by every rank.
    (1) Newton's third law: the forces of all atoms, over all ranks, add up to zero.
    (2) halo mode: the partitioned frame is the ``copies``-fold periodic supercell of ``base_frame`` (or the base frame
        itself), so owned atom g must carry the force of base atom ``g % n_base`` in the UNSHARDED call
        ``unsharded_model(base_frame)`` (eager, same weights and kernels, evaluated on each rank), and the total energy
        must be ``copies`` times the base frame's."""
    import torch.distributed as dist

    last = step()
    f_last = last["forces"].detach().clone()
    e_last = last["total_energy"].detach().double().reshape(-1)[:1].clone()
    chk = torch.zeros(5, dtype=torch.float64, device=dev)
    try:
        chk = force_sum_vector(f_last).to(dev)
    except Exception as exc:
        print(f"[bench rank {rank}] force-sum check failed: {type(exc).__name__}: {exc}", file=sys.stderr, flush=True)
        chk = torch.zeros(5, dtype=torch.float64, device=dev)
    par = torch.zeros(4, dtype=torch.float64, device=dev)  # max|dF|, max|F_base|, |dE| / (copies sum|E_i|), rank ok
    n_base = 0
    if halo_mode:
        try:
            n_base = int(base_frame["pos"].shape[0])
            ref = unsharded_model(base_frame)
            idx = (owned_ids % n_base).to(f_last.device)
            par[0] = (f_last - ref["forces"][idx]).abs().max()
            par[1] = ref["forces"].abs().max()
            par[2] = (e_last - copies * ref["total_energy"].detach().double().reshape(-1)[:1]).abs().max() / (
                copies * ref["atomic_energy"].detach().double().abs().sum())
            par[3] = 1.0
            del ref
        except Exception as exc:
            print(f"[bench rank {rank}] partition-parity check failed: {type(exc).__name__}: {exc}", file=sys.stderr, flush=True)
            par = torch.zeros(4, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(chk)
        ok_ranks = par[3:4].clone()
        dist.all_reduce(par, op=dist.ReduceOp.MAX)
        dist.all_reduce(ok_ranks)
        par[3] = ok_ranks[0]
    chk, par = chk.tolist(), par.tolist()

    def num(x):  # a NaN / inf must not make the JSON line unparsable
        return x if (x is None or math.isfinite(x)) else repr(x)

    checks = {"sum_forces_over_sum_abs_forces": num(math.sqrt(chk[0] ** 2 + chk[1] ** 2 + chk[2] ** 2) / chk[3]) if chk[3] > 0 else None,
              "ranks_reporting": int(round(chk[4])),
              "note": "Newton's third law over the whole frame (all ranks): a lost or doubled ghost contribution shows as ~1e-2"}
    if halo_mode:
        checks["partition_parity"] = {
            "max_dF_over_max_F": num(par[0] / par[1]) if par[1] > 0 else None,
            "dE_over_sum_abs_Ei": num(par[2]) if par[3] > 0 else None,
            "ranks_reporting": int(round(par[3])),
            "what": (f"forces of every owned atom and the total energy of the frame sharded over {world} ranks vs the "
                     f"UNSHARDED {n_base}-atom base frame evaluated eagerly on each rank (the sharded frame is its "
                     f"{copies}-fold periodic supercell); max over ranks, fp32 kernels: expect <= 1e-5")}
    return checks


def halo_exchange_profile(dims, plan, halo, dev, world, reps=10):
    """The data-path collective of the halo mode, timed alone: for every interaction layer >= 1 the forward exchange
    (owned rows -> owned + ghost rows: index_select, all_to_all_single with split sizes into the tail of the feature
    buffer) and forward + transposed backward (ghost gradients added into their owners), with feature rows of the
    layer's width.  Every rank runs the same sequence of collectives; times are the max over ranks."""
    import torch.distributed as dist

    cuda = torch.device(dev).type == "cuda"

    def sync():
        if cuda:
            torch.cuda.synchronize()

    def timeit(fn):
        fn()
        sync()
        if world > 1:
            dist.barrier()
        if cuda:  # device time (CUDA events on the launching stream)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            sync()
            return e0.elapsed_time(e1) / reps
        t0 = time.perf_counter()  # CPU / gloo (tests)
        for _ in range(reps):
            fn()
        return (time.perf_counter() - t0) / reps * 1e3

    out = []
    for li, d in dims:
        x = torch.randn(plan.n_own, d, device=dev, dtype=torch.float32)
        gy = torch.randn(plan.n_own + plan.n_ghost, d, device=dev, dtype=torch.float32)

        def fwd():
            return halo(x)

        def fwd_bwd():
            xr = x.detach().requires_grad_(True)
            halo(xr).backward(gy)

        t = torch.tensor([timeit(fwd), timeit(fwd_bwd)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t = t.tolist()
        out.append({"layer": li, "row_floats": d, "rows_sent": int(sum(plan.send_splits)), "rows_received": int(plan.n_ghost),
                    "bytes_sent_per_exchange": int(sum(plan.send_splits)) * d * 4,
                    "ms_forward": t[0], "ms_forward_plus_backward": t[1]})
    return out


DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def output_arrays(out, exclude=()):
    """Host copies of the floating-point tensors of one step's result dict (keys in ``exclude``, the step's inputs,
    are skipped), as float32 / float64 numpy arrays."""
    arrs = {}
    for k, v in out.items():
        if k in exclude or not torch.is_tensor(v) or not v.is_floating_point():
            continue
        v = v.detach()
        if v.dtype not in (torch.float32, torch.float64):
            v = v.float()
        arrs[k] = v.cpu().numpy().copy()
    return arrs


def dump_outputs(arrs, out_dir, suffix=""):
    """``out_dir/<name><suffix>.npy`` for every array, DUMP_LIMIT_BYTES in all: an array over its share of the limit
    is replaced by a fixed seeded sample of its flattened elements, with their flat positions (float64) in
    ``<name><suffix>.index.npy``."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_LIMIT_BYTES // max(1, len(arrs))
    for name, a in sorted(arrs.items()):
        if a.nbytes > share:
            flat = a.reshape(-1)
            keep = share // (a.itemsize + 8)
            idx = np.sort(np.random.default_rng(0).choice(flat.size, keep, replace=False))
            np.save(os.path.join(out_dir, f"{name}{suffix}.index.npy"), idx.astype(np.float64))
            a = flat[idx]
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


def _time_cuda(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_rooflines(model, resident, n_atoms, n_edges, reps, ms_step, dev):
    """Isolated timing of the hot kernels of every interaction layer with the step's shapes.

    Algorithmic bytes (SURVEY.md section 8d / DESIGN.md section 4): TP forward  4 (N D_in + E S + E W + N D_mid) + 16 E,
    TP backward 4 (N D_mid + 2 N D_in + 2 E S + 2 E W) + 16 E, radial GEMM 4 E (K + W) + 4 K W; the fused forward
    kernel reads 4 (N D_in + E S + E K) + 16 E + weights and writes 4 N D_mid (+ 4 E W when the weights are kept for
    the backward).  Tensor work of the 3xTF32 GEMMs: 3 x 2 E K W flop."""
    from nequip_b200 import ops
    from nequip_b200.nn import dense
    from nequip_b200.nn.model import ScalarLinearLayer

    peak_hbm, peak_src = load_peaks()
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        tf32_peak = float(pk["bf16_tflops_sustained"]) / 2.0  # no TF32 measurement exists: half the measured bf16 rate
        tf32_src = "estimated: measured sustained bf16 cuBLAS rate / 2"
    except Exception:
        tf32_peak, tf32_src = 1590.0 / 2.0, "estimated: fallback bf16 rate / 2"
    N, E = n_atoms, n_edges
    ei = resident["edge_index"]
    csr = ops.build_csr(ei[0].contiguous(), N)
    src = ei[1].contiguous()
    g = torch.Generator(device=dev).manual_seed(0)
    classes = {}

    def add(cls, entry):
        c = classes.setdefault(cls, {"ms_per_step": 0.0, "launches_per_step": 0, "largest": None})
        c["ms_per_step"] += entry["ms_per_launch"]
        c["launches_per_step"] += 1
        if c["largest"] is None or entry["ms_per_launch"] > c["largest"]["ms_per_launch"]:
            c["largest"] = entry

    def hbm_entry(kernel, ms, alg, layer, extra=None):
        ach = alg / (ms * 1e-3) / 1e9
        d = {"kernel": kernel, "layer": layer, "bound": "hbm", "achieved": ach, "peak": peak_hbm, "unit": "GB/s",
             "frac": ach / peak_hbm, "alg_bytes_per_launch": alg, "ms_per_launch": ms}
        if extra:
            d.update(extra)
        return d

    with torch.no_grad():
        for li, layer in enumerate(model.layers):
            conv = layer.conv
            plan = conv.tp_scatter._plan
            sig = plan.sig
            W, K = sig.weight_numel, 128
            lins = [m for m in conv.edge_mlp.mlp if isinstance(m, ScalarLinearLayer)]
            if len(lins) != 2 or not dense.RadialMLPGemm.supported(lins[0], lins[1], torch.float32):
                continue
            K = lins[1].weight.shape[0]
            x = torch.randn(N, sig.d_in, device=dev, generator=g)
            y = torch.randn(E, sig.s_dim, device=dev, generator=g)
            emb = torch.rand(E, lins[0].weight.shape[0], device=dev, generator=g)
            go = torch.randn(N, sig.d_out, device=dev, generator=g)
            mlp = dense.RadialMLPGemm(lins[0], lins[1], dev)
            h = torch.nn.functional.silu(emb @ mlp.w1s)
            w = torch.empty(E, W, device=dev)
            gh = torch.empty(E, K, device=dev)
            flops3 = 3 * 2.0 * E * K * W
            if emb.shape[1] == 8 and K == 128:  # the CUDA-core hidden layer (k_hidden_fwd / k_hidden_bwd), both directions
                gemb = torch.empty_like(emb)
                ms = _time_cuda(lambda: ops.mlp_hidden_fwd(emb, mlp.w1s, h, None), reps)
                add("k_hidden_fwd", hbm_entry("k_hidden_fwd (radial MLP first layer + SiLU, CUDA cores)", ms, 4 * E * (8 + K), li))
                ms = _time_cuda(lambda: ops.mlp_hidden_bwd(emb, mlp.w1s, h, gemb), reps)
                add("k_hidden_bwd", hbm_entry("k_hidden_bwd (its backward, pre-activation recomputed)", ms, 4 * E * (8 + K + 8), li))
            tc = conv._tc_cache[1] if conv._tc_cache else None
            fused = tc["fused"] if (tc and tc["fused"] is not None and (conv.use_fused_radial_tp is True or conv._fused_choice)) else None
            if fused is not None:
                ms = _time_cuda(lambda: ops.tp_fused_fwd(fused.fw, x, y, h, src, csr, want_w=True), reps)
                alg = 4 * (N * sig.d_in + E * sig.s_dim + E * K + N * sig.d_out + E * W) + 16 * E + 8 * K * W
                tfl = flops3 / (ms * 1e-3) / 1e12
                add("tp_fused_fwd_kernel", hbm_entry("tp_fused_fwd_kernel (radial GEMM + TP + scatter, tcgen05 + FFMA2)", ms, alg, li, {
                    "tensor": {"achieved": tfl, "peak": tf32_peak, "unit": "TFLOP/s (3xTF32 issue)", "frac": tfl / tf32_peak,
                               "peak_source": tf32_src}}))
            else:
                ms = _time_cuda(lambda: mlp.fwd.run(h, w, E), reps)
                alg = 4 * E * (K + W) + 8 * K * W
                tfl = flops3 / (ms * 1e-3) / 1e12
                add("k_gemm3x", hbm_entry("k_gemm3x (radial MLP last layer forward, tcgen05 3xTF32)", ms, alg, li, {
                    "tensor": {"achieved": tfl, "peak": tf32_peak, "unit": "TFLOP/s (3xTF32 issue)", "frac": tfl / tf32_peak,
                               "peak_source": tf32_src,
                               "pipe_tensor_cycles_active_pct": ncu_summary("k_gemm3x", "pipe_tensor_pct")}}))
                ms = _time_cuda(lambda: ops.tp_scatter(plan, x, y, w, ei[0], src, csr=csr), reps)
                name = "tp_fwd2_kernel" if TPGen(sig, plan.opts).ring_fwd() else "tp_fwd_kernel<float>"
                add(name, hbm_entry(name + " (fused TP + scatter forward)", ms, tp_algorithmic_bytes(sig, N, E), li))
            # backward: TP + scatter, then the radial GEMM for grad_h
            ms = _time_cuda(lambda: ops.tp_scatter_bwd_raw(plan, x, y, w, src, csr, go, need_x=(li != 0)), reps)
            name = "tp_bwd2_kernel" if TPGen(sig, plan.opts).ring_bwd() else "tp_bwd_kernel<float>"
            add(name, hbm_entry(name + " (fused TP + scatter backward; incl. the zero fills of grad_x / grad_Y)", ms,
                                tp_algorithmic_bytes(sig, N, E, backward=True), li,
                                {"fma": {"note": "FP32-FMA bound for l_max >= 2 layers", "mults_per_edge_channel_fwd": sig.fma_count()}}))
            ms = _time_cuda(lambda: mlp.bwd.run(w, gh, E), reps)
            alg = 4 * E * (K + W) + 8 * K * W
            tfl = flops3 / (ms * 1e-3) / 1e12
            add("k_gemm3x", hbm_entry("k_gemm3x (radial MLP last layer backward, K = W)", ms, alg, li, {
                "tensor": {"achieved": tfl, "peak": tf32_peak, "unit": "TFLOP/s (3xTF32 issue)", "frac": tfl / tf32_peak,
                           "peak_source": tf32_src,
                           "pipe_tensor_cycles_active_pct": ncu_summary("k_gemm3x", "pipe_tensor_pct")}}))
            del x, y, emb, go, h, w, gh
    for k, c in classes.items():
        c["share_of_step"] = c["ms_per_step"] / ms_step
    top_name = max(classes, key=lambda k: classes[k]["ms_per_step"])
    top = dict(classes[top_name]["largest"])
    top["traffic"] = ncu_summary(top_name.split("<")[0], "traffic")
    top["peak_source"] = peak_src
    top["share_of_step"] = classes[top_name]["share_of_step"]
    top["selection"] = ("kernel class with the largest summed isolated time over the layers of one step; numbers are for "
                        "its largest launch")
    top["inputs"] = "per-edge operands of the step's size (>> 126 MB L2)"
    top["by_kernel"] = {k: {"ms_per_step_isolated": c["ms_per_step"], "share_of_step": c["share_of_step"],
                            "launches_per_step": c["launches_per_step"],
                            "traffic": ncu_summary(k.split("<")[0], "traffic"), **c["largest"]}
                        for k, c in sorted(classes.items(), key=lambda kv: -kv[1]["ms_per_step"])}
    return top


class TPGen:
    """Which forward / backward kernel variant the generator picked for a signature."""

    def __init__(self, sig, opts):
        from nequip_b200.codegen import TPGenerator

        self.g = TPGenerator(sig, opts)
        self.g.source()

    def ring_fwd(self):
        return bool(self.g.use_ring)

    def ring_bwd(self):
        return bool(self.g.use_ring_bwd)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="li3po4_10k_l2_f64", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--decomp", default="halo", choices=["frames", "halo"],
                    help="N>1: 'halo' (default) = ONE frame partitioned by atoms into N bricks with halo (ghost) atoms, "
                         "per-layer NCCL halo exchange, energy all-reduce, ghost forces returned to their owners -- the "
                         "north_star partition; 'frames' = one independent frame per GPU (the reference's DDP axis)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="halo mode: 'weak' = the frame grows with N (the N-fold periodic supercell of the workload's frame "
                         "along x); 'strong' = the workload's own frame split N ways")
    ap.add_argument("--no-graph", action="store_true", help="eager step (no CUDA-graph replay)")
    ap.add_argument("--profile-step", action="store_true",
                    help="run one warm-up step, then ONE step between cudaProfilerStart/Stop (for ncu "
                         "--profile-from-start off); prints no bench line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the floating-point outputs of the last timed step as DIR/<name>.npy (float32/float64, "
                         "at most 64 MB in all; a larger output is replaced by a fixed seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist

    from nequip_b200 import _capi, ops
    from nequip_b200 import data as D
    from nequip_b200.nn.model import NequIPEnergyModel

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl b200) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False

    halo_mode = world > 1 and args.decomp == "halo"
    base_frame, copies = None, 1
    if halo_mode:
        from nequip_b200 import parallel as P

        full, base_frame, meta, mk, copies = build_partitioned_frame(args.workload, world, args.scaling)
        lengths = torch.diagonal(full["cell"]).tolist()
        grid = P.brick_grid(world, lengths, halo=R_MAX)
        owner = P.brick_owner(full["pos"], grid)
        plan = P.make_plans(full["edge_index"], owner, world)[rank]
        sysd = P.shard_data(full, plan)
        n_total_atoms = full["pos"].shape[0]
        del full
    else:
        # every rank owns its own frame (same size/density, different seed)
        sysd, meta, mk = build_system(args.workload, seed=rank)
    n_atoms, n_edges = sysd["pos"].shape[0], sysd["edge_index"].shape[1]
    model = NequIPEnergyModel(r_max=R_MAX, type_names=meta["type_names"], parity=True,
                              avg_num_neighbors=meta["avg_num_neighbors"], **mk).to(dev)
    for p in model.parameters():
        p.requires_grad_(False)  # inference: forces only need d/dpos

    host = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in sysd.items()}
    resident = D.to_device(sysd, dev)
    e_buf = torch.zeros(1, dtype=torch.float64, device=dev)

    if halo_mode:
        halo = P.HaloExchange(plan, dev)
    for layer in model.layers:
        layer.conv.strict_fast_path = True  # a torch.matmul fallback of a dense block must not be timed silently

    graphed, graph_error = None, None
    if not args.no_graph:
        from nequip_b200.graph import GraphedEnergyForces, GraphedShardedEnergyForces

        try:
            if halo_mode:  # the sharded step incl. its NCCL exchanges as one graph per rank
                graphed = GraphedShardedEnergyForces(model, resident, plan, halo)
            else:
                graphed = GraphedEnergyForces(model, resident)  # captured once; replayed every step
        except Exception as exc:  # e.g. a driver / NCCL build that cannot capture: time the eager step, and say so
            graphed, graph_error = None, f"{type(exc).__name__}: {exc}"[:300]
            print(f"[bench rank {rank}] CUDA-graph capture failed, falling back to eager launches: {graph_error}",
                  file=sys.stderr, flush=True)
        if world > 1:  # either every rank replays a graph or none does (the collectives must match)
            ok = torch.tensor([1 if graphed is not None else 0], dtype=torch.int32, device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0:
                graphed = None
                graph_error = graph_error or "capture failed on another rank"

    def step_resident():
        if graphed is not None:
            out = graphed.replay()
            if world > 1 and not halo_mode:
                e_buf.copy_(out["total_energy"].view(-1))
                dist.all_reduce(e_buf)
            return out
        if halo_mode:
            e, f = P.sharded_energy_forces(model, resident, plan, halo, reduce_forces="owner")
            return {"total_energy": e, "forces": f}
        out = model(resident)
        if world > 1:
            e_buf.copy_(out["total_energy"].view(-1))
            dist.all_reduce(e_buf)
        return out

    f_host = torch.empty((plan.n_own if halo_mode else n_atoms, 3), dtype=torch.float64).pin_memory()
    e_host = torch.empty((1,), dtype=torch.float64).pin_memory()

    def step_e2e():
        if graphed is not None:
            out = graphed(host)  # pinned host -> static device buffers (H2D) -> replay
            if world > 1 and not halo_mode:
                e_buf.copy_(out["total_energy"].view(-1))
                dist.all_reduce(e_buf)
            f_host.copy_(out["forces"], non_blocking=True)
            e_host.copy_(out["total_energy"].view(-1), non_blocking=True)
            return out
        d = {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) else v) for k, v in host.items()}
        if halo_mode:
            e, f = P.sharded_energy_forces(model, d, plan, halo, reduce_forces="owner")
            out = {"total_energy": e, "forces": f}
        else:
            out = model(d)
        if world > 1 and not halo_mode:
            e_buf.copy_(out["total_energy"].view(-1))
            dist.all_reduce(e_buf)
        f_host.copy_(out["forces"], non_blocking=True)
        e_host.copy_(out["total_energy"].view(-1), non_blocking=True)
        return out

    def step_e2e_device_nl():
        """Host positions in, forces out, with the neighbour list built ON THE DEVICE (ops.neighbor_list, SURVEY 8f-2):
        the host ships 24 bytes per atom instead of ~40 bytes per edge."""
        pos_d = host["pos"].to(dev, non_blocking=True)
        nl = ops.neighbor_list(pos_d, sysd["cell"], True, R_MAX)
        if graphed is not None and tuple(nl["edge_index"].shape) == tuple(graphed.static["edge_index"].shape):
            graphed.static["pos"].copy_(pos_d)
            graphed.static["edge_index"].copy_(nl["edge_index"])
            graphed.static["edge_cell_shift"].copy_(nl["edge_cell_shift"])
            out = graphed.replay()
        else:
            d = dict(resident)
            d.update(pos=pos_d, edge_index=nl["edge_index"], edge_cell_shift=nl["edge_cell_shift"])
            out = model(d)
        f_host.copy_(out["forces"], non_blocking=True)
        e_host.copy_(out["total_energy"].view(-1), non_blocking=True)
        return out

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = _capi.launch_count()
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1) / steps
        launches = _capi.launch_count() - n0
        if graphed is not None:
            launches += graphed.launches_per_replay * steps  # kernels inside the replayed graph
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches, out

    if args.profile_step:
        step_resident()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStart()
        step_resident()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
        return

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_res, launches, last = timed(step_resident, args.steps, args.warmup)
    if args.dump_outputs:  # host copies now: the replays of the e2e legs below overwrite the graph's output buffers
        dump_outputs(output_arrays(last, exclude=resident), args.dump_outputs, f".rank{rank}" if world > 1 else "")
    del last
    ms_e2e, _, _ = timed(step_e2e, args.steps, 1)
    ms_e2e_nl = None
    if world == 1 and "cell" in sysd:
        ms_e2e_nl, _, _ = timed(step_e2e_device_nl, args.steps, 1)
    clocks = sampler.stop() if rank == 0 else None
    if graphed is not None:
        graphed.check_sorted()  # the in-graph "edges grouped by destination" flag of the last replay

    # ---- parity properties of the very step that was timed, on this hardware and at this size
    checks = parity_checks(step_resident, (lambda frame: model(D.to_device(frame, dev))), base_frame, copies,
                           (plan.owned if halo_mode else None), halo_mode, world, rank, dev)

    # the collective of the data path, timed alone (halo mode): bytes and milliseconds per layer, max over ranks
    exchange = None
    if halo_mode:
        dims = [(li, int(layer.conv.feature_irreps_in.dim)) for li, layer in enumerate(model.layers) if li > 0]
        exchange = halo_exchange_profile(dims, plan, halo, dev, world)

    h2d = sum(v.numel() * v.element_size() for v in host.values() if torch.is_tensor(v))
    d2h = f_host.numel() * 8 + 8

    # ---- rooflines, measured live: every hot kernel class of every layer is timed ALONE (CUDA events on the
    # launching stream, inputs of the step's shapes, > L2); the class with the largest share of the step is the
    # headline `roofline`, the others are listed under `roofline.by_kernel`
    roof = None
    if rank == 0:
        try:  # rank-local: a failure here must not cost the run its bench line
            roof = kernel_rooflines(model, resident, n_atoms, n_edges, max(5, args.steps), ms_res, dev)
        except Exception as exc:
            roof = {"error": f"{type(exc).__name__}: {exc}"[:300]}
            print(f"[bench] per-kernel rooflines failed: {roof['error']}", file=sys.stderr, flush=True)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:  # reported at N = 1 only
        try:
            cpu = cpu_baseline(args.workload)
        except Exception as exc:
            cpu = {"error": f"{type(exc).__name__}: {exc}"[:300]}
            print(f"[bench] cpu_baseline failed: {cpu['error']}", file=sys.stderr, flush=True)

    if rank == 0:
        total_atoms = n_total_atoms if halo_mode else n_atoms * world
        line = {
            "metric": "atom-steps/sec (energy+forces)",
            "value": total_atoms / (ms_res * 1e-3),
            "unit": "atom-steps/s",
            "n_gpus": world,
            "steps": args.steps,
            "warmup": args.warmup,
            "ms_per_step": ms_res,
            "higher_is_better": True,
            "scaling": (args.scaling if halo_mode else "weak"),
            "vs_baseline": None,
            "dtype": "f32",
            "data": "synthetic",
            "config": {
                "workload": args.workload,
                "atoms_per_gpu": n_atoms, "edges_per_gpu": n_edges, "r_max": R_MAX, "parity": True, **mk,
                "parallelism": (f"halo{world}: one {total_atoms}-atom frame (the {copies}-fold periodic supercell of the N=1 "
                                f"workload frame) partitioned by atoms into {grid[0]}x{grid[1]}x{grid[2]} "
                                f"bricks, {plan.n_own} owned + {plan.n_ghost} ghost atoms on rank 0, per-layer NCCL halo "
                                f"exchange of ghost features, energy all-reduce, ghost forces reduced to owners ({args.scaling} scaling)"
                                if halo_mode
                                else f"dp{world} over frames (one {n_atoms}-atom frame per GPU)"),
                "launch": ("one CUDA-graph replay per step (nequip_b200/graph.py)" if graphed is not None
                           else ("eager launches" + (f" (graph capture failed: {graph_error})" if graph_error else ""))),
                "radial_tp_path": [
                    {"layer": i, "choice": ("fused (nqb_tp_fused_fwd)" if l.conv._fused_choice else "k_gemm3x + tp_fwd*"),
                     **{k: round(v, 4) for k, v in (getattr(l.conv, "fused_timing_ms", None) or {}).items()}}
                    for i, l in enumerate(model.layers)],
                "hidden_layer_kernels": "v%d (nqb_mlp.cu)" % ops.mlp_hidden_variant(0),
                "l2_policy": "inputs larger than L2 (edge weights of one layer: %.2f GB)" % (
                    n_edges * max(l.conv.tp_scatter.weight_numel for l in model.layers) * 4 / 1e9),
            },
            "e2e": {"value": total_atoms / (ms_e2e * 1e-3), "unit": "atom-steps/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "e2e_device_neighbor_list": (None if ms_e2e_nl is None else {
                "value": total_atoms / (ms_e2e_nl * 1e-3), "unit": "atom-steps/s", "ms_per_step": ms_e2e_nl,
                "h2d_bytes_per_step": int(host["pos"].numel() * 8), "d2h_bytes_per_step": d2h,
                "note": "positions in, forces out; neighbour list (cell list) built on the GPU inside the timed region"}),
            "gpu_launches": launches,
            "checks": checks,
            "halo_exchange": (None if exchange is None else {
                "per_layer": exchange,
                "ms_per_step_all_layers": sum(e["ms_forward_plus_backward"] for e in exchange),
                "share_of_step": sum(e["ms_forward_plus_backward"] for e in exchange) / ms_res,
                "note": ("the only data-path collective: per-layer all_to_all_single of the ghost rows (NCCL) and its transposed "
                         "backward, timed alone with feature rows of each layer's width; plus one 8-byte energy all-reduce and "
                         "one [n_ghost, 3] float64 reverse exchange of the ghost forces per step")}),
            "clocks": clocks,
            "roofline": roof,
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
