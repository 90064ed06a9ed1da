"""CPU: host-side logic of the product (irreps, CG tables, path tables, generator, neighbour
lists) and the C-ABI surface (library loads, exports every symbol include/nqb.h declares)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from nequip_b200 import _capi, build, cg
from nequip_b200 import data as D
from nequip_b200 import known_signatures as ks
from nequip_b200.codegen import GenOptions, TPSignature, generate
from nequip_b200.irreps import Irrep, Irreps, build_tp_instructions
from oracle import irreps as OI
from oracle import wigner

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_irreps_parse_sort_simplify():
    ir = Irreps("32x0e + 32x1o+1e + 2x2e")
    assert ir.dim == 32 + 96 + 3 + 10 and len(ir) == 4 and ir.num_irreps == 67
    assert repr(ir) == "32x0e+32x1o+1x1e+2x2e"
    s, p, inv = Irreps("2x1e+3x0e+1x1o+4x0e").sort()
    assert repr(s) == "3x0e+4x0e+1x1o+2x1e"  # (l,p) order: 1o=(1,-1) before 1e=(1,+1); stable
    assert p == (3, 0, 2, 1) and inv == (1, 3, 2, 0)
    assert repr(s.simplify()) == "7x0e+1x1o+2x1e"
    assert repr(Irreps.spherical_harmonics(3)) == "1x0e+1x1o+1x2e+1x3o"
    assert [repr(x) for x in Irrep(1, -1) * Irrep(2, 1)] == ["1o", "2o", "3o"]
    # the product and oracle bookkeeping agree
    assert OI.fmt(OI.sort(OI.parse("2x1e+3x0e+1x1o+4x0e"))[0]) == repr(s)


@pytest.mark.parametrize("cfg,expect", [
    ((2, 64, 4), [(64, 3, 192, 576), (576, 15, 960, 3264), (1088, 27, 1728, 5952), (1152, 3, 192, 192)]),
    ((2, 32, 4), [(32, 3, 96, 288), (288, 15, 480, 1632), (544, 27, 864, 2976), (576, 3, 96, 96)]),
    ((3, 32, 5), [(32, 4, 128, 512), (512, 34, 1088, 4992), (992, 64, 2048, 9472), (1024, 68, 2176, 9984), (1024, 4, 128, 128)]),
    ((1, 32, 4), [(32, 2, 64, 128), (128, 5, 160, 352), (224, 8, 256, 576), (256, 2, 64, 64)]),
])
def test_layer_shapes_match_survey_appendix_B(cfg, expect):
    got = [(s.d_in, len(s.paths), s.weight_numel, s.d_out) for s in ks.nequip_layer_signatures(*cfg)]
    assert got == expect


def test_instruction_builder_matches_oracle_bookkeeping():
    fin, fout = "8x0e+8x1e+8x1o+8x2e+8x2o", "8x0e+8x0o+8x1e+8x1o+8x2e+8x2o"
    mid, ins = build_tp_instructions(fin, Irreps.spherical_harmonics(2), fout)
    omid, oins = OI.build_tp_instructions(fin, OI.spherical_harmonics(2), fout)
    assert repr(mid) == OI.fmt(omid)
    assert [tuple(i[:3]) for i in ins] == [tuple(i[:3]) for i in oins]


def test_cg_tables_match_oracle():
    for l1 in range(4):
        for l2 in range(4):
            for l3 in range(abs(l1 - l2), min(3, l1 + l2) + 1):
                np.testing.assert_allclose(np.array(cg.real_w3j(l1, l2, l3)), wigner.wigner_3j(l1, l2, l3), atol=1e-15)
    assert len(cg.sparse_w3j(2, 2, 2)) == 25 and len(cg.sparse_w3j(3, 3, 3)) == 42


def test_signature_validation():
    with pytest.raises(NotImplementedError):
        TPSignature(Irreps("2x0e"), Irreps("2x0e"), Irreps("2x0e"), [(0, 0, 0)])  # edge attr mul > 1
    with pytest.raises(ValueError):
        TPSignature(Irreps("2x0e"), Irreps("1x1o"), Irreps("2x0e"), [(0, 0, 0)])  # 0e x 1o !-> 0e
    with pytest.raises(NotImplementedError):
        TPSignature(Irreps("2x0e"), Irreps("1x0e"), Irreps("2x0e"), [(0, 0, 0, "uvw", True)])
    s = ks.nequip_layer_signatures(2, 64, 4)[2]
    assert s.fma_count() == 487
    assert all(abs(p.coef - (2 * p.l3 + 1) ** 0.5) < 1e-15 for p in s.paths)


def test_generator_emits_packed_fma_source():
    sig = ks.nequip_layer_signatures(2, 32, 4)[1]
    src = generate(sig, GenOptions())
    assert "tp_fwd_kernel" in src and "tp_bwd_kernel" in src and "vfmai(" in src
    assert 'extern "C" int nqb_spec_fwd' in src and sig.canonical() in src
    # every path's weight slice is loaded exactly once in the forward
    # software-pipelined loop: two register sets (A/B), each path's weight slice loaded into both,
    # in the forward and in the backward kernel
    for p in sig.paths:
        assert len(re.findall(rf"\bw{p.idx}A = vloadw", src)) == 4
        assert len(re.findall(rf"\bw{p.idx}B = vloadw", src)) == 2


def test_capi_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "nqb.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(nqb_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    lib = ctypes.CDLL(build.ensure_runtime())
    for name in sorted(declared):
        assert hasattr(lib, name), f"libnqb.so does not export {name}"
    assert declared == set(_capi.SIGNATURES), declared ^ set(_capi.SIGNATURES)
    assert _capi.lib().nqb_abi_version() == 1


def test_plan_create_validates_signature():
    """Host-only C-ABI calls: plan creation binds the prebuilt kernel library and rejects a mismatched one."""
    from nequip_b200 import ops

    sigs = ks.nequip_layer_signatures(1, 8, 2)
    plan = ops.TPPlan(sigs[0].irreps_in1, sigs[0].irreps_in2, sigs[0].irreps_out, sigs[0].instructions)
    assert (plan.d_in, plan.s_dim, plan.weight_numel, plan.d_out) == (sigs[0].d_in, 4, sigs[0].weight_numel, sigs[0].d_out)
    L = _capi.lib()
    buf = ctypes.create_string_buffer(4096)
    L.nqb_plan_signature(plan.handle, buf, 4096)
    assert buf.value.decode() == sigs[0].canonical()
    # wrong library for this signature
    wrong = build.ensure_spec(sigs[1])
    in1 = (_capi.NqbIrrep * 1)(_capi.NqbIrrep(8, 0, 1))
    in2 = (_capi.NqbIrrep * 1)(_capi.NqbIrrep(1, 0, 1))
    ins = (_capi.NqbInstruction * 1)(_capi.NqbInstruction(0, 0, 0))
    h = ctypes.c_void_p()
    rc = L.nqb_plan_create(in1, 1, in2, 1, in1, 1, ins, 1, wrong.encode(), ctypes.byref(h))
    assert rc != 0 and b"different signature" in L.nqb_last_error()
    # selection-rule violation is caught by the C side too
    in2b = (_capi.NqbIrrep * 1)(_capi.NqbIrrep(1, 1, -1))
    rc = L.nqb_plan_create(in1, 1, in2b, 1, in1, 1, ins, 1, wrong.encode(), ctypes.byref(h))
    assert rc != 0 and b"selection rules" in L.nqb_last_error()


def test_ops_reject_cpu_tensors():
    from nequip_b200 import ops

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.spherical_harmonics(torch.randn(4, 3, dtype=torch.float64), 2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.edge_embed(torch.randn(4, 3), torch.zeros(2, 3, dtype=torch.long), lmax=1, r_max=5.0)


def test_neighbor_list_cell_list_vs_bruteforce():
    pos, cell = D.jittered_lattice(8, 0.104, seed=3)
    ei, sh = D.neighbor_list(pos, cell, 5.0)
    ei2, sh2 = D._nl_bruteforce(pos, np.diag(cell), 5.0)
    assert np.array_equal(ei, ei2) and np.array_equal(sh, sh2)
    v = pos[ei[1]] - pos[ei[0]] + sh @ cell
    r = np.linalg.norm(v, axis=1)
    assert r.max() < 5.0 and r.min() > 0.5
    # full list: every edge has its reverse
    fwd = set(zip(ei[0].tolist(), ei[1].tolist(), map(tuple, sh.astype(int).tolist())))
    assert all((j, i, (-a, -b, -c)) in fwd for (i, j, (a, b, c)) in list(fwd)[:2000])
    # sorted by (centre, neighbour)
    assert np.all(np.diff(ei[0]) >= 0)


@pytest.mark.parametrize("layout", ["mul_ir", "ir_mul"])
def test_gate_tables_reproduce_the_torch_gate(layout):
    """The column tables fed to nqb_gate_fwd/bwd, evaluated in plain torch exactly as the kernels do, must
    reproduce Gate.forward and its autograd gradient (e3nn nn.Gate semantics, convnetlayer.py:104-112)."""
    import torch

    from nequip_b200 import ops
    from nequip_b200.nn.model import C_SILU, C_TANH, Gate

    scal, gates, gated = "8x0e+4x0o", "8x0e+4x0o+4x0e", "8x1o+4x1e+4x2e"
    g = Gate(scal, gates, gated, layout)
    t = ops.GateTables(scal, gates, gated, layout, "cpu")
    gen = torch.Generator().manual_seed(0)
    x = torch.randn(5, t.d_in, generator=gen, dtype=torch.float64, requires_grad=True)
    ref = g(x)
    go = torch.randn(ref.shape, generator=gen, dtype=torch.float64)
    (gx_ref,) = torch.autograd.grad(ref, x, go)

    def act(v, k):
        return torch.where(k == 0, C_SILU * v * torch.sigmoid(v), C_TANH * torch.tanh(v))

    def dact(v, k):
        s = torch.sigmoid(v)
        return torch.where(k == 0, C_SILU * s * (1 + v * (1 - s)), C_TANH * (1 - torch.tanh(v) ** 2))

    xd = x.detach()
    src, gate, kind = t.src.long(), t.gate.long(), t.kind.long()
    v = xd[:, src]
    out = torch.where(gate < 0, act(v, kind), v * act(xd[:, gate.clamp(min=0)], kind))
    torch.testing.assert_close(out, ref.detach(), rtol=1e-12, atol=1e-12)
    tab = t.tab.view(-1, 6).long()
    gx = torch.zeros_like(xd)
    for i in range(t.d_in):
        role, a, b, c, d, k = (int(z) for z in tab[i])
        kk = torch.tensor(k)
        if role == 0:
            gx[:, i] = go[:, a] * dact(xd[:, i], kk)
        elif role == 1:
            gx[:, i] = go[:, a] * act(xd[:, b], kk)
        else:
            ssum = sum(go[:, a + cc * c] * xd[:, b + cc * c] for cc in range(d))
            gx[:, i] = ssum * dact(xd[:, i], kk)
    torch.testing.assert_close(gx, gx_ref, rtol=1e-12, atol=1e-12)


def test_weighted_cta_split_covers_the_grid(monkeypatch):
    """ops.GroupedGemm._weighted_split: every N-tile gets >= 1 CTA, ranges are disjoint and contiguous, the grid
    is fully used, expensive tiles (long K, reduce-add stores) get more CTAs; uniform launches keep the even split."""
    import types

    import torch

    from nequip_b200 import ops

    monkeypatch.setattr(torch.cuda, "get_device_properties", lambda d: types.SimpleNamespace(multi_processor_count=148))
    made = {}
    real_tensor = torch.tensor

    def fake_tensor(data, dtype=None, device=None):
        made["tab"] = list(data)
        return real_tensor(data, dtype=dtype)

    monkeypatch.setattr(torch, "tensor", fake_tensor)
    # rows: [a_off, c_off, b_off, rs_off, lda, ldc, K, N, kchunks, ntiles, tile0, flags]
    rows = [[0, 0, 0, -1, 64, 64, 64, 64, 2, 1, 0, 0], [0, 0, 0, -1, 64, 64, 448, 384, 14, 3, 1, 4],
            [0, 0, 0, -1, 64, 64, 64, 300, 2, 3, 4, 0]]
    tab, G = ops.GroupedGemm._weighted_split(rows, "cuda")
    t = made["tab"]
    c0, n = t[0::2], t[1::2]
    assert G == 148 and len(n) == 7 and min(n) >= 1 and sum(n) == 148
    assert c0 == [sum(n[:i]) for i in range(7)]
    assert min(n[1:4]) > max(n[0], *n[4:])  # K = 448 with reduce-adds is the expensive problem
    # uniform launch: even split (None)
    rows_u = [[0, 0, 0, -1, 128, 1728, 128, 1728, 4, 14, 0, 0]]
    assert ops.GroupedGemm._weighted_split(rows_u, "cuda") == (None, 0)


def test_per_type_scale_shift_accepts_scalar_and_per_type_tables():
    """PerTypeScaleShift (atomwise.py:236-284): a float / one-element list broadcasts over the types."""
    from nequip_b200.nn.model import NequIPEnergyModel

    kw = dict(r_max=4.0, type_names=["H", "O", "C"], l_max=1, num_layers=2, num_features=4, radial_mlp_width=8)
    m = NequIPEnergyModel(per_type_energy_scales=2.5, per_type_energy_shifts=[-1.0], **kw)
    assert m.scales.shape == (3, 1) and torch.all(m.scales == 2.5) and torch.all(m.shifts == -1.0)
    types = torch.tensor([0, 2, 1, 2])
    assert m.scales[types].shape == (4, 1)  # indexable by any type id (was out of bounds for a [1,1] table)
    m = NequIPEnergyModel(per_type_energy_scales=[1.0, 2.0, 3.0], **kw)
    assert m.scales.view(-1).tolist() == [1.0, 2.0, 3.0] and m.shifts.numel() == 0
    with pytest.raises(ValueError):
        NequIPEnergyModel(per_type_energy_scales=[1.0, 2.0], **kw)


def test_total_energy_is_reduced_per_graph():
    """AtomwiseReduce (atomwise.py:92-113): [num_graphs, 1] for batched input, [1, 1] for a single frame."""
    from nequip_b200.nn.model import NequIPEnergyModel

    e = torch.arange(6, dtype=torch.float64).view(6, 1)
    assert NequIPEnergyModel._reduce_energy(e, {}).tolist() == [[15.0]]
    batch = torch.tensor([0, 0, 1, 1, 1, 2])
    out = NequIPEnergyModel._reduce_energy(e, {"batch": batch, "ptr": torch.tensor([0, 2, 5, 6])})
    assert out.tolist() == [[1.0], [9.0], [5.0]]
    out = NequIPEnergyModel._reduce_energy(e, {"batch": batch, "num_atoms": torch.tensor([2, 3, 1, 0])})
    assert out.shape == (4, 1) and out[3, 0] == 0


def test_model_construction_loads_no_native_code_and_strict_flag_propagates():
    """bench.py's CPU reference arm builds the model only for its state dict: that must not dlopen the kernels."""
    import subprocess
    import sys

    code = ("import sys; sys.path.insert(0, %r)\n"
            "from nequip_b200.nn.model import NequIPEnergyModel\n"
            "m = NequIPEnergyModel(r_max=4.0, type_names=['A'], l_max=2, num_layers=2, num_features=8, radial_mlp_width=16,"
            " strict_fast_path=True)\n"
            "assert all(l.conv.strict_fast_path for l in m.layers)\n"
            "sd = m.state_dict()\n"
            "maps = open('/proc/self/maps').read()\n"
            "assert 'libnqb' not in maps and 'nqbspec' not in maps, 'native kernels were loaded'\n"
            "print('ok')\n") % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_reference_checkpoint_key_mapping_round_trip():
    """nequip_b200/nn/checkpoint.py: parameters travel under the reference's module names
    (nequip/model/nequip_models.py:288-399) with any wrapper prefix; e3nn buffers are ignored."""
    from nequip_b200.nn.checkpoint import load_reference_state_dict, reference_key_map, to_reference_state_dict
    from nequip_b200.nn.model import NequIPEnergyModel

    kw = dict(r_max=4.0, type_names=["H", "O"], l_max=2, num_layers=3, num_features=8, radial_mlp_width=16)
    a = NequIPEnergyModel(per_type_energy_scales=[1.5, 2.0], per_type_energy_shifts=0.25, seed=1, **kw)
    ref = to_reference_state_dict(a, prefix="model.func.")
    assert "model.func.type_embed.embed_module.weight" in ref
    assert "model.func.layer2_convnet.conv.sc.weight" in ref and "model.func.layer0_convnet.conv.sc.weight" not in ref
    assert "model.func.per_atom_energy_readout.mlp_module.mlp.0.weight" in ref
    assert len(ref) == len(reference_key_map(3))
    # what a real checkpoint additionally holds: e3nn buffers of the un-used self.tp, output masks
    ref["model.func.layer1_convnet.conv.tp_scatter.tp._w3j_1_1_2"] = torch.zeros(3)
    ref["model.func.layer1_convnet.conv.linear_1.output_mask"] = torch.ones(5)
    b = NequIPEnergyModel(per_type_energy_scales=[1.0, 1.0], per_type_energy_shifts=[0.0, 0.0], seed=2, **kw)
    missing, unexpected = load_reference_state_dict(b, ref)
    assert missing == [] and unexpected == []
    for (ka, va), (kb, vb) in zip(a.state_dict().items(), b.state_dict().items()):
        assert ka == kb and torch.equal(va, vb), ka
    ref["model.func.something_else.weight"] = torch.zeros(2)
    with pytest.raises(KeyError):
        load_reference_state_dict(b, ref)
    with pytest.raises(ValueError):
        load_reference_state_dict(b, {"func.type_embed.embed_module.weight": torch.zeros(3, 3)}, strict=False)


def test_bench_reference_arm_json_contract(tmp_path):
    """``bench.py --impl reference`` (the CPU arm timed beside the GPU arm): one JSON line with the metric /
    unit / higher_is_better of the own arm, ``impl``, a ``cpu_baseline`` describing the run, zero-copy ``e2e`` and the
    workload + model keys in ``config``; ``--dump-outputs`` writes the outputs of its last step."""
    import json
    import subprocess
    import sys

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny",
                        "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "atom-steps/sec (energy+forces)"
    assert line["unit"] == "atom-steps/s" and line["higher_is_better"] is True and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["value"] == line["value"] == line["e2e"]["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    cfg = line["config"]
    assert cfg["workload"] == "tiny" and cfg["l_max"] == 2 and cfg["num_layers"] == 3 and cfg["num_features"] == 8
    assert cfg["atoms_per_step_sample"] > 0 and cfg["edges_per_step_sample"] > 0
    f = np.load(tmp_path / "forces.npy")
    assert f.shape == (cfg["atoms_per_step_sample"], 3) and f.dtype in (np.float32, np.float64)
    assert np.load(tmp_path / "total_energy.npy").size == 1 and (tmp_path / "atomic_energy.npy").exists()


def test_bench_cpu_sample_size_respects_the_budget():
    sys_path_bench = os.path.join(ROOT, "bench.py")
    import importlib.util

    spec = importlib.util.spec_from_file_location("nqb_bench", sys_path_bench)
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    wl = "li3po4_10k_l2_f64"
    lo, hi = bench.CPU_SAMPLE_NSIDE_MIN[wl], bench.CPU_SAMPLE_NSIDE_MAX[wl]
    assert bench.pick_sample_nside(wl, 1e-9, 3) == hi           # cheap: the largest sample (1000 atoms)
    assert bench.pick_sample_nside(wl, 1e3, 3) == lo            # hopeless: the smallest allowed
    n = bench.pick_sample_nside(wl, 0.0137, 25, budget_s=bench.REF_ARM_BUDGET_S)  # the driver's 20 + 5 steps on this pool's host
    assert lo <= n <= hi and 25 * 0.0137 * n ** 3 <= bench.REF_ARM_BUDGET_S < 25 * 0.0137 * (n + 1) ** 3
    # algorithmic bytes of the TP kernels (SURVEY 8d): forward = x + Y + w + out + two index arrays
    sig = type("S", (), dict(d_in=10, s_dim=4, weight_numel=6, d_out=20))
    assert bench.tp_algorithmic_bytes(sig, 3, 7) == 4 * (3 * 10 + 7 * 4 + 7 * 6 + 3 * 20) + 16 * 7


def test_bench_force_sum_property_vector():
    """bench.py's size-independent parity property (sum of all forces = 0): the per-rank vector that is all-reduced."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("nqb_bench2", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    f = torch.randn(50, 3, dtype=torch.float32)
    v = bench.force_sum_vector(f)
    assert v.dtype == torch.float64 and v.shape == (5,)
    assert torch.allclose(v[:3], f.double().sum(0)) and float(v[3]) == pytest.approx(float(f.double().abs().sum())) and float(v[4]) == 1.0
    # two "ranks" whose forces cancel
    tot = bench.force_sum_vector(f) + bench.force_sum_vector(-f)
    assert float(tot[:3].abs().max()) == 0.0 and float(tot[4]) == 2.0


def test_bench_dump_outputs(tmp_path):
    """``bench.py --dump-outputs``: the floating-point outputs of a step (not its inputs, not integer flags) as float32 /
    float64 .npy files, 64 MB in all, a larger array replaced by the same seeded sample on every run."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("nqb_bench3", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    out = {"total_energy": torch.tensor([1.5], dtype=torch.float64), "forces": torch.randn(7, 3),
           "atomic_energy": torch.randn(7, 1, dtype=torch.float16), "edges_sorted": torch.ones(1, dtype=torch.int32),
           "pos": torch.randn(7, 3, dtype=torch.float64)}
    arrs = bench.output_arrays(out, exclude={"pos": None})
    assert sorted(arrs) == ["atomic_energy", "forces", "total_energy"]
    assert arrs["forces"].dtype == np.float32 and arrs["total_energy"].dtype == np.float64
    assert arrs["atomic_energy"].dtype == np.float32
    bench.dump_outputs(arrs, str(tmp_path / "a"))
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "forces.npy"), out["forces"].numpy())
    assert np.load(tmp_path / "a" / "total_energy.npy").tolist() == [1.5]
    # over the limit: a seeded sample of the flattened elements and their positions
    big = {"x": np.arange(bench.DUMP_LIMIT_BYTES // 8 + 1000, dtype=np.float64), "e": np.zeros(1)}
    for d in ("b", "c"):
        bench.dump_outputs(big, str(tmp_path / d), suffix=".rank1")
    x, idx = np.load(tmp_path / "b" / "x.rank1.npy"), np.load(tmp_path / "b" / "x.rank1.index.npy")
    assert idx.dtype == np.float64 and x.dtype == np.float64 and np.array_equal(x, idx) and 0 < x.size < big["x"].size
    assert np.array_equal(idx, np.load(tmp_path / "c" / "x.rank1.index.npy"))
    assert sum(f.stat().st_size for f in (tmp_path / "b").iterdir()) <= bench.DUMP_LIMIT_BYTES
