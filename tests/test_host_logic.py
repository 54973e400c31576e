"""CPU: the C-ABI library loads and exports what include/difflinker_b200.h declares; the Python mirrors keep the
reference's interface (constructor kwargs, state_dict keys, exception attributes); sharding logic under gloo."""
import os
import re
import shutil
import subprocess
import sys

import pytest
import torch

import difflinker_b200
from difflinker_b200 import _native, synthetic
from difflinker_b200.distributed import batch_ids_for_rank, shard_range
from difflinker_b200.utils import FoundNaNException
import dl_helpers as helpers
from oracle import difflinker_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "difflinker_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dl_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = _native.load_library()
    names = header_functions()
    assert len(names) >= 14
    for n in names:
        assert hasattr(lib, n), f"{n} declared in the header but not exported"
        assert n in _native.SYMBOLS, f"{n} has no ctypes prototype"
    assert b"sm_100a" in lib.dl_version()


def test_state_dict_keys_and_param_count_match_reference_layout():
    m, hp = helpers.build_ddpm(synthetic.SPECS["cfg2_zinc"], 0)
    keys = list(m.state_dict().keys())
    assert keys[0] == "edm.gamma.gamma"
    assert "edm.dynamics.dynamics.embedding.weight" in keys
    assert "edm.dynamics.dynamics.e_block_5.gcl_1.edge_mlp.2.weight" in keys
    assert "edm.dynamics.dynamics.e_block_0.gcl_equiv.coord_mlp.4.weight" in keys
    assert "edm.dynamics.dynamics.e_block_0.gcl_equiv.coord_mlp.4.bias" not in keys
    sd = m.state_dict()
    assert tuple(sd["edm.dynamics.dynamics.e_block_0.gcl_0.edge_mlp.0.weight"].shape) == (128, 258)
    assert tuple(sd["edm.dynamics.dynamics.embedding.weight"].shape) == (128, 10)
    n_dyn = sum(v.numel() for k, v in sd.items() if k.startswith("edm.dynamics."))
    assert n_dyn + 501 == 1490815                                       # SURVEY.md section 8(b): L=6, D=10, incl. gamma
    assert sd["edm.gamma.gamma"].numel() == 501


def test_unsupported_options_refuse_loudly():
    with pytest.raises(NotImplementedError):
        difflinker_b200.Dynamics(n_dims=3, in_node_nf=8, context_node_nf=1, hidden_nf=128, attention=True)
    with pytest.raises(NotImplementedError):
        difflinker_b200.Dynamics(n_dims=3, in_node_nf=8, context_node_nf=1, hidden_nf=128, model='gnn_dynamics')
    with pytest.raises(NotImplementedError):
        difflinker_b200.EDM(dynamics=None, in_node_nf=8, n_dims=3, noise_schedule='learned')


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback_without_gpu():
    dyn, hp = helpers.build_dynamics(helpers.EXTRA_SPECS["small_fc"], 0)
    z = torch.zeros(1, 4, 11)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        dyn(torch.zeros(1, 1), z, torch.ones(1, 4, 1), torch.ones(1, 4, 1), torch.ones(16, 1), torch.ones(1, 4, 1))


def test_normalization_hyperparameter_is_ignored_like_the_reference():
    """Every published config / checkpoint carries normalization='batch_norm'; for model='egnn_dynamics' the reference
    never reads it (src/egnn.py:340-368), so neither constructor may refuse it."""
    d = difflinker_b200.Dynamics(n_dims=3, in_node_nf=8, context_node_nf=1, hidden_nf=128, normalization='batch_norm')
    assert isinstance(d, torch.nn.Module)
    spec = synthetic.SPECS["cfg1_plumbing"]
    hp = synthetic.model_hparams(spec)
    assert hp['normalization'] == 'batch_norm'
    m, _ = helpers.build_ddpm(spec, 0)
    assert isinstance(m.edm.dynamics, difflinker_b200.Dynamics)


def test_nan_exception_is_catchable_as_the_reference_class():
    """generate.py:154-159 retries on `except FoundNaNException` with the class imported from src.utils; the native
    sampler must raise something that clause catches (and that this package's own class catches too)."""
    import sys, types
    from difflinker_b200.utils import nan_exception_class
    saved = sys.modules.get('src.utils')
    try:
        sys.modules.pop('src.utils', None)
        assert nan_exception_class() is FoundNaNException
        mod = types.ModuleType('src.utils')

        class RefNaN(Exception):                     # constructor signature of src/utils.py:274-282
            def __init__(self, x, h):
                self.x_h_nan_idx = set()
        mod.FoundNaNException = RefNaN
        sys.modules['src.utils'] = mod
        cls = nan_exception_class()
        assert issubclass(cls, RefNaN) and issubclass(cls, FoundNaNException) and nan_exception_class() is cls
        with pytest.raises(RefNaN) as ei:
            raise cls(flags=[0, 1, 3])
        assert ei.value.only_x_nan_idx == {1} and ei.value.x_h_nan_idx == {2}
    finally:
        if saved is not None:
            sys.modules['src.utils'] = saved
        else:
            sys.modules.pop('src.utils', None)


def test_nan_exception_mapping():
    e = FoundNaNException(flags=[0, 1, 2, 3 | (7 << 8), 1 | (9 << 8)])
    assert e.x_h_nan_idx == {3} and e.only_x_nan_idx == {1, 4} and e.only_h_nan_idx == {2}
    assert e.first_step == 6
    x = torch.zeros(3, 2, 3); h = torch.zeros(3, 2, 8)
    x[1, 0, 0] = float('nan'); h[1, 1, 1] = float('nan'); h[2, 0, 0] = float('nan')
    e2 = FoundNaNException(x, h)
    assert e2.x_h_nan_idx == {1} and e2.only_h_nan_idx == {2} and e2.only_x_nan_idx == set()


def test_shard_helpers():
    for n, w in [(10, 3), (8, 8), (3, 4), (0, 2)]:
        spans = [shard_range(n, r, w) for r in range(w)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))
        assert max(hi - lo for lo, hi in spans) - min(hi - lo for lo, hi in spans) <= 1
    assert batch_ids_for_rank(7, 1, 3) == [1, 4]
    assert sorted(sum((batch_ids_for_rank(7, r, 3) for r in range(3)), [])) == list(range(7))


def test_weight_broadcast_world_size_2_gloo(tmp_path):
    """N>1 path on CPU: rank 1 starts from different weights and must end up with rank 0's after the single
    broadcast; per-rank batches are disjoint."""
    script = tmp_path / "w.py"
    script.write_text(f"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {ROOT!r} + '/tests')
from difflinker_b200 import synthetic
from difflinker_b200.distributed import broadcast_module_weights, batch_ids_for_rank
import dl_helpers as helpers
dist.init_process_group("gloo")
rank = dist.get_rank()
m, hp = helpers.build_ddpm(helpers.EXTRA_SPECS["small_fc"], seed=rank)
n = broadcast_module_weights(m, src=0)
sha = helpers.state_sha(m.state_dict())
ref, _ = helpers.build_ddpm(helpers.EXTRA_SPECS["small_fc"], seed=0)
assert sha == helpers.state_sha(ref.state_dict()), rank
assert n == sum(p.numel() for p in m.parameters())
ids = batch_ids_for_rank(5, rank, 2)
gathered = [None, None]
dist.all_gather_object(gathered, ids)
assert sorted(gathered[0] + gathered[1]) == [0, 1, 2, 3, 4]
dist.destroy_process_group()
print("rank", rank, "ok")
""")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29517", str(script)],
                         capture_output=True, text=True, env=env, timeout=300)
    assert res.returncode == 0, res.stdout + res.stderr
    assert res.stdout.count("ok") == 2


def test_sharded_sampling_gathers_the_full_batch_world_size_2_gloo(tmp_path):
    """distributed.sample_chain_sharded under gloo, world size 2 (uneven split 3 + 2): every rank builds the same template
    batch, samples its slice (stand-in EDM: a deterministic function of the slice, no GPU here) and the all_gather
    reassembles the batch order."""
    script = tmp_path / "sharded.py"
    script.write_text(f"""
import os, sys, types, torch, torch.distributed as dist
sys.path.insert(0, {str(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))!r})
from difflinker_b200 import synthetic
from difflinker_b200.batching import collate
from difflinker_b200.distributed import sample_chain_sharded, shard_range
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:" + sys.argv[1], rank=int(sys.argv[2]), world_size=2)
spec = synthetic.SPECS["cfg1_plumbing"]
data = collate(synthetic.make_items(spec, batch=5))
seen = dict()
class FakeEDM:
    def sample_chain(self, x, h, node_mask, fragment_mask, linker_mask, edge_mask, context, keep_frames=None, batch_slice=None):
        seen["slice"] = batch_slice; seen["B"] = x.shape[0]
        assert edge_mask.shape[0] == x.shape[0] * x.shape[1] * x.shape[1]
        return torch.stack([torch.cat([x, h], dim=2) * (f + 1) for f in range(keep_frames)])
model = types.SimpleNamespace(inpainting=False, anchors_context=False, train_data_prefix="zinc_train", center_of_mass="fragments",
                              val_dataset=None, edm=FakeEDM())
chain, node_mask = sample_chain_sharded(model, data, keep_frames=2)
lo, hi = shard_range(5, dist.get_rank(), 2)
assert seen["slice"] == (lo, 5) and seen["B"] == hi - lo, seen
dist.destroy_process_group()
single = types.SimpleNamespace(**{{**model.__dict__}})
full, nm = sample_chain_sharded(single, data, keep_frames=2)           # world size 1 path
assert torch.equal(chain, full) and torch.equal(node_mask, nm) and chain.shape[1] == 5
print("ok")
""")
    import socket
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    procs = [subprocess.Popen([sys.executable, str(script), str(port), str(r)], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                              text=True) for r in range(2)]
    for pr in procs:
        out, err = pr.communicate(timeout=240)
        assert pr.returncode == 0 and "ok" in out, out + err


def test_accelerate_swaps_reference_edm():
    """Whole-loop drop-in: a *reference* DDPM gets the native EDM with the same weights; strict state_dict load proves the
    key layout. accelerate() reads `hparams`, `edm.state_dict()` and `edm.T` of the reference DDPM; the stand-in carries
    the reference EDM's state_dict as recorded by oracle/make_golden.py (keys in its order, shapes, sha256 of the values
    its constructor draws for the seed), and the seeded native DDPM reproduces those values."""
    import types
    meta, _ = helpers.load_golden("ref_edm_small_fc")
    assert meta["cls"] == "EDM"
    hp = synthetic.model_hparams(helpers.spec_by_name(meta["spec"]))
    torch.manual_seed(meta["seed"])
    sd = difflinker_b200.DDPM(**hp).edm.state_dict()
    assert list(sd) == meta["keys"] and [list(v.shape) for v in sd.values()] == meta["shapes"]
    assert helpers.state_sha(sd) == meta["sha"]
    ref_edm = types.SimpleNamespace(state_dict=lambda: sd, T=meta["T"])
    ref = types.SimpleNamespace(hparams=hp, edm=ref_edm)
    before = {k: v.clone() for k, v in ref.edm.state_dict().items()}
    ref.edm.T = 7
    out = difflinker_b200.accelerate(ref)
    assert out is ref and isinstance(ref.edm, difflinker_b200.EDM) and ref.edm.T == 7
    after = ref.edm.state_dict()
    assert list(after.keys()) == list(before.keys())
    assert all(torch.equal(after[k], before[k]) for k in before)


# ------------------------------------------------------------------------------------------------
# output stage (generate.py:163-180, visualizer.py:14-31)
# ------------------------------------------------------------------------------------------------
def _xyz_golden(name):
    meta, a = helpers.load_golden(name)
    blob, offs = bytes(a["text"].tolist()), a["offsets"].tolist()
    return meta, a, [blob[offs[i]:offs[i + 1]].decode() for i in range(len(offs) - 1)]


@pytest.mark.parametrize("name", ["xyz_zinc", "xyz_geom"])
def test_xyz_text_oracle_and_native_formatter_match_reference_files(name, tmp_path):
    """The reference's own save_xyz_file output (written by oracle/make_golden.py) pins both the oracle restatement and
    the batched native formatter, byte for byte -- incl. -0.0, nan/inf, 1e38 and last-digit rounding cases."""
    from difflinker_b200 import output
    meta, a, want = _xyz_golden(name)
    idx2atom = output.GEOM_IDX2ATOM if meta["is_geom"] else output.IDX2ATOM
    assert orc.xyz_text(a["one_hot"], a["positions"], a["node_mask"], idx2atom) == want
    assert output.format_xyz(a["one_hot"], a["positions"], a["node_mask"], meta["is_geom"]) == want
    names = [f"output_{i}_mol" for i in range(len(want))]
    output.save_xyz_file(str(tmp_path), a["one_hot"], a["positions"], a["node_mask"], names, meta["is_geom"], suffix='')
    for n, w in zip(names, want):
        assert (tmp_path / f"{n}_.xyz").read_text() == w           # generate.py:176 reads `<name>_.xyz`


def test_xyz_formatter_edge_cases():
    from difflinker_b200 import output
    # empty molecule: header only; chain[0]-style strided input (3+F columns) is accepted as positions
    oh = torch.zeros((2, 3, 8)); oh[:, :, 2] = 1
    xh = torch.cat([torch.arange(18.).view(2, 3, 3), oh], dim=2)
    nm = torch.tensor([[0, 0, 0], [1, 0, 1]], dtype=torch.int8).unsqueeze(-1)
    got = output.format_xyz(oh, xh, nm, False)
    assert got[0] == "0\n\n"
    assert got[1] == "2\n\nN 9.000000000 10.000000000 11.000000000\nN 15.000000000 16.000000000 17.000000000\n"
    with pytest.raises(KeyError):
        output.format_xyz(torch.zeros((1, 2, 10)), torch.zeros((1, 2, 3)), torch.ones((1, 2, 1)), True)
    with pytest.raises(RuntimeError):
        output.restore_frame(torch.zeros((1, 2, 3)), torch.zeros((1, 2, 3)), torch.ones((1, 2, 1)), torch.ones((1, 2, 1)))


# ------------------------------------------------------------------------------------------------
# linker-size classifier host mirror (linker_size.py, linker_size_lightning.py)
# ------------------------------------------------------------------------------------------------
def test_size_classifier_host_mirror_layout_and_errors():
    from difflinker_b200 import SizeClassifier, linker_size
    m = SizeClassifier(in_node_nf=8, out_node_nf=10, n_layers=3, normalization='batch_norm')
    keys = list(m.state_dict())
    assert keys[0] == 'gnn.embedding_in.weight' and keys[-1] == 'gnn.embedding_out.bias'
    assert 'gnn.gcl_layers.1.node_mlp.4.running_var' in keys and 'gnn.gcl1.edge_mlp.2.bias' in keys
    assert m.state_dict()['gnn.gcl1.edge_mlp.0.weight'].shape == (128, 257)       # [h_i | h_j | radial], linker_size.py:59
    data = linker_size.collate_with_fragment_edges(synthetic.make_items(synthetic.SPECS["cfg1_plumbing"], batch=3))
    B, N = data['positions'].shape[:2]
    em = data['edge_mask'].view(B, N, N)
    fm = data['fragment_mask'].squeeze(-1)
    assert set(em.unique().tolist()) <= {0.0, -1.0, -2.0}                           # datasets.py:396-399
    assert torch.equal(em != 0, (fm[:, :, None] * fm[:, None, :]) != 0)            # fragment pairs, self loops live
    assert torch.equal(data['edges'][0][:N * N], torch.arange(N).repeat_interleave(N))
    with pytest.raises(RuntimeError):                                              # no CPU fallback
        m.eval().forward(data, return_loss=False)
    assert m.get_true_labels(data['linker_mask']).tolist() == [m.linker_size2id.get(int(v), m.linker_size2id[12])
                                                               for v in data['linker_mask'].sum((1, 2)).tolist()]


@pytest.mark.parametrize("spec_name,nb", [("cfg1_plumbing", 4), ("cfg2_zinc_ragged", 9), ("cfg4_pockets", 2)])
def test_batched_template_creation_equals_per_molecule_formulation(spec_name, nb):
    """datasets.create_templates_for_linker_generation (483-512): the batched masked-select version must reproduce the
    decouple-and-recollate formulation key by key (order, dtype, shape, values) for shrinking, growing and zero linkers."""
    from difflinker_b200 import batching
    spec = synthetic.SPECS[spec_name]
    data = batching.collate(synthetic.make_items(spec, batch=nb))
    g = torch.Generator().manual_seed(nb)
    for trial in range(3):
        sizes = torch.randint(0, 15, (nb,), generator=g).to(torch.int8)
        if trial == 2:
            sizes = data['linker_mask'].sum(1).view(-1).int()               # what DDPM.sample_chain passes by default
        a = batching.create_templates_for_linker_generation(data, sizes)
        b = batching._create_templates_per_molecule(data, sizes)
        assert list(a.keys()) == list(b.keys())
        for k in a:
            if torch.is_tensor(a[k]):
                assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape and torch.equal(a[k], b[k]), k
            else:
                assert a[k] == b[k], k


def test_draw_noise_follows_the_reference_call_order():
    """edm.py:328-340 / utils.py:189-192: per draw randn(B,N,3) then randn(B,N,F); same seed -> same stream."""
    spec = synthetic.SPECS["cfg1_plumbing"]
    ddpm, hp = helpers.build_ddpm(spec, 0)
    g = torch.Generator().manual_seed(1000)
    got = ddpm.edm.draw_noise(7, 4, 30, torch.device('cpu'), generator=g)
    assert torch.equal(got, helpers.noise_tensor(1000, 5, 4, 30, spec.F))


def test_header_is_plain_c_and_a_c_program_links_against_the_library(tmp_path):
    """The drop-in boundary is a C ABI: include/difflinker_b200.h must compile as strict C99 (and C++), and a C program that
    only includes the header links against libdifflinker_b200.so and reaches the version / error entry points."""
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    lib = _native.LIB_PATH
    _native.load_library()
    src = tmp_path / "abi.c"
    src.write_text(
        '#include <stdio.h>\n#include "difflinker_b200.h"\n'
        "int main(void) {\n"
        "  dl_config c; dl_sizegnn_config s; dl_engine* e = 0; dl_status st;\n"
        "  (void)s; if (sizeof(dl_step_coef) != 32) return 2;\n"
        "  c.n_dims = 3; c.in_node_nf = 8; c.context_node_nf = 1; c.hidden_nf = 64; c.n_layers = 1; c.inv_sublayers = 1;\n"
        "  c.condition_time = 1; c.centering = 0; c.graph_type = DL_GRAPH_FC; c.device = 0; c.edge_impl = DL_EDGE_AUTO;\n"
        "  c.norm_constant = 0.f; c.normalization_factor = 1.f;\n"
        "  st = dl_create(&c, &e);            /* hidden_nf = 64 is refused before any CUDA call */\n"
        '  printf("%s|%d|%s\\n", dl_version(), (int)st, dl_last_error());\n'
        "  return st < 0 ? 0 : 3;\n}\n")
    exe = tmp_path / "abi"
    inc = os.path.join(ROOT, "include")
    subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", f"-I{inc}", str(src), "-o", str(exe), lib,
                    f"-Wl,-rpath,{os.path.dirname(lib)}"], check=True, capture_output=True)
    res = subprocess.run([str(exe)], capture_output=True, text=True)
    assert res.returncode == 0, (res.stdout, res.stderr)
    version, status, err = res.stdout.strip().split("|", 2)
    assert version.startswith("difflinker_b200") and int(status) < 0 and "hidden_nf" in err


def test_bench_reference_arm_contract_on_cpu():
    """`bench.py --impl reference` (the reference's CPU path: its own staged `src.egnn.Dynamics.forward` when oracle/_ref/ exists
    -- oracle/build_ref.py -- else the oracle port) prints ONE JSON line with the contract's keys; it needs no GPU, so the
    arm itself is checked here on the plumbing config."""
    import json
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg1_plumbing",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "molecules/s" and d["value"] > 0 and d["higher_is_better"] is True
    staged = os.path.isfile(os.path.join(ROOT, "oracle", "_ref", "src", "egnn.py"))
    assert d["config"]["workload"] == "cfg1_plumbing" and d["cpu_baseline"]["kind"] == ("reference" if staged else "port")
    if staged:
        assert d["cpu_baseline"]["port_value"] > 0
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_bench_clock_sampler_keeps_the_samples_of_the_timed_region(tmp_path):
    """bench.py's nvidia-smi sampler runs from before the warm-up; `stop()` must report only the samples whose timestamps fall
    between mark_begin() and mark_end() (the timed steps), and the throttle reasons seen there."""
    import datetime, importlib.util, time
    spec_ = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec_)
    spec_.loader.exec_module(bench)
    s = bench.ClockSampler(0)
    t0 = time.time()
    fmt = lambda t: datetime.datetime.fromtimestamp(t).strftime("%Y/%m/%d %H:%M:%S.%f")[:-3]
    rows = [(t0 - 3.0, 1200, "Not Active", "Not Active"), (t0 - 2.8, 1300, "Not Active", "Active"),      # warm-up: ignored
            (t0 + 0.1, 1965, "Not Active", "Not Active"), (t0 + 0.3, 1950, "Not Active", "Active"),
            (t0 + 0.5, 1965, "Not Active", "Not Active"), (t0 + 5.0, 900, "Active", "Not Active")]       # after the end: ignored
    path = tmp_path / "clocks.csv"
    path.write_text("".join(f"{fmt(t)}, 0, {clk}, 1965, 700.00, {hw}, Not Active, Not Active, {cap}\n" for t, clk, hw, cap in rows)
                    + "garbage line\n")

    class Done:
        def terminate(self): pass
        def wait(self, timeout=None): return 0
    s.proc, s.path, s.out = Done(), str(path), open(os.devnull, "w")
    s.t_begin, s.t_end = t0, t0 + 1.0
    got = s.stop()
    assert got == {"sm_mhz": 1965.0, "sm_max_mhz": 1965.0, "reasons": ["sw_power_cap"], "samples": 3, "samples_outside_timed_region": 3}
    assert not path.exists()


def test_plain_c_caller_builds_and_refuses_to_run_without_a_gpu(tmp_path):
    """examples/c_sampler.c -- a C99 program that samples through the C-ABI with device-side noise (`dl_sample_chain_rng`) from a job
    file written by difflinker_b200/export_job.py -- compiles warning-free against include/difflinker_b200.h, links against the
    in-tree library, and without a B200 fails loudly at dl_create (no CPU fallback). The GPU suite runs it for real."""
    from difflinker_b200 import export_job
    from difflinker_b200.batching import collate
    from difflinker_b200.ddpm import sampler_inputs
    _native.load_library()
    spec = synthetic.SPECS["cfg1_plumbing"]
    ddpm, hp = helpers.build_ddpm(spec, 0)
    ddpm.edm.T = 6
    kw = sampler_inputs(ddpm, collate(synthetic.make_items(spec)))
    job = str(tmp_path / "job.bin")
    meta = export_job.write_job(job, ddpm.edm, **kw, keep_frames=2, seed=1234)
    n_w = sum(p.numel() for p in ddpm.edm.dynamics.dynamics.state_dict().values())
    assert meta == {"B": 4, "N": 30, "T": 6, "keep_frames": 2, "xd": 3 + spec.F} and os.path.getsize(job) > 4 * n_w
    exe = helpers.build_c_example(tmp_path)
    res = subprocess.run([exe, job, str(tmp_path / "out.bin")], capture_output=True, text=True, timeout=300)
    if not torch.cuda.is_available():
        assert res.returncode == 2 and "dl_create" in res.stderr and not os.path.exists(tmp_path / "out.bin"), (res.stdout, res.stderr)
    else:
        assert res.returncode == 0, res.stderr


def test_load_from_checkpoint_reads_lightning_checkpoints(tmp_path):
    """generate.py:101 / :88 -- `DDPM.load_from_checkpoint(path, map_location)` and `SizeClassifier.load_from_checkpoint`
    on the Lightning checkpoint layout ({'hyper_parameters', 'state_dict', ...}), strict key match, overrides as kwargs."""
    from difflinker_b200 import DDPM, SizeClassifier
    spec = synthetic.SPECS["cfg1_plumbing"]
    m, hp = helpers.build_ddpm(spec, 0)
    path = str(tmp_path / "difflinker.ckpt")
    torch.save({"epoch": 3, "global_step": 7, "hyper_parameters": hp, "state_dict": m.state_dict()}, path)
    m2 = DDPM.load_from_checkpoint(path, map_location="cpu")
    assert list(m2.state_dict()) == list(m.state_dict())
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))
    assert m2.edm.T == hp['diffusion_steps'] and m2.inpainting is False
    assert DDPM.load_from_checkpoint(path, center_of_mass='anchors').center_of_mass == 'anchors'
    bad = dict(m.state_dict()); bad.pop(next(iter(bad)))
    torch.save({"hyper_parameters": hp, "state_dict": bad}, path)
    with pytest.raises(RuntimeError):
        DDPM.load_from_checkpoint(path)                                   # strict=True: a missing key is an error
    torch.save({"state_dict": m.state_dict()}, path)
    with pytest.raises(KeyError):
        DDPM.load_from_checkpoint(path)
    sc = SizeClassifier(in_node_nf=8, out_node_nf=10, n_layers=3, normalization='batch_norm')
    torch.save({"hyper_parameters": sc.hparams, "state_dict": sc.state_dict()}, path)
    sc2 = SizeClassifier.load_from_checkpoint(path)
    assert all(torch.equal(a, b) for a, b in zip(sc.state_dict().values(), sc2.state_dict().values()))
