"""CPU: the C-ABI library loads and exports every symbol include/aotb200.h declares; host-side
logic that needs no GPU (config mirror, overlay resolution, loud failure without CUDA)."""
import ctypes
import os
import subprocess
import sys

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cuobjdump(*args):
    """cuobjdump of the toolkit whose nvcc built the library (found next to it, not on PATH)."""
    from aot_benchmark_b200.build import NVCC
    return subprocess.run([os.path.join(os.path.dirname(NVCC), "cuobjdump"), *args], capture_output=True, text=True)


def test_library_exports_every_declared_symbol():
    from aot_benchmark_b200 import _lib
    decl = _lib.parse_header()
    assert len(decl) >= 20
    assert os.path.exists(_lib.LIB_PATH), "run __graft_entry__.build() first"
    h = ctypes.CDLL(_lib.LIB_PATH)
    for name in decl:
        assert hasattr(h, name), f"{name} declared in include/aotb200.h but not exported"
    L = _lib.lib()
    assert L.aotb_version() >= 100 and L.aotb_arch() == b"sm_100a"


def test_sass_is_sm100a_only():
    from aot_benchmark_b200 import _lib
    r = _cuobjdump("-lelf", _lib.LIB_PATH)
    if r.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    archs = {l.split(".")[-2] for l in r.stdout.splitlines() if "sm_" in l}
    assert archs == {"sm_100a"}, archs


def test_no_cpu_path():
    from aot_benchmark_b200 import EngineConfig, build_engine, build_vos_model
    cfg = EngineConfig("t", "aott")
    model = build_vos_model(cfg.MODEL_VOS, cfg).eval()
    eng = build_engine(cfg.MODEL_ENGINE, phase="eval", aot_model=model, gpu_id=-1)
    with pytest.raises(RuntimeError):
        eng.add_reference_frame(torch.zeros(1, 3, 65, 65), torch.zeros(1, 1, 65, 65), obj_nums=[1], frame_step=0)
    with pytest.raises(RuntimeError):
        model(torch.zeros(1, 3, 65, 65))
    with pytest.raises(NotImplementedError):
        eng.aot_engines and None
        build_engine(cfg.MODEL_ENGINE, phase="train", aot_model=model).forward()


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: nothing under aot_benchmark_b200/ may import it."""
    bad = []
    for root, _, files in os.walk(os.path.join(REPO, "aot_benchmark_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(root, f)).read()
                if "import oracle" in src or "from oracle" in src:
                    bad.append(f)
    assert not bad, bad


def test_separate_mask_matches_reference_semantics(monkeypatch):
    """Host logic of AOTInferEngine.separate_mask (object counts per sub-engine) with the label kernel emulated on CPU; the
    kernel itself is checked on the GPU (tests/test_gpu_ops.py)."""
    sys.path.insert(0, os.path.join(REPO, "tests"))
    import emu_ops
    emu_ops.install_engine(monkeypatch)
    from aot_benchmark_b200 import EngineConfig, build_engine, build_vos_model
    cfg = EngineConfig("t", "aott")
    eng = build_engine(cfg.MODEL_ENGINE, phase="eval", aot_model=build_vos_model(cfg.MODEL_VOS, cfg))
    eng.aot_engines = [object(), object(), object()]
    mask = torch.arange(0, 26).float().view(1, 1, 2, 13)
    ms, nums = eng.separate_mask(mask, 25)
    assert nums == [10, 10, 5]
    assert ms[0].max() == 10 and ms[1].max() == 10 and ms[2].max() == 5
    assert torch.equal(ms[1][0, 0].flatten()[11:21], torch.arange(1, 11).float())
    eng.aot_engines = []


def test_overlay_resolves_in_front_of_reference(golden_dir, tmp_path):
    """The overlay in front of a reference checkout (a stand-in with the reference's recorded `networks` layout and imports):
    engines and models resolve to this package, everything else -- and the evaluator's own imports -- to the checkout."""
    from oracle.fixtures import load_reference_contract, write_reference_standin
    ref = str(tmp_path / "reference")
    write_reference_standin(ref, load_reference_contract(golden_dir)["networks"])
    code = ("import sys; sys.path[:0]=[%r, %r, %r];"
            "from networks.engines import build_engine; from networks.models import build_vos_model;"
            "import networks.layers.attention as A; import networks.managers.evaluator as E;"
            "assert build_engine.__module__=='aot_benchmark_b200.engine';"
            "assert build_vos_model.__module__=='aot_benchmark_b200.model';"
            "assert E.build_engine is build_engine and E.build_vos_model is build_vos_model;"
            "assert A.__file__.startswith(%r); print('OK')") % (
                REPO, os.path.join(REPO, "aot_benchmark_b200", "overlay"), ref, ref)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=str(tmp_path))
    assert "OK" in r.stdout, r.stderr[-1500:]


def test_every_ops_attribute_used_by_the_engine_exists():
    """Static check (no GPU here): every `ops.<name>` / `engine_mod.<name>` referenced by the engine, the bench and
    the entry points exists -- a missing wrapper must fail on the CPU box, not on a GPU trip."""
    import ast
    from aot_benchmark_b200 import engine, ops
    for path, aliases in ((os.path.join(REPO, "aot_benchmark_b200", "engine.py"), {"ops": ops}),
                          (os.path.join(REPO, "bench.py"), {"ops": ops, "engine_mod": engine}),
                          (os.path.join(REPO, "__graft_entry__.py"), {})):
        tree = ast.parse(open(path).read())
        for node in ast.walk(tree):
            if isinstance(node, ast.Attribute) and isinstance(node.value, ast.Name) and node.value.id in aliases:
                assert hasattr(aliases[node.value.id], node.attr), f"{path}: {node.value.id}.{node.attr} does not exist"


def test_every_ops_wrapper_binds_a_declared_symbol():
    import ast
    import inspect
    from aot_benchmark_b200 import _lib, ops
    decl = set(_lib.parse_header())
    src = inspect.getsource(ops)
    used = set()
    for node in ast.walk(ast.parse(src)):
        if isinstance(node, ast.Attribute) and node.attr.startswith("aotb_"):
            used.add(node.attr)
    assert used <= decl, used - decl


def test_kernel_register_budgets_fit_their_block_sizes():
    """A kernel whose registers x threads exceed the 64K register file (allocation granularity: 4 warps) fails at launch
    with 'too many resources requested' -- catch that here, without a GPU, from the cubin resource usage."""
    import re
    from aot_benchmark_b200 import _lib
    r = _cuobjdump("-res-usage", _lib.LIB_PATH)
    if r.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    blocks = {"lt_attn_tc_kernel": 576, "lt_attn_tc3_kernel": 576, "gp_attn_tc_kernel": 608, "conv_tc_kernel": 320, "local_attn_tile_kernel": 512,
              "conv_igemm_kernel": 256, "attn_f32_kernel": 256, "local_attn_kernel": 256, "window_attn_kernel": 64}
    cur, seen = None, 0
    for line in r.stdout.splitlines():
        m = re.search(r"Function (\S+):", line)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r"REG:(\d+)", line)
        if m and cur:
            regs = int(m.group(1))
            for name, threads in blocks.items():
                if name in cur:
                    warps = (threads + 31) // 32
                    warps4 = (warps + 3) // 4 * 4
                    assert regs * 32 * warps4 <= 65536, f"{cur}: {regs} regs x {threads} threads does not fit"
                    seen += 1
    assert seen >= 9
