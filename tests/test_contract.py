"""Repo-level contract checks that need no GPU: the product path never touches the oracle, the library refuses to run
without its CUDA extension, and the `bench.py --impl reference` line has the shape the driver parses."""
import ast
import importlib
import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _python_files(*dirs):
    for d in dirs:
        for base, _, files in os.walk(os.path.join(ROOT, d)):
            if "__pycache__" in base:
                continue
            for f in files:
                if f.endswith(".py"):
                    yield os.path.join(base, f)


def _imported_modules(path):
    tree = ast.parse(open(path).read(), path)
    for node in ast.walk(tree):
        if isinstance(node, ast.Import):
            for a in node.names:
                yield a.name
        elif isinstance(node, ast.ImportFrom):
            yield ("." * node.level) + (node.module or "")


def test_product_path_never_imports_the_oracle():
    """oracle/ is test infrastructure: only tests/, __graft_entry__.smoke() and bench.py's baseline legs may import it.
    The package and the drop-in shims must not -- neither by import statement nor by loading a file from oracle/."""
    offenders = []
    for path in _python_files("hypernet_image_captioning_b200", "dropin"):
        mods = list(_imported_modules(path))
        if any(m == "oracle" or m.startswith("oracle.") for m in mods):
            offenders.append(path)
    assert not offenders, offenders


def test_bench_confines_the_oracle_to_the_baseline_legs():
    """bench.py may execute the oracle in the CPU baseline / reference arm (and the torch-eager-GPU comparison column,
    which is a baseline too) -- never at module level and never inside run_ours' timed step."""
    path = os.path.join(ROOT, "bench.py")
    tree = ast.parse(open(path).read(), path)
    allowed = {"cpu_reference_arm", "torch_eager_gpu_arm"}
    for node in tree.body:
        if isinstance(node, (ast.Import, ast.ImportFrom)):
            names = [a.name for a in node.names] if isinstance(node, ast.Import) else [node.module or ""]
            assert not any(n.split(".")[0] == "oracle" for n in names), "module-level oracle import in bench.py"
        if isinstance(node, ast.FunctionDef):
            uses = any(isinstance(n, ast.ImportFrom) and (n.module or "").split(".")[0] == "oracle"
                       or isinstance(n, ast.Import) and any(a.name.split(".")[0] == "oracle" for a in n.names)
                       for n in ast.walk(node))
            assert not uses or node.name in allowed, f"bench.py:{node.name} imports the oracle"


def test_missing_extension_fails_loudly(monkeypatch, tmp_path):
    """No CPU fallback: with the shared library absent, loading raises instead of degrading to torch ops."""
    from hypernet_image_captioning_b200 import _cabi, build

    def no_nvcc(*a, **k):
        raise RuntimeError("nvcc not found")

    monkeypatch.setattr(_cabi, "LIB_PATH", str(tmp_path / "libcaphn_b200.so"))
    monkeypatch.setattr(_cabi, "_lib", None)
    monkeypatch.setattr(build, "build", no_nvcc)
    with pytest.raises(_cabi.CaphnError):
        _cabi.load()
    (tmp_path / "libcaphn_b200.so").write_bytes(b"not an ELF file")        # present but unusable: loud as well
    with pytest.raises(_cabi.CaphnError):
        _cabi.load()


def _bench():
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    return importlib.import_module("bench")


class _Args:
    gpus, steps, warmup, batch, impl = 1, 20, 5, 512, "reference"


def _fake_arm(steps, warmup, B=512):
    return {"value": 900.0, "unit": "captions/s", "cores": 16, "kind": "port", "sample": "fake", "ms_per_step": 568.9}


def test_reference_arm_line_has_the_contract_keys(monkeypatch, capsys):
    bench = _bench()
    monkeypatch.setattr(bench, "cpu_reference_arm", _fake_arm)
    monkeypatch.setenv("RANK", "0")
    args = _Args()
    bench.run_reference(args)
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["metric"] == "hypernet-GRU train captions/s" and line["unit"] == "captions/s"
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "captions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0
    # same `config` as our arm prints for the same command line (the driver compares them)
    assert line["config"] == bench.workload_config(args, args.gpus)


def test_dump_outputs_writes_float32_samples_at_fixed_positions(tmp_path):
    """bench.py --dump-outputs: loss, logits rows and every parameter gradient as float32 .npy; arrays larger than the
    per-array budget are sampled at positions that depend on the array's name only, so two runs write the same entries."""
    import numpy as np
    import torch
    bench = _bench()
    torch.manual_seed(0)
    model = torch.nn.Linear(300, 2000)                       # weight: 600 000 entries, more than DUMP_GRAD_ENTRIES
    (model(torch.randn(4, 300)) * torch.randn(4, 2000)).sum().backward()
    loss, logits = torch.tensor(2.5), torch.randn(8, 5, 97)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), loss, logits, model)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["grad.bias.npy", "grad.weight.npy", "logits_rows.npy", "loss.npy"]
    got = {n: np.load(tmp_path / "a" / n) for n in names}
    assert all(v.dtype == np.float32 for v in got.values())
    assert all(np.array_equal(v, np.load(tmp_path / "b" / n)) for n, v in got.items())
    assert got["loss.npy"].tolist() == [2.5]
    assert np.array_equal(got["logits_rows.npy"], logits.reshape(40, 97).numpy())         # 40 rows: all of them
    assert np.array_equal(got["grad.bias.npy"], model.bias.grad.numpy())
    w = got["grad.weight.npy"]
    assert w.shape == (bench.DUMP_GRAD_ENTRIES,) and np.isin(w, model.weight.grad.numpy()).all()


def test_reference_arm_uses_our_arms_config_at_n_gpus_and_only_rank0_prints(monkeypatch, capsys):
    bench = _bench()
    monkeypatch.setattr(bench, "cpu_reference_arm", _fake_arm)
    args = _Args()
    args.gpus = 8
    monkeypatch.setenv("RANK", "3")
    bench.run_reference(args)
    assert capsys.readouterr().out == ""
    monkeypatch.setenv("RANK", "0")
    bench.run_reference(args)
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["n_gpus"] == 8 and line["config"]["parallelism"] == "dp8" and line["config"]["global_batch"] == 8 * 512
