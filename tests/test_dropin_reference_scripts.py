"""The UNEDITED reference scripts import and run on top of the dropin/ shims (SURVEY.md 8(b)).

cc_train_hypernet.py:10-28, train_hyper_combine.py:10-28 and test_hn.py:13-16 import ``models.decoderlstm``,
``models.encoder`` and ``hypernet_attention``; with dropin/ first on sys.path the first and last must resolve to the B200
classes while ``models.encoder`` keeps resolving to the reference's own file (dropin/models/__init__.py extends
``__path__``).  The first two tests need a checkout of the reference project (zacharie12/Hypernet-image-captioning, with
its data/vocab.pkl) named by $REFERENCE_DIR; this repository does not ship the reference, so they skip without one.
"""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("REFERENCE_DIR", "")
HAVE_REF = bool(REF) and os.path.isfile(os.path.join(REF, "cc_train_hypernet.py"))
needs_ref = pytest.mark.skipif(not HAVE_REF, reason="REFERENCE CHECKOUT ABSENT: set REFERENCE_DIR to a checkout of "
                                                    "zacharie12/Hypernet-image-captioning to import its unedited scripts")


def _drive(mode):
    res = subprocess.run([sys.executable, "-W", "ignore", os.path.join(ROOT, "tests", "dropin_ref_driver.py"), mode],
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    return json.loads(res.stdout.strip().splitlines()[-1])


@needs_ref
def test_reference_scripts_import_unedited_on_the_shims():
    out = _drive("cpu")
    assert out["HyperNet_cc"] and out["HyperNet_combine"] and out["HyperNet_test_hn"] and out["AttentionGru"]
    # models.encoder must be the REFERENCE's module (the shim package only replaces decoderlstm / attention)
    assert out["EncoderCNN_module"] == "models.encoder"
    assert out["EncoderCNN_file"] == os.path.realpath(os.path.join(REF, "models", "encoder.py"))
    # HyperNetCC(...) (cc_train_hypernet.py:43-108) builds OUR hypernet with he = #domains (one-hot)
    assert out["hypernet_is_ours"] and out["captioner_is_ours"] and out["he"] == 5
    # its unedited training_step (:134-160) reaches the CUDA path: on a CPU-only host that is a loud error, not a fallback
    assert out["training_step"] == "CaphnError", out


@needs_ref
@pytest.mark.gpu
def test_reference_training_step_through_the_shims_matches_oracle():
    """cc_train_hypernet.py:134-160 executed unedited (metric_score stubbed: nltk/datasets metrics are absent) on a
    synthetic batch; loss vs the oracle port on the same parameters."""
    out = _drive("gpu")
    assert out["hypernet_is_ours"]
    assert abs(out["loss"] - out["oracle_loss"]) <= 1e-4 * abs(out["oracle_loss"]), out
    assert out["head_grad_set"]


def test_launcher_orders_sys_path(tmp_path):
    """dropin/run_reference.py puts dropin/ ahead of the script's directory (plain ``python script.py`` cannot)."""
    (tmp_path / "hypernet_attention.py").write_text("HyperNet = 'reference'\n")
    (tmp_path / "models").mkdir()
    (tmp_path / "models" / "__init__.py").write_text("")
    (tmp_path / "models" / "encoder.py").write_text("EncoderCNN = 'reference encoder'\n")
    (tmp_path / "models" / "decoderlstm.py").write_text("AttentionGru = 'reference'\n")
    (tmp_path / "script.py").write_text(
        "from hypernet_attention import HyperNet\nfrom models.encoder import EncoderCNN\n"
        "from models.decoderlstm import AttentionGru\nimport os\n"
        "print(HyperNet.__name__, EncoderCNN, AttentionGru.__name__, os.path.basename(os.getcwd()))\n")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "dropin", "run_reference.py"), str(tmp_path / "script.py")],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    assert res.stdout.split() == ["HyperNetAttention", "reference", "encoder", "AttentionGru", tmp_path.name]
