"""The reference's import paths resolve to the B200-native modules through the overlay WITHOUT hiding
the rest of the reference package (losses, argument parsers, the other model families), and a
whole-module pickle written against those paths loads (README.md:75 `torch.load(model.pt)`).

The import block under test is the reference's own: dnn/experiments/run_improved_sudormrf.py:23-29
and utils/simple_whamr_evaluation.py:40-44 (minus the modules that need comet_ml / glob2 /
speechbrain).

The reference checkout is stood in for by a tree with its package layout (regular packages with empty
``__init__.py``), holding the modules that block imports, with placeholder contents: placeholders of the
accelerated modules that the overlay has to hide, and of the other modules that it must leave visible."""
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_PLACEHOLDER_MODEL = "class {0}:\n    '''placeholder: the overlay must resolve this name to sudo_rm_rf_b200'''\n"
STAND_IN = {
    "sudo_rm_rf/__init__.py": "",
    "sudo_rm_rf/dnn/__init__.py": "",
    "sudo_rm_rf/dnn/losses/__init__.py": "",
    "sudo_rm_rf/dnn/losses/sisdr.py": "class PermInvariantSISDR:\n    def __init__(self, **kwargs):\n        pass\n",
    "sudo_rm_rf/dnn/losses/snr.py": "class PermInvariantSNRwithZeroRefs:\n    pass\n",
    "sudo_rm_rf/dnn/models/__init__.py": "",
    "sudo_rm_rf/dnn/models/improved_sudormrf.py": _PLACEHOLDER_MODEL.format("SuDORMRF"),
    "sudo_rm_rf/dnn/models/groupcomm_sudormrf_v2.py": _PLACEHOLDER_MODEL.format("GroupCommSudoRmRf"),
    "sudo_rm_rf/dnn/models/causal_improved_sudormrf_v3.py": _PLACEHOLDER_MODEL.format("CausalSuDORMRF"),
    "sudo_rm_rf/dnn/models/sudormrf.py": _PLACEHOLDER_MODEL.format("SuDORMRF"),
    "sudo_rm_rf/dnn/experiments/__init__.py": "",
    "sudo_rm_rf/dnn/experiments/utils/__init__.py": "",
    "sudo_rm_rf/dnn/experiments/utils/improved_cmd_args_parser_v2.py": "def get_args():\n    return None\n",
    "sudo_rm_rf/dnn/experiments/utils/mixture_consistency.py": "def apply(pr_batch, input_mixture, mix_weights_type='uniform'):\n"
                                                                "    raise AssertionError('placeholder')\n",
}


@pytest.fixture(scope="module")
def reference(tmp_path_factory):
    """Root of a stand-in for the reference checkout."""
    root = tmp_path_factory.mktemp("reference")
    for rel, text in STAND_IN.items():
        path = root / rel
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_text(text)
    return str(root)

PICKLE = r"""
import io, sys, torch
sys.path.insert(0, {repo!r}); sys.path.insert(0, {repo!r} + "/sudo_rm_rf_b200/dropin")
import sudo_rm_rf.dnn.models.improved_sudormrf as improved_sudormrf
import sudo_rm_rf.dnn.models.groupcomm_sudormrf_v2 as sudormrf_gc_v2
import sudo_rm_rf.dnn.experiments.utils.mixture_consistency as mixture_consistency
import sudo_rm_rf_b200 as P
assert improved_sudormrf.SuDORMRF is P.SuDORMRF
assert sudormrf_gc_v2.GroupCommSudoRmRf is P.GroupCommSudoRmRf
assert mixture_consistency.apply is P.mixture_consistency.apply
m = improved_sudormrf.SuDORMRF(16, 32, 2, 3, 21, 24, 2)
m.__class__.__module__ = "sudo_rm_rf.dnn.models.improved_sudormrf"   # what a reference pickle records
buf = io.BytesIO(); torch.save(m, buf); buf.seek(0)
m2 = torch.load(buf, weights_only=False)
assert type(m2).__name__ == "SuDORMRF" and m2.enc_num_basis == 24
assert list(m2.state_dict().keys()) == list(m.state_dict().keys())
print("overlay ok")
"""

# sys.path order as the runner builds it: the overlay comes first (PYTHONPATH), the reference root is APPENDED
# by the script itself (run_improved_sudormrf.py:11-13) before its import block runs.
RUNNER_IMPORTS = r"""
import sys, warnings
warnings.simplefilter("ignore")
{setup}
import sudo_rm_rf.dnn.experiments.utils.improved_cmd_args_parser_v2 as parser      # run_improved_sudormrf.py:23
import sudo_rm_rf.dnn.losses.sisdr as sisdr_lib                                    # :25
import sudo_rm_rf.dnn.models.improved_sudormrf as improved_sudormrf                # :26
import sudo_rm_rf.dnn.models.sudormrf as initial_sudormrf                          # :27
import sudo_rm_rf.dnn.models.groupcomm_sudormrf_v2 as sudormrf_gc_v2               # simple_whamr_evaluation.py:41
import sudo_rm_rf.dnn.experiments.utils.mixture_consistency as mixture_consistency # :44
import sudo_rm_rf.dnn.models.causal_improved_sudormrf_v3 as causal                 # run_fuss_separation.py
import sudo_rm_rf.dnn.losses.snr as snr_lib
import sudo_rm_rf_b200 as P
ref = {reference!r}
# accelerated names -> this repo
assert improved_sudormrf.SuDORMRF is P.SuDORMRF, improved_sudormrf.__file__
assert sudormrf_gc_v2.GroupCommSudoRmRf is P.GroupCommSudoRmRf
assert mixture_consistency.apply is P.mixture_consistency.apply
assert causal.CausalSuDORMRF is P.CausalSuDORMRF
assert initial_sudormrf.SuDORMRF is P.OriginalSuDORMRF and initial_sudormrf.SuDORMRF is not P.SuDORMRF
# everything else -> the reference's own files
for mod in (parser, sisdr_lib, snr_lib):
    assert mod.__file__.startswith(ref), mod.__file__
# the objects the runner builds from them (run_improved_sudormrf.py:66-70,82-85,88-96)
loss = sisdr_lib.PermInvariantSISDR(batch_size=2, n_sources=2, zero_mean=True, backward_loss=False,
                                    improvement=True, return_individual_results=True)
model = improved_sudormrf.SuDORMRF(out_channels=16, in_channels=32, num_blocks=2, upsampling_depth=3,
                                   enc_kernel_size=21, enc_num_basis=24, num_sources=2)
assert sum(f.numel() for f in model.parameters() if f.requires_grad) > 0                # :111-114
assert parser.get_args.__module__.endswith("improved_cmd_args_parser_v2")
print("runner imports ok")
"""


def _run(script, cwd):
    out = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, cwd=cwd)
    assert out.returncode == 0, out.stderr[-3000:]
    return out.stdout


def test_overlay_import_paths_and_pickle(tmp_path):
    assert "overlay ok" in _run(PICKLE.format(repo=REPO), tmp_path)


def test_overlay_keeps_rest_of_reference_importable(reference, tmp_path):
    setup = (f"sys.path.insert(0, {REPO!r}); sys.path.insert(0, {REPO!r} + '/sudo_rm_rf_b200/dropin')\n"
             f"sys.path.append({reference!r})")
    assert "runner imports ok" in _run(RUNNER_IMPORTS.format(setup=setup, reference=reference), tmp_path)


def test_meta_path_redirect_with_reference_first(reference, tmp_path):
    """`sudo_rm_rf_b200.dropin.install()`: reference FIRST on sys.path, only the accelerated names are redirected."""
    setup = (f"sys.path.insert(0, {REPO!r}); sys.path.insert(0, {reference!r})\n"
             "import sudo_rm_rf_b200.dropin as D; D.install()")
    assert "runner imports ok" in _run(RUNNER_IMPORTS.format(setup=setup, reference=reference), tmp_path)


def test_overlay_without_reference_modules_fails_normally(reference, tmp_path):
    """A module neither the overlay nor the reference has is a plain ModuleNotFoundError."""
    script = (f"import sys; sys.path.insert(0, {REPO!r}); sys.path.insert(0, {REPO!r} + '/sudo_rm_rf_b200/dropin')\n"
              f"sys.path.append({reference!r})\n"
              "try:\n    import sudo_rm_rf.dnn.models.no_such_model\n"
              "except ModuleNotFoundError:\n    print('fine')\n")
    assert "fine" in _run(script, tmp_path)
