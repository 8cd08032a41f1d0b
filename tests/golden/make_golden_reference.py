"""Golden fixtures of the comparisons with the unmodified reference that used to need its checkout
at test time.  Needs a checkout of the reference (etzinis/sudo_rm_rf):

    python tests/golden/make_golden_reference.py --reference PATH/TO/sudo_rm_rf_checkout

* ``oracle_vs_reference.npz``: the reference models' forward on the seeded cases of
  ``tests/test_oracle_vs_reference.py`` (output, state_dict key order, input fingerprint).
* ``reference_sisdr.npz``: ``PermInvariantSISDR`` (dnn/losses/sisdr.py) on the seeded inputs of
  ``test_prepost_oracle.py::test_pit_sisdr_live_against_reference`` (best SI-SDRi + permutations), and on
  the oracle's estimates of the two validation batches of
  ``test_gpu_model.py::test_validation_loop_of_the_reference_runner``.
"""
import argparse
import json
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
REPO = os.path.dirname(TESTS)


def js(obj):
    return np.frombuffer(json.dumps(obj).encode(), dtype=np.uint8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True, help="root of the reference checkout (holds sudo_rm_rf/)")
    args = ap.parse_args()
    sys.path.insert(0, REPO)
    sys.path.insert(0, TESTS)
    sys.path.insert(0, os.path.abspath(args.reference))
    warnings.filterwarnings("ignore")
    import sudo_rm_rf.dnn.models.improved_sudormrf as ri
    import sudo_rm_rf.dnn.models.groupcomm_sudormrf_v2 as rg
    import sudo_rm_rf.dnn.models.causal_improved_sudormrf_v3 as rc
    import sudo_rm_rf.dnn.models.sudormrf as ro
    import sudo_rm_rf.dnn.losses.sisdr as rs
    from oracle import sudormrf_oracle as O
    import test_oracle_vs_reference as TV
    import test_prepost_oracle as TP
    classes = {"improved": ri.SuDORMRF, "groupcomm": rg.GroupCommSudoRmRf, "causal": rc.CausalSuDORMRF,
               "original": ro.SuDORMRF}

    out = {}
    for ci, (variant, kw, T) in enumerate(TV.CASES):
        cfg, sd, x = TV.case_inputs(variant, kw, T)
        m = classes[variant](**kw).eval()
        m.load_state_dict(sd)
        with torch.no_grad():
            y = m(x)
        out[f"c{ci}/meta"] = js(dict(variant=variant, kwargs=kw, T=T))
        out[f"c{ci}/keys"] = js(list(m.state_dict().keys()))
        out[f"c{ci}/fingerprint"] = TV.fingerprint(sd, x)
        out[f"c{ci}/out"] = y.numpy().astype(np.float32)
    np.savez_compressed(os.path.join(HERE, "oracle_vs_reference.npz"), **out)

    out = {}
    est, tgt, mix = TP.pit_live_inputs()
    fn = rs.PermInvariantSISDR(batch_size=6, zero_mean=True, n_sources=3, backward_loss=False,
                               improvement=True, return_individual_results=True)
    best, perms = fn(est, tgt, initial_mixtures=mix, return_best_permutation=True)
    out["pit_live/fingerprint"] = np.array([float(est.double().sum()), float(tgt.double().sum())])
    out["pit_live/best"] = best.numpy().astype(np.float32)
    out["pit_live/perms"] = np.array([[int(v) for v in r] for r in perms], dtype=np.int64)

    # the validation half of run_improved_sudormrf.py, as the GPU test runs it (improved model, weights seed 9)
    kw = dict(out_channels=64, in_channels=128, num_blocks=2, upsampling_depth=4,
              enc_kernel_size=21, enc_num_basis=64, num_sources=2)
    cfg = O.Config(variant="improved", **kw)
    sd = O.make_state_dict(cfg, seed=9)
    fn = rs.PermInvariantSISDR(batch_size=4, n_sources=2, zero_mean=True, backward_loss=False, improvement=True,
                               return_individual_results=True)
    g = torch.Generator().manual_seed(3)
    losses = []
    with torch.no_grad():
        for _ in range(2):
            clean = torch.randn(4, 2, 8000, generator=g)
            m1wavs = clean.sum(1)
            m1wavs = (m1wavs - m1wavs.mean(-1, keepdim=True)) / (m1wavs.std(-1, keepdim=True) + 1e-9)
            rec = O.forward(cfg, sd, m1wavs.unsqueeze(1))
            losses += fn(rec, clean, initial_mixtures=m1wavs.unsqueeze(1)).tolist()
    out["runner_val/loss"] = np.array(losses, dtype=np.float32)
    np.savez_compressed(os.path.join(HERE, "reference_sisdr.npz"), **out)


if __name__ == "__main__":
    main()
