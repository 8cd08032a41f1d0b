"""Pins the oracle's restatement of the steps either side of the forward (SURVEY 8f rows 1-2:
the README inference recipe and the PIT SI-SDR metric) against golden vectors produced by the
unmodified reference (tests/golden/make_golden_prepost.py).  CPU only."""
import glob
import itertools
import json
import os

import numpy as np
import pytest
import torch

from oracle import sudormrf_oracle as O

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SEPARATE = sorted(glob.glob(os.path.join(GOLDEN_DIR, "prepost_separate_*.npz")))


def load_separate(path):
    z = np.load(path)
    meta = json.loads(bytes(z["meta"]).decode())
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd/")}
    return meta, sd, torch.from_numpy(z["wav"]), torch.from_numpy(z["out/plain"]), torch.from_numpy(z["out/mc"])


def load_sisdr():
    z = np.load(os.path.join(GOLDEN_DIR, "prepost_sisdr.npz"))
    meta = json.loads(bytes(z["meta"]).decode())
    out = []
    for ci, c in enumerate(meta["cases"]):
        k = f"c{ci}/"
        out.append((c, {n: torch.from_numpy(z[k + n]) for n in ("est", "tgt", "mix", "best", "perms", "loss")}))
    return out


@pytest.mark.parametrize("path", SEPARATE, ids=lambda p: os.path.basename(p)[17:-4])
def test_separate_matches_reference_golden(path):
    meta, sd, wav, plain, with_mc = load_separate(path)
    cfg = O.Config(variant=meta["variant"], **meta["kwargs"])
    got = O.separate(cfg, sd, wav, apply_mixture_consistency=False)
    assert got.shape == plain.shape
    assert max(O.parity_errors(got, plain)) < 2e-5
    got = O.separate(cfg, sd, wav, apply_mixture_consistency=True)
    assert max(O.parity_errors(got, with_mc)) < 2e-5


def test_separate_fixture_is_not_trivial():
    """The raw mixtures carry a per-utterance gain and DC offset, so a missing rescale is visible."""
    meta, sd, wav, plain, with_mc = load_separate(SEPARATE[0])
    assert float(wav.mean(-1).abs().max()) > 0.3 and float(wav.std(-1).max() / wav.std(-1).min()) > 10
    cfg = O.Config(variant=meta["variant"], **meta["kwargs"])
    raw = O.forward(cfg, sd, wav.unsqueeze(1))
    assert max(O.parity_errors(raw, plain)) > 1e-2


@pytest.mark.parametrize("ci", range(6))
def test_pit_sisdr_matches_reference_golden(ci):
    c, t = load_sisdr()[ci]
    best, idx = O.pit_sisdr(t["est"], t["tgt"], t["mix"], zero_mean=c["zero_mean"],
                            improvement=c["improvement"])
    assert torch.allclose(best, t["best"], atol=1e-4, rtol=0)
    perms = list(itertools.permutations(range(c["S"])))
    assert [perms[int(i)] for i in idx] == [tuple(int(v) for v in row) for row in t["perms"]]
    # backward_loss=True, return_individual_results=False: the negated batch mean (sisdr.py:150-154)
    assert torch.allclose(-best.mean(), t["loss"][0], atol=1e-4, rtol=0)


def pit_live_inputs():
    """Seeded (estimates, targets, mixtures): 6 items, 3 sources, estimates a permutation of the targets + noise."""
    g = torch.Generator().manual_seed(5)
    tgt = torch.randn(6, 3, 3000, generator=g)
    est = tgt[:, [2, 0, 1]] + 0.3 * torch.randn(6, 3, 3000, generator=g)
    mix = tgt.sum(1, keepdim=True)
    return est, tgt, mix


def test_pit_sisdr_live_against_reference():
    """The reference's PermInvariantSISDR(zero_mean, improvement, return_best_permutation) on these seeded inputs,
    stored by golden/make_golden_reference.py."""
    est, tgt, mix = pit_live_inputs()
    z = np.load(os.path.join(GOLDEN_DIR, "reference_sisdr.npz"))
    np.testing.assert_allclose([float(est.double().sum()), float(tgt.double().sum())], z["pit_live/fingerprint"],
                               rtol=1e-12)
    want, perms = torch.from_numpy(z["pit_live/best"]), z["pit_live/perms"]
    best, idx = O.pit_sisdr(est, tgt, mix, zero_mean=True, improvement=True)
    assert torch.allclose(best, want, atol=1e-5, rtol=0)
    allp = list(itertools.permutations(range(3)))
    assert [allp[int(i)] for i in idx] == [tuple(int(v) for v in r) for r in perms]


def load_pairwise():
    z = np.load(os.path.join(GOLDEN_DIR, "prepost_pairwise.npz"))
    cases = []
    ci = 0
    while f"c{ci}/meta" in z.files:
        meta = json.loads(bytes(z[f"c{ci}/meta"]).decode())
        si = meta["signals"]
        cases.append((meta, dict(est=torch.from_numpy(z[f"s{si}/est"]), tgt=torch.from_numpy(z[f"s{si}/tgt"]),
                                 pw=torch.from_numpy(z[f"c{ci}/pw"]), pit_loss=torch.from_numpy(z[f"c{ci}/pit_loss"]))))
        ci += 1
    return cases


def test_pairwise_neg_sdr_matches_reference_golden():
    """The oracle restatement of PairwiseNegSDR / PITLossWrapper.find_best_perm against reference-generated goldens
    (tests/golden/make_golden_prepost.py::make_pairwise): 4 signal sets x 3 sdr types x 3 flag combinations."""
    cases = load_pairwise()
    assert len(cases) == 36
    for meta, t in cases:
        pw = O.pairwise_neg_sdr(t["est"], t["tgt"], meta["sdr_type"], meta["zero_mean"], meta["take_log"])
        assert torch.equal(pw, t["pw"]), meta               # same torch op sequence: bit-exact
        loss, _ = O.pit_from_pairwise(pw)
        assert torch.allclose(loss.mean(), t["pit_loss"], rtol=1e-6, atol=1e-6), meta


def load_stabilized():
    z = np.load(os.path.join(GOLDEN_DIR, "prepost_stabilized.npz"))
    meta = json.loads(bytes(z["meta"]).decode())
    return [(c, {n: torch.from_numpy(z[f"c{ci}/" + n]) for n in ("est", "tgt", "best", "perms", "loss")})
            for ci, c in enumerate(meta["cases"])]


@pytest.mark.parametrize("ci", range(8))
def test_stabilized_sisdr_matches_reference_golden(ci):
    """StabilizedPermInvSISDRMetric (sisdr.py:460-591): more estimated than actual sources, single_source, SI-SDRi."""
    c, t = load_stabilized()[ci]
    best, idx = O.stabilized_pit_sisdr(t["est"], t["tgt"], zero_mean=c["zero_mean"], single_source=c["single_source"],
                                       improvement=c["improvement"])
    assert torch.allclose(best, t["best"], atol=1e-4, rtol=0)
    n_est = 1 if c["single_source"] else c["n_est"]
    perms = list(itertools.permutations(range(n_est), r=c["n_act"]))
    assert [perms[int(i)] for i in idx] == [tuple(int(v) for v in row) for row in t["perms"]]
    assert torch.allclose(-best.mean(), t["loss"][0], atol=1e-4, rtol=0)
