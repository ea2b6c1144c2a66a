"""CPU tests of the host-side model compiler (nanosim_b200/model.py) against the oracle's own parsing/sampling."""
import os
import random
import sys

import numpy as np
import pytest

from conftest import DATA, oracle_model

import nanosim_oracle as no
from nanosim_b200 import model as M
from parity_checks import chi2_two_sample

CASES = ["guppy", "dorado"]


def _oracle_pmf(items):
    """Exact pmf of the oracle's interval sampler (all interval bounds are integers in shipped models)."""
    vmax = int(max(x[3] for x in items))
    pmf = np.zeros(vmax + 1)
    covered = 0.0
    for clo, chi, vlo, vhi in items:
        assert float(vlo).is_integer() and float(vhi).is_integer()
        n = int(vhi - vlo)
        covered += chi - clo
        if n == 0:
            pmf[int(vlo)] += chi - clo
        for s in range(int(vlo), int(vhi)):
            pmf[s] += (chi - clo) / n
    return pmf, covered


@pytest.mark.parametrize("tag", CASES)
def test_ecdf_pmfs_match_oracle_intervals(tag, compiled_models, tmp_path):
    cm = compiled_models[tag]
    om = oracle_model(cm, tmp_path, fastq=True)
    t = M.DeviceTables(cm, fastq=True)
    assert [tuple(b) for b in t.match_bins] == list(om.match_markov.keys())
    for b, pm in zip(om.match_markov.keys(), t.match_pmf):
        ref, covered = _oracle_pmf(om.match_markov[b])
        body = pm[:-1]
        assert len(body) == len(ref)
        np.testing.assert_allclose(body / body.sum(), ref / ref.sum(), atol=1e-13)
        # the miss slot is what the intervals leave uncovered
        assert abs(pm[-1] - max(0.0, 1.0 - covered)) < 1e-9
    fm_ref, _ = _oracle_pmf(om.first_match[list(om.first_match.keys())[0]])
    fm_ref[2] += fm_ref[0] + fm_ref[1]
    fm_ref[0] = fm_ref[1] = 0
    np.testing.assert_allclose(t.pmfs[M.T_FIRST][:len(fm_ref)], fm_ref / fm_ref.sum(), atol=1e-9)


@pytest.mark.parametrize("tag", CASES)
def test_alias_tables_realise_pmfs(tag, compiled_models):
    t = M.DeviceTables(compiled_models[tag], fastq=True)
    for i, pm in enumerate(t.pmfs):
        off, n = (int(x) for x in t.alias_desc[i])
        assert n == len(pm)
        got = M.alias_pmf(t.alias_prob[off:off + n], t.alias_idx[off:off + n])
        np.testing.assert_allclose(got, pm / pm.sum(), atol=2e-9)
        assert (t.alias_idx[off:off + n] < n).all()


@pytest.mark.parametrize("tag", CASES)
def test_error_length_pmfs_vs_oracle_sampling(tag, compiled_models, tmp_path):
    cm = compiled_models[tag]
    om = oracle_model(cm, tmp_path, fastq=True)
    t = M.DeviceTables(cm, fastq=True)
    n = 200000
    np.random.seed(5)
    random.seed(5)
    p = om.error_par["mis"]
    draws = {"mis": [no.pois_geom(p[0], p[2], p[3]) for _ in range(n)],
             "ins": [no.wei_geom(*om.error_par["ins"]) for _ in range(n)],
             "del": [no.wei_geom(*om.error_par["del"]) for _ in range(n)]}
    for tid, k in ((M.T_MIS, "mis"), (M.T_INS, "ins"), (M.T_DEL, "del")):
        pm = t.pmfs[tid]
        assert pm[0] == 0.0 and abs(pm.sum() - 1) < 1e-12
        emp = np.bincount(np.minimum(draws[k], len(pm) - 1), minlength=len(pm)).astype(float)
        stat, dof, pval = chi2_two_sample(emp, pm * 1e9)
        assert pval > 1e-4, (k, stat, dof, pval)


@pytest.mark.parametrize("tag", CASES)
def test_quality_pmf_vs_oracle_sampling(tag, compiled_models, tmp_path):
    cm = compiled_models[tag]
    om = oracle_model(cm, tmp_path, fastq=True)
    t = M.DeviceTables(cm, fastq=True)
    np.random.seed(9)
    for i, st in enumerate(M.QUAL_STATES):
        q = np.asarray(no.base_qualities(om.base_qual[st], 300000))
        assert q.min() >= 1 and q.max() <= 93
        emp = np.bincount(q, minlength=94).astype(float)
        stat, dof, pval = chi2_two_sample(emp, t.qual_pmf[i] * 1e10)
        assert pval > 1e-4, (st, stat, dof, pval)
        cdf = t.qual_cdf[i].astype(np.float64) / 2 ** 32
        np.testing.assert_allclose(np.diff(np.concatenate([[0], cdf])), t.qual_pmf[i], atol=1e-9)


@pytest.mark.parametrize("tag", CASES)
def test_transition_thresholds_and_counts(tag, compiled_models, tmp_path):
    cm = compiled_models[tag]
    om = oracle_model(cm, tmp_path, fastq=True)
    t = M.DeviceTables(cm, fastq=True)
    for i, st in enumerate(M.ERR_STATES):
        (a, b), (c, d), (e, f) = [iv for iv, _ in om.trans_error_pr[st]]
        assert abs(t.trans[i, 0] / 2 ** 32 - b) < 1e-9
        assert abs(t.trans[i, 1] / 2 ** 32 - d) < 1e-9
        assert abs(t.trans[i, 2] / 2 ** 32 - e) < 1e-9
    for n in (1000, 20000, 12345):
        assert t.split_counts(n) == om.split_counts(n)
    assert abs(t.strandness - om.strandness_rate) < 1e-7
    assert t.mean_ref_per_event > 1.0


def test_compiled_model_roundtrip(tmp_path, compiled_models):
    cm = compiled_models["guppy"]
    p = os.path.join(str(tmp_path), "m.npz")
    cm.save(p)
    cm2 = M.CompiledModel.load(p)
    assert cm2.text == cm.text
    for k in cm.kde:
        assert np.array_equal(cm.kde[k][0], cm2.kde[k][0]) and cm.kde[k][1] == cm2.kde[k][1]


# the original NanoSim's pre-trained_models/ directory (its model archives are hundreds of MB, not part of this repository)
REF_MODELS = os.environ.get("NANOSIM_PRETRAINED_MODELS", "")


@pytest.mark.skipif(not os.path.isdir(REF_MODELS), reason="set NANOSIM_PRETRAINED_MODELS to the original NanoSim's pre-trained_models directory")
@pytest.mark.parametrize("tarball,prefix,shipped", [
    ("human_NA12878_DNA_FAB49712_guppy.tar.gz", "human_NA12878_DNA_FAB49712_guppy/training", "guppy_fab49712_plusq.npz"),
    ("human_NA12878_DNA_FAB49712_guppy_flipflop.tar.gz", "human_NA12878_DNA_FAB49712_guppy_flipflop/training", None),
    ("human_giab_hg002_sub1M_kitv14_dorado.tar.gz", "human_giab_hg002_sub1M_kitv14_dorado/hg002_nanosim_sub1M", None),
])
def test_reference_model_directories_load_and_tabulate(tmp_path, tarball, prefix, shipped):
    """`-c <model_dir>/<prefix>` on the reference's own model archives: text tables + sklearn KDE pickles -> device tables;
    the shipped .npz is a lossless copy of the directory it was compiled from (plus the quality table of config 2)."""
    import tarfile
    from nanosim_b200.model import CompiledModel, DeviceTables, load_model
    with tarfile.open(os.path.join(REF_MODELS, tarball)) as tf:
        tf.extractall(str(tmp_path), filter="data")
    cm = load_model(os.path.join(str(tmp_path), prefix))
    t = DeviceTables(cm, fastq=False, chimeric="chimeric_info" in cm.text)
    assert len(t.alias_prob) > 1000 and len(cm.kde) >= 5
    if shipped:
        ours = CompiledModel.load(os.path.join(DATA, shipped))
        for k, v in cm.text.items():
            assert ours.text[k] == v, k
        for k, (data, bw) in cm.kde.items():
            assert np.array_equal(ours.kde[k][0], data) and ours.kde[k][1] == bw, k


def _write_sklearn_kde_pickle(path, data, bandwidth, monkeypatch):
    """joblib.dump of a KernelDensity as scikit-learn 0.22 lays it out: the estimator's __dict__ (bandwidth, kernel,
    tree_, ...) with tree_ a KDTree reduced through ``newObj`` to the state tuple (data, idx_array, node_data,
    node_bounds, leaf_size, ..., dist_metric).  Stand-in classes under the sklearn module names write the same globals
    without scikit-learn installed."""
    import joblib
    import types

    mods = {n: types.ModuleType(n) for n in ("sklearn", "sklearn.neighbors", "sklearn.neighbors._kde",
                                             "sklearn.neighbors._kd_tree", "sklearn.neighbors._dist_metrics")}
    for n, m in mods.items():
        monkeypatch.setitem(sys.modules, n, m)

    def newObj(cls):
        return cls.__new__(cls)

    class KDTree:
        def __init__(self, state):
            self.state = state

        def __reduce__(self):
            return newObj, (KDTree,), self.state

    class EuclideanDistance:
        def __reduce__(self):
            return newObj, (EuclideanDistance,), {"p": 2.0}

    class KernelDensity:
        pass

    for obj, mod in ((newObj, "_kd_tree"), (KDTree, "_kd_tree"), (EuclideanDistance, "_dist_metrics"), (KernelDensity, "_kde")):
        obj.__module__, obj.__qualname__ = "sklearn.neighbors." + mod, obj.__name__
        setattr(mods["sklearn.neighbors." + mod], obj.__name__, obj)
    n = len(data)
    kd = KernelDensity()
    kd.__dict__.update(bandwidth=bandwidth, algorithm="auto", kernel="gaussian", metric="euclidean", atol=0, rtol=0,
                       breadth_first=True, leaf_size=40, metric_params=None, _sklearn_version="0.22.1",
                       tree_=KDTree((data, np.arange(n, dtype=np.intp), np.zeros(1), np.zeros((2, 1, data.shape[1])),
                                     40, 1, 1, 0, 1, 0, 0, EuclideanDistance())))
    joblib.dump(kd, path)


@pytest.mark.parametrize("tag", CASES)
def test_reference_format_directory_loads_as_shipped_model(tag, compiled_models, tmp_path, monkeypatch):
    """`-c <dir>/<prefix>` with a model directory in the reference's on-disk format: text tables under their file names
    and one KernelDensity pickle per KDE.  The directory is written from the shipped model, so load_model must return
    it unchanged, and the device tables must build from it."""
    from nanosim_b200.model import DeviceTables, load_model
    cm = compiled_models[tag]
    prefix = os.path.join(str(tmp_path), "training")
    for name, text in cm.text.items():
        with open(prefix + "_" + name, "w") as f:
            f.write(text)
    for name, (data, bw) in cm.kde.items():
        _write_sklearn_kde_pickle(prefix + "_" + name + ".pkl", data, bw, monkeypatch)
    monkeypatch.undo()                              # the stand-in modules are gone: the loader reads the pickles without them
    got = load_model(prefix)
    assert got.text == cm.text
    assert sorted(got.kde) == sorted(cm.kde)
    for k, (data, bw) in cm.kde.items():
        assert got.kde[k][0].dtype == np.float64 and np.array_equal(got.kde[k][0], data) and got.kde[k][1] == bw, k
    t = DeviceTables(got, fastq=True, chimeric="chimeric_info" in got.text)
    assert len(t.alias_prob) > 1000 and len(got.kde) >= 5
