"""Model archives in the reference's format (Base/DataIO.py): the reader against an archive the reference's own DataIO
wrote (tests/golden/dataio_ref.zip), a round trip through the writer, and the writer's archive against the reference's
one, member for member."""
import io
import os
import zipfile

import numpy as np
import pytest
import scipy.sparse as sps

from recsys2019_deeplearning_evaluation_b200.dataio import DataIO

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden") + "/"


def _payload():
    import pandas as pd
    rng = np.random.default_rng(5)
    return {"W_sparse": sps.random(30, 30, 0.1, format="csr", random_state=3, dtype=np.float32),
            "USER_factors": rng.random((7, 4)), "use_bias": False, "topK": np.int64(50), "name": "x",
            "mapper": {3: "a", 9: "b"}, "nested": {"A": rng.random(3), "k": 2},
            "frame": pd.DataFrame({"a": [1, 2], "b": [0.5, 1.5]})}


def _check(d):
    want = _payload()
    assert set(d.keys()) == set(want.keys())
    assert abs(d["W_sparse"] - want["W_sparse"]).nnz == 0 and d["W_sparse"].dtype == np.float32
    assert np.array_equal(d["USER_factors"], want["USER_factors"])
    assert d["use_bias"] is False and d["topK"] == 50 and d["name"] == "x"
    assert d["mapper"] == {"3": "a", "9": "b"}  # JSON keys are strings (Base/DataIO.py:81-102)
    assert np.array_equal(d["nested"]["A"], want["nested"]["A"]) and d["nested"]["k"] == 2
    assert d["frame"].equals(want["frame"])


def test_reads_archive_written_by_the_reference():
    _check(DataIO(GOLDEN).load_data("dataio_ref"))


def test_round_trip(tmp_path):
    io = DataIO(str(tmp_path) + "/sub/")
    io.save_data("model.zip", _payload())
    _check(io.load_data("model"))
    assert sorted(os.listdir(str(tmp_path) + "/sub/")) == ["model.zip"]  # no temp folder left behind
    with pytest.raises(TypeError):
        io.save_data("bad", {"x": object()})


def _same_archive(raw, ref):
    """Same members under the same names, each with the same payload (sparse members compared as matrices: the bytes of
    scipy's .npz may depend on the numpy version); nested archives recursively."""
    a, b = zipfile.ZipFile(io.BytesIO(raw)), zipfile.ZipFile(io.BytesIO(ref))
    assert sorted(a.namelist()) == sorted(b.namelist())
    for name in b.namelist():
        x, y = a.read(name), b.read(name)
        if name.endswith(".zip"):
            _same_archive(x, y)
        elif name.endswith(".npz"):
            X, Y = sps.load_npz(io.BytesIO(x)), sps.load_npz(io.BytesIO(y))
            assert X.format == Y.format and X.dtype == Y.dtype and X.shape == Y.shape and abs(X - Y).nnz == 0, name
        else:
            assert x == y, name


def test_reference_reads_what_this_writer_wrote(tmp_path):
    """The reference's DataIO reads an archive through its manifest and the file type of each member: an archive that
    holds the members the reference's own writer produced from the same payload is one it reads."""
    DataIO(str(tmp_path) + "/").save_data("m", _payload())
    with open(str(tmp_path) + "/m.zip", "rb") as f, open(GOLDEN + "dataio_ref.zip", "rb") as g:
        _same_archive(f.read(), g.read())


@pytest.mark.gpu
def test_recommender_save_load(tmp_path):
    from recsys2019_deeplearning_evaluation_b200.recommenders import ItemKNNCFRecommender, IALSRecommender, EASE_R_Recommender
    from recsys2019_deeplearning_evaluation_b200.synth import synth_urm
    X = synth_urm(300, 120, 0.06, seed=3, values="ratings")
    folder = str(tmp_path) + "/"
    users = np.arange(40)
    for make, fit_kw in ((ItemKNNCFRecommender, dict(topK=10, shrink=2)), (IALSRecommender, dict(epochs=2, num_factors=8)),
                         (EASE_R_Recommender, dict(l2_norm=500.0, verbose=False))):
        a = make(X, verbose=False)
        a.fit(**fit_kw)
        a.save_model(folder)
        b = make(X, verbose=False)
        b.load_model(folder)
        assert np.allclose(a._compute_item_score(users), b._compute_item_score(users), rtol=1e-5, atol=1e-6)
        assert os.path.exists(folder + a.RECOMMENDER_NAME + ".zip")
