import os
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from oracle.ref import REF_DATA  # noqa: E402  the reference project's data/, None unless CRF_REFERENCE names a checkout

GOLDEN = Path(__file__).resolve().parent / "golden"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    # Contexts created with default options run MeanShift in the reference's exact summation order under the tests, so that
    # iteration counts and integer landmarks compare bit for bit; the tolerance mode (the library's default) is requested
    # explicitly where it is tested (ms_mode="fast").
    os.environ.setdefault("CRF_MS_MODE", "exact")


@pytest.fixture(scope="session")
def native():
    """Builds libcrf_b200.so and the oracle if they are stale."""
    import __graft_entry__ as g
    g.build()
    return True


@pytest.fixture(scope="session")
def O(native):
    from oracle import oracle
    return oracle


@pytest.fixture(scope="session")
def crf(native):
    import face_alignment_cvpr_2012_b200
    return face_alignment_cvpr_2012_b200


@pytest.fixture(scope="session")
def synth_dirs(tmp_path_factory):
    from face_alignment_cvpr_2012_b200 import synthetic_model as sm
    d = tmp_path_factory.mktemp("synth_model")
    return sm.write_model(d, seed=5)


@pytest.fixture(scope="session")
def synth_models(crf, O, synth_dirs):
    hp, ffd = synth_dirs
    return crf.Model(hp, ffd, 15, 20), O.Model(hp, ffd, 15, 20)


@pytest.fixture(scope="session")
def shipped():
    """True when the shipped forests and the LFW fixtures are staged (tools/stage_data.py, from a checkout of the reference
    project).  Otherwise the tests that use them run on the synthetic forests and workloads.procedural_lfw(), against golden
    vectors made for exactly those inputs (tests/golden/make_synth_golden.py)."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    return wl.staged_model_path() is not None and bool(wl.load_lfw())


@pytest.fixture(scope="session")
def staged_models(crf, O, shipped, synth_models):
    if not shipped:
        return synth_models
    from face_alignment_cvpr_2012_b200 import workloads as wl
    p = wl.staged_model_path()
    return crf.Model(packed=str(p)), O.Model(packed=str(p))


@pytest.fixture(scope="session")
def cv2_golden():
    return np.load(GOLDEN / "cv2_stages.npz")


@pytest.fixture(scope="session")
def lfw_golden(shipped):
    return np.load(GOLDEN / ("lfw_e2e.npz" if shipped else "synth_lfw.npz"))


@pytest.fixture(scope="session")
def faces(shipped):
    """The 20 LFW fixtures when staged, else their procedural stand-ins (same format, no landmark annotation)."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    return wl.load_lfw() if shipped else wl.procedural_lfw()


@pytest.fixture(scope="session")
def lfw_faces(shipped):
    """The real LFW fixtures, for the tests that need real faces with annotated landmarks (a face detector, accuracy against the
    annotation).  Only together with the shipped forests, which lfw_golden and staged_models pair with them."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    if not shipped:
        pytest.skip("staged/imgs and staged/model.crfb200 not present (tools/stage_data.py writes them from a checkout of the reference project)")
    return wl.load_lfw()
