import glob
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def load_golden(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    d = {k: z[k] for k in z.files}
    d["state_dict"] = {k[3:]: d[k] for k in d if k.startswith("sd.")}
    if "gen.seed" in d:  # a compact token golden: the canvas and weights come from their seed (make_golden_tokens.py)
        from oracle import tokens_oracle as to

        h, w = (int(v) for v in d["gen.hw"])
        bev, sd = to.golden_token_inputs(int(d["gen.batch"]), int(d["c_in"]), int(d["d_model"]), h, w, int(d["gen.seed"]),
                                         float(d["gen.occupancy"]))
        b = d["out.tokens"].shape[0]
        d["bev"], d["state_dict"] = bev[:b], sd
        assert np.array_equal(to.golden_inputs_sha256(d["bev"], sd), d["gen.sha256"]), f"{name}: regenerated inputs differ"
    return d


def vfe_golden_names():
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, "vfe_*.npz")))


@pytest.fixture(scope="session")
def oracle():
    from oracle import pillar_oracle

    pillar_oracle.build_oracle_lib()
    return pillar_oracle
