"""Host-side input preparation against the reference's own function, through its recorded outputs
(tests/golden/reference_io.npz, written by tests/golden/make_reference_io.py from the unmodified reference)."""
import json
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import reference_cases  # noqa: E402

G = os.path.join(os.path.dirname(__file__), "golden")


def test_pil2tensor_matches_reference_function():
    """supir_b200.util.PIL2Tensor (host-side input preparation, restated) against the reference's own function
    (SUPIR/util.py:60-84) on random image sizes (24 of them) and every argument combination test.py / gradio_demo use:
    same working size, same reported size, same pixels (sha256 of the tensor)."""
    pytest.importorskip("PIL")
    from PIL import Image
    from supir_b200 import util
    want = json.loads(str(np.load(os.path.join(G, "reference_io.npz"))["pil2tensor"]))
    cases = list(reference_cases.pil2tensor_cases(Image))
    assert len(cases) == len(want) == 120
    for (img, args), (digest, h0, w0) in zip(cases, want):
        t, h, w = util.PIL2Tensor(img, **args)
        assert (h, w) == (h0, w0) and reference_cases.digest(t) == digest, (img.size, args)
