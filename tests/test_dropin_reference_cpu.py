"""The drop-in claim of INTEGRATION.md §1, executed: the reference's own `model/vcmr.py` +
`model/pretrain.py` (unmodified) run on top of a copy of its `model/model.py` whose three encoder
imports point at hero_b200 — (A) keeping the reference's HierarchicalVlModel / HeroModel classes
over hero_b200's CrossModalTrm / TemporalTrm / LinearLayer, (B) also re-exporting hero_b200's
packed-path classes — and reproduce the goldens of the unmodified reference. Needs the reference
sources (a checkout named by HERO_REFERENCE, or the copy baseline/stage_ref.py staged under
baseline/_ref): skipped elsewhere."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _reference_dir():
    for cand in (os.environ.get("HERO_REFERENCE"), os.path.join(ROOT, "baseline", "_ref")):
        if cand and os.path.isfile(os.path.join(cand, "model", "model.py")):
            return cand
    return None


@pytest.mark.parametrize("variant", ["A", "B"])
def test_reference_heads_run_on_swapped_encoder_imports(tmp_path, variant):
    ref = _reference_dir()
    if ref is None:
        pytest.skip("reference sources not available")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_script.py"), ref,
                        str(tmp_path), variant], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["encoder_class"] == "hero_b200.encoder"
    assert out["model_class"] == ("hero_b200.model" if variant == "B" else "model.model")
