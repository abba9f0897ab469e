"""Static drop-in check against the original project's OWN call sites, as recorded in tests/golden/dropin_callsites.json
(oracle/gen_golden_dropin.py; tests/test_loader_gpu.py replays the same call sequence on the device).  Every
`visualcla.<name>(...)` call in scripts/inference/inference.py and scripts/inference/gradio_demo.py must resolve in this
package with a signature that accepts the keywords the script passes, and every method / attribute the scripts touch on the
model object must exist on VisualCLAModel."""
import inspect
import json
import os

import pytest

import visualcla
from visualcla.modeling_visualcla import VisualCLAModel, _SubModel

SCRIPTS = ["inference.py", "gradio_demo.py"]


@pytest.fixture(scope="module")
def callsites(golden_dir):
    with open(os.path.join(golden_dir, "dropin_callsites.json")) as fh:
        return json.load(fh)


@pytest.mark.parametrize("script", SCRIPTS)
def test_reference_scripts_resolve_against_this_package(callsites, script):
    rec = callsites["scripts"][script]
    seen = []
    for call in rec["visualcla_calls"]:
        chain, kws, npos = call["chain"], call["keywords"], call["n_positional"]
        obj = visualcla
        for name in chain:
            assert hasattr(obj, name), f"{script}: visualcla.{'.'.join(chain)} does not exist in the drop-in package"
            obj = getattr(obj, name)
        if callable(obj):
            params = inspect.signature(obj).parameters
            accepts_kwargs = any(p.kind is inspect.Parameter.VAR_KEYWORD for p in params.values())
            for k in kws:
                assert k in params or accepts_kwargs, f"{script}: visualcla.{'.'.join(chain)}() is called with {k}= which the drop-in does not accept"
            assert npos <= len([p for p in params.values() if p.kind in (p.POSITIONAL_ONLY, p.POSITIONAL_OR_KEYWORD)])
        seen.append(".".join(chain))
    assert seen, f"{script} makes no visualcla.* call?"
    # attribute imports:  from visualcla.modeling_utils import DEFAULT_GENERATION_CONFIG  (gradio_demo.py:2)
    for imp in rec["imports"]:
        mod = __import__(imp["module"], fromlist=["x"])
        for name in imp["names"]:
            assert hasattr(mod, name), f"{script}: from {imp['module']} import {name}"
    # methods / attributes the scripts use on the model objects
    for root, chains in rec["model_calls"].items():
        for chain in chains:
            cls = VisualCLAModel
            for name in chain:
                if name in ("text_model", "vision_model", "visual_resampler"):      # set per instance in __init__: handles of type _SubModel
                    cls = _SubModel
                    continue
                assert hasattr(cls, name) or name in ("tokenizer", "image_processor", "num_patch", "device", "config"), \
                    f"{script}: {root}.{'.'.join(chain)}: '{name}' is missing on {cls.__name__}"
                break
    if script == "inference.py":
        assert "get_model_and_tokenizer_and_processor" in seen and "chat" in seen


def test_loader_signature_matches_the_reference_definition(callsites):
    """Same parameter names in the same order as the original models/visualcla/modeling_utils.py:83-92 (plus **engine_kwargs)."""
    for fn, want in callsites["loader_parameters"].items():
        have = [p.name for p in inspect.signature(getattr(visualcla.modeling_utils, fn)).parameters.values()
                if p.kind in (p.POSITIONAL_ONLY, p.POSITIONAL_OR_KEYWORD)]
        assert have[: len(want)] == want, f"{fn}: reference parameters {want}, drop-in {have}"
    assert set(callsites["loader_parameters"]) == {"get_model_and_tokenizer_and_processor", "chat", "chat_in_stream", "encoding_text"}
