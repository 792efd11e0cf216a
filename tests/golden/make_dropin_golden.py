"""Golden data of tests/test_cpu_dropin.py, produced by the REFERENCE's own ``create_model_config`` / ``create_model``
(hydragnn/models/create.py:41-108,112-766).  The two functions are AST-extracted from the reference checkout named by
``make_golden.REF`` (never copied into this repo) and exec'd with the absent third-party packages stubbed exactly as
make_golden.py does.

    python tests/golden/make_dropin_golden.py     # writes tests/golden/dropin.json

For each configuration of the test it records the keyword arguments ``create_model`` receives (the locals the INTEGRATION.md
dispatch reads), the seeded state dict of the returned model and of the stack inside it (shape, dtype and SHA-256 of the bytes of
every tensor: equal digests mean bitwise-equal values), the attributes the reference's train / validate / test loop reads through
``model.module`` (train_validate_test.py:225-242,498,731,736,1006-1018) and ``str()`` of the stack.  It also records the
reference's error for an unknown ``mpnn_type`` (create.py:584).
"""
import ast
import copy
import hashlib
import importlib.util
import json
import os
import sys
import typing

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
CASES = [("EGNN", True), ("PAINN", False), ("EGNN", False)]
ATTRS = ("num_heads", "head_dims", "head_type", "loss_weights", "var_output", "graph_pooling")


def case_id(mpnn_type, mlip):
    return "%s-%s" % (mpnn_type, "mlip" if mlip else "graph")


def digest(state_dict):
    """{name: [shape, dtype, sha256 of the tensor's bytes]} in state-dict order"""
    return {k: [list(v.shape), str(v.dtype), hashlib.sha256(v.detach().cpu().contiguous().numpy().tobytes()).hexdigest()]
            for k, v in state_dict.items()}


def _reference_create(mg, record):
    """(create_model_config, create_model) of the reference; ``create_model`` first appends a copy of its arguments to ``record``."""
    egcl, painn = mg.install_stubs()
    path = mg.REF + "/hydragnn/models/create.py"
    tree = ast.parse(open(path).read())
    fns = {n.name: n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in ("create_model_config", "create_model")}
    assert set(fns) == {"create_model_config", "create_model"}
    fns["create_model"].body = ast.parse("_RECORD.append(_copy.deepcopy(dict(locals())))").body + fns["create_model"].body
    glb = {"torch": torch, "os": os, "_RECORD": record, "_copy": copy}
    mg._extract(mg.REF + "/hydragnn/utils/model/model.py", ["update_multibranch_heads"], glb)

    class Timer:
        def __init__(self, *_): pass
        def start(self): pass
        def stop(self): pass

    def resolve_precision(p):                         # hydragnn/train/train_validate_test.py:43-63, fp32 / bf16 branch
        return ("fp32", torch.float32, None) if str(p).lower() in ("fp32", "float32") else ("bf16", torch.float32, torch.bfloat16)

    glb.update(Timer=Timer, resolve_precision=resolve_precision, get_device=lambda *a, **k: torch.device("cpu"),
               EGCLStack=egcl.EGCLStack, PAINNStack=painn.PAINNStack, Base=sys.modules["hydragnn.models.Base"].Base,
               List=typing.List, Union=typing.Union, Data=object, torch_scatter=sys.modules["torch_scatter"])
    for name in ("GINStack", "PNAStack", "PNAPlusStack", "GATStack", "MFCStack", "CGCNNStack", "SAGEStack", "SCFStack", "DIMEStack",
                 "PNAEqStack", "MACEStack", "MultiTaskModelMP"):
        glb.setdefault(name, None)
    for n in ("create_model_config", "create_model"):
        exec(compile(ast.Module(body=[fns[n]], type_ignores=[]), path, "exec"), glb)
    return glb["create_model_config"], glb["create_model"]


def config(mpnn_type, mlip):
    """config["NeuralNetwork"] after update_config, LennardJones-like (examples/LennardJones/LJ.json with mpnn_type switched)"""
    arch = dict(mpnn_type=mpnn_type, input_dim=1, hidden_dim=32, output_dim=[1], pe_dim=0, global_attn_engine=None, global_attn_type=None,
                global_attn_heads=0, output_type=["node"] if mlip else ["graph"], activation_function="relu", task_weights=[1.0],
                num_conv_layers=2, freeze_conv_layers=False, initial_bias=None, num_nodes=None, max_neighbours=5, edge_dim=None,
                pna_deg=None, num_before_skip=None, num_after_skip=None, num_radial=5, radial_type=None, distance_transform=None,
                basis_emb_size=None, int_emb_size=None, out_emb_size=None, envelope_exponent=None, num_spherical=None,
                num_gaussians=None, num_filters=None, radius=5.0, equivariance=False, correlation=None, max_ell=None, node_max_ell=None,
                avg_num_neighbors=None)
    if mlip:
        # heads in the list-of-branches form that update_config produces (hydragnn/utils/model/model.py:314-349)
        arch.update(output_heads={"node": [{"type": "branch-0", "architecture": {"num_headlayers": 2, "dim_headlayers": [60, 20],
                                                                                  "type": "mlp"}}]},
                    enable_interatomic_potential=True, energy_weight=1.0, energy_peratom_weight=1.0, force_weight=1.0)
    else:
        arch.update(output_heads={"graph": [{"type": "branch-0", "architecture": {"num_sharedlayers": 2, "dim_sharedlayers": 5,
                                                                                   "num_headlayers": 2, "dim_headlayers": [50, 25]}}]})
    return {"Architecture": arch, "Training": {"loss_function_type": "mse", "conv_checkpointing": False, "precision": "fp32"}}


def main():
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    record = []
    create_model_config, _ = _reference_create(mg, record)
    out = {}
    for mpnn_type, mlip in CASES:
        del record[:]
        model = create_model_config(config(mpnn_type, mlip), verbosity=0, use_gpu=False)
        stack = model.model if mlip else model
        assert len(record) == 1
        out[case_id(mpnn_type, mlip)] = {
            "create_model_args": record[0], "state_dict": digest(model.state_dict()),
            "stack_state_dict": digest(stack.state_dict()),
            "attrs": {a: getattr(model, a) for a in ATTRS}, "str": str(stack)}
    try:
        create_model_config(config("NOPE", False), verbosity=0, use_gpu=False)
        raise AssertionError("the reference accepted an unknown mpnn_type")
    except ValueError as ex:
        out["unknown_mpnn_type"] = {"error": type(ex).__name__, "message": str(ex)}
    with open(os.path.join(HERE, "dropin.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("drop-in golden data written to", os.path.join(HERE, "dropin.json"))


if __name__ == "__main__":
    main()
