"""Generate tests/golden/dropin_callsites.json from a checkout of the original VisualCLA project:

    python oracle/gen_golden_dropin.py <original project checkout>

What tests/test_dropin_conformance_cpu.py checks this package against: every `visualcla.<name>(...)` call in
scripts/inference/inference.py and scripts/inference/gradio_demo.py (attribute chain, keyword names, number of positional
arguments), every `from visualcla... import ...` in them, the method / attribute chains they use on `model` and
`base_model`, and the positional parameter names of the public functions of models/visualcla/modeling_utils.py.
Only these names are stored, no source text."""
import ast
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(os.path.dirname(HERE), "tests", "golden", "dropin_callsites.json")
SCRIPTS = ["inference.py", "gradio_demo.py"]
LOADER_FUNCTIONS = ["get_model_and_tokenizer_and_processor", "chat", "chat_in_stream", "encoding_text"]


def _calls(tree, root_name):
    """(attribute chain, keyword names, n positional) of every call whose function is an attribute chain starting at `root_name`."""
    out = []
    for node in ast.walk(tree):
        if not isinstance(node, ast.Call):
            continue
        chain, f = [], node.func
        while isinstance(f, ast.Attribute):
            chain.append(f.attr)
            f = f.value
        if isinstance(f, ast.Call):          # e.g. model.text_model.get_input_embeddings().weight.size(0): follow the inner call too
            continue
        if isinstance(f, ast.Name) and f.id == root_name and chain:
            out.append({"chain": list(reversed(chain)), "keywords": [k.arg for k in node.keywords if k.arg], "n_positional": len(node.args)})
    return out


def _imports(tree):
    return [{"module": n.module, "names": [a.name for a in n.names]} for n in ast.walk(tree)
            if isinstance(n, ast.ImportFrom) and n.module and n.module.startswith("visualcla")]


def main(root):
    scripts = {}
    for s in SCRIPTS:
        with open(os.path.join(root, "scripts", "inference", s)) as fh:
            tree = ast.parse(fh.read())
        scripts[s] = {"visualcla_calls": _calls(tree, "visualcla"), "imports": _imports(tree),
                      "model_calls": {r: [c["chain"] for c in _calls(tree, r)] for r in ("model", "base_model")}}
    with open(os.path.join(root, "models", "visualcla", "modeling_utils.py")) as fh:
        defs = {n.name: n for n in ast.walk(ast.parse(fh.read())) if isinstance(n, ast.FunctionDef)}
    params = {fn: [a.arg for a in defs[fn].args.args] for fn in LOADER_FUNCTIONS}
    with open(OUT, "w") as fh:
        json.dump({"scripts": scripts, "loader_parameters": params}, fh, indent=1)
        fh.write("\n")
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
