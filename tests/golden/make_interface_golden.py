"""Record what the REFERENCE's `train.py` needs from this repo's drop-in packages, by importing it unmodified
through tests/ref_launcher.py in "dropin" mode (repo root first on sys.path).  Needs the reference tree.

    BDBNN_REFERENCE_ROOT=<reference checkout> python tests/golden/make_interface_golden.py
        ->  tests/golden/reference_interface.json

Recorded: every name train.py imports (`from M import N`) that resolved to a file of this repo; the attributes train.py
reads on the drop-in modules it imported (`utils.X`, `KD_loss.X`, ...); the model-name lists it builds from
`models.cifar10` / `models.imagenet`; the parser defaults of the flags that bdbnn_b200.step.StepConfig mirrors.
tests/test_ref_train.py checks this repo against the record without the reference."""
import ast
import dataclasses
import json
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import ref_launcher as RL        # noqa: E402


def in_repo(mod):
    f = getattr(mod, "__file__", None)
    return f is not None and os.path.abspath(f).startswith(RL.REPO_ROOT + os.sep)


def main():
    train = RL.import_reference_train("dropin")
    with open(train.__file__) as fh:
        tree = ast.parse(fh.read())
    imports, module_alias = [], {}
    for node in tree.body:
        if not (isinstance(node, ast.ImportFrom) and node.level == 0):
            continue
        for a in node.names:
            bound = getattr(train, a.asname or a.name)
            is_mod = isinstance(bound, types.ModuleType)
            if in_repo(bound if is_mod else sys.modules[node.module]):
                imports.append({"module": node.module, "name": a.name})
                if is_mod:
                    module_alias[a.asname or a.name] = bound.__name__
    attributes = {}
    for node in ast.walk(tree):
        if (isinstance(node, ast.Attribute) and isinstance(node.value, ast.Name) and node.value.id in module_alias
                and not node.attr.startswith("__")):
            attributes.setdefault(module_alias[node.value.id], set()).add(node.attr)
    from bdbnn_b200.step import StepConfig
    args = vars(train.parser.parse_args(["/nonexistent-data"]))
    shared = [f.name for f in dataclasses.fields(StepConfig) if f.name in args]
    rec = {"imports": imports,
           "attributes": {m: sorted(v) for m, v in sorted(attributes.items())},
           "model_names": {"cifar10": train.CIFAR10_MODEL_NAMES, "imagenet": train.IMAGENET_MODEL_NAMES},
           "parser_defaults": {k: args[k] for k in shared}}
    out = os.path.join(os.environ.get("BDBNN_GOLDEN_OUT", HERE), "reference_interface.json")
    with open(out, "w") as fh:
        json.dump(rec, fh, indent=1, sort_keys=True)
        fh.write("\n")
    print(out)


if __name__ == "__main__":
    main()
