"""Generates tests/golden/dn_config_specs.json: what the REFERENCE's dn_config.py (/root/reference/dn_splatter/dn_config.py)
passes to nerfstudio for its three methods, recorded by executing that file unmodified against stand-in classes that only
remember their constructor arguments; and tests/golden/dn_model_config_fields.json: every field of the reference's
DNSplatterModelConfig (dn_splatter/dn_model.py) with the source of its default, in declaration order.

    python tests/golden/make_golden_config.py
"""
import json
import os
import sys
import types

REF = "/root/reference"
OUT = os.path.dirname(os.path.abspath(__file__))


class Rec:
    def __init__(self, *args, **kw):
        assert not args
        self.kw = kw

    def dump(self):
        def enc(v):
            if isinstance(v, Rec):
                return {"__class__": type(v).__name__, **{k: enc(x) for k, x in v.kw.items()}}
            if isinstance(v, dict):
                return {k: enc(x) for k, x in v.items()}
            return v
        return enc(self)


def recording_modules(names):
    """{module path: [class names]} -> installs stub modules whose classes record their kwargs."""
    for mod, classes in names.items():
        parts = mod.split(".")
        for i in range(1, len(parts) + 1):
            sys.modules.setdefault(".".join(parts[:i]), types.ModuleType(".".join(parts[:i])))
        for c in classes:
            setattr(sys.modules[mod], c, type(c, (Rec,), {}))


NERFSTUDIO = {
    "nerfstudio.configs.base_config": ["ViewerConfig"],
    "nerfstudio.engine.optimizers": ["AdamOptimizerConfig"],
    "nerfstudio.engine.schedulers": ["ExponentialDecaySchedulerConfig"],
    "nerfstudio.engine.trainer": ["TrainerConfig"],
    "nerfstudio.plugins.types": ["MethodSpecification"],
}
REFERENCE_SIDE = {
    "dn_splatter.data.normal_nerfstudio": ["NormalNerfstudioConfig"],
    "dn_splatter.dn_datamanager": ["DNSplatterManagerConfig"],
    "dn_splatter.dn_model": ["DNSplatterModelConfig"],
    "dn_splatter.dn_pipeline": ["DNSplatterPipelineConfig"],
}


def model_config_fields():
    """{field name: default expression as source} of the reference's DNSplatterModelConfig class body."""
    import ast

    tree = ast.parse(open(os.path.join(REF, "dn_splatter", "dn_model.py")).read())
    cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "DNSplatterModelConfig")
    return {n.target.id: ast.unparse(n.value) for n in cls.body if isinstance(n, ast.AnnAssign)}


def main():
    recording_modules({**NERFSTUDIO, **REFERENCE_SIDE})
    ns = {"__name__": "dn_splatter.dn_config"}
    exec(compile(open(os.path.join(REF, "dn_splatter", "dn_config.py")).read(), "dn_config.py", "exec"), ns)
    specs = {v.kw["config"].kw["method_name"]: v.dump() for v in ns.values() if type(v).__name__ == "MethodSpecification"}
    with open(os.path.join(OUT, "dn_config_specs.json"), "w") as f:
        json.dump(specs, f, indent=1, sort_keys=True)
    print(sorted(specs))
    fields = model_config_fields()
    with open(os.path.join(OUT, "dn_model_config_fields.json"), "w") as f:
        json.dump(fields, f, indent=1)
        f.write("\n")
    print(list(fields))


if __name__ == "__main__":
    main()
