"""The UNMODIFIED reference's ``models.SynthesizerTrn`` surface that ``patch_reference`` builds on: constructor and ``infer``
parameter names, and the state_dict layout (key -> shape) for the default config.  Needs the reference source tree
(``SOVITS_REF_DIR``, see make_golden.py):

    python tests/golden/make_golden_surface.py
"""
import inspect
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as MG  # noqa: E402  (sets up the reference import with stubbed audio modules)

with open(MG.sovits_b200.DEFAULT_CONFIG) as f:
    model_kw = json.load(f)["model"]
cls = MG.ref_models.SynthesizerTrn
code = cls.__init__.__code__
net = cls(2048 // 2 + 1, 10240 // 512, **model_kw)
layout = {k: list(v.shape) for k, v in net.state_dict().items()}
with open(os.path.join(HERE, "ref_surface.json"), "w") as f:         # one state_dict entry per line
    f.write('{\n "init_params": %s,\n "infer_params": %s,\n "state_dict": {\n' % (
        json.dumps(list(code.co_varnames[1:code.co_argcount])), json.dumps(list(inspect.signature(cls.infer).parameters))))
    f.write(",\n".join(f"  {json.dumps(k)}: {json.dumps(s)}" for k, s in layout.items()))
    f.write("\n }\n}\n")
print("reference surface:", len(layout), "state_dict entries")
