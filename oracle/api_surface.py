#!/usr/bin/env python
"""The public API surface of the six `epropnp` modules, by introspection in a fresh interpreter: every public function,
class, method and static method, with each parameter's name, kind and default (repr).

    python oracle/api_surface.py <reference checkout>    # writes tests/golden/api_surface.json

The reference surface is recorded from the UNMODIFIED reference package (imported with oracle/pyro_shim on the path)
and stored as golden data; tests/test_api_surface_cpu.py computes ours the same way and compares the two."""
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(ROOT, "tests", "golden", "api_surface.json")
MODULES = ("epropnp.epropnp", "epropnp.levenberg_marquardt", "epropnp.camera", "epropnp.cost_fun", "epropnp.common",
           "epropnp.distributions")

_DUMP = r'''
import importlib, inspect, json, sys
def params(f):
    try:
        return [[p.name, p.kind.name, None if p.default is inspect.Parameter.empty else repr(p.default)]
                for p in inspect.signature(f).parameters.values()]
    except (TypeError, ValueError):
        return None
out = {}
for m in sys.argv[2:]:
    mod = importlib.import_module(m)
    for n, o in vars(mod).items():
        if n.startswith('_'):
            continue
        own = getattr(o, '__module__', None) == m
        if inspect.isclass(o) and (own or sys.argv[1] == 'all'):
            for kls in (o.__mro__ if sys.argv[1] == 'all' else (o,)):
                for mn, mo in vars(kls).items():
                    if mn.startswith('__') and mn != '__init__':
                        continue
                    f = mo.__func__ if isinstance(mo, (staticmethod, classmethod)) else mo
                    if callable(f):
                        out.setdefault(f'{m}:{n}.{mn}', params(f))
        elif callable(o) and not inspect.isclass(o) and (own or sys.argv[1] == 'all'):
            out[f'{m}:{n}'] = params(o)
print(json.dumps(out))
'''


def surface(paths, mode):
    """{'<module>:<name>[.<method>]': [[param, kind, repr(default) | None], ...] | None} of MODULES imported from
    `paths`.  mode 'own': only names defined in each module; 'all': also imported names and inherited methods."""
    env = dict(os.environ, PYTHONPATH=os.pathsep.join(paths))
    r = subprocess.run([sys.executable, "-c", _DUMP, mode, *MODULES], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


if __name__ == "__main__":
    if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "epropnp")):
        sys.exit("usage: python oracle/api_surface.py <reference checkout containing epropnp/>")
    ref = surface([os.path.join(HERE, "pyro_shim"), os.path.abspath(sys.argv[1])], "own")
    with open(GOLDEN, "w") as f:
        json.dump(ref, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"wrote {GOLDEN}: {len(ref)} names")
