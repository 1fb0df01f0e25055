"""Drop-in check by introspection: every public function, class, method and static method of the six reference modules
(epropnp.epropnp, .levenberg_marquardt, .camera, .cost_fun, .common, .distributions) exists under the same name in the
package, and every parameter of the reference signature is present in ours, in the same order, with the same default
(ours may append optional keyword arguments).  The reference surface is tests/golden/api_surface.json, recorded from the
unmodified reference package by oracle/api_surface.py."""
import json
import os

from conftest import ROOT
from oracle.api_surface import GOLDEN, surface


def test_every_public_name_and_parameter_of_the_reference_exists_here():
    with open(GOLDEN) as f:
        ref = json.load(f)
    ours = surface([os.path.join(ROOT, "epro-pnp_b200"), ROOT], "all")
    assert len(ref) > 60
    missing = sorted(k for k in ref if k not in ours)
    assert not missing, missing
    problems = []
    for name, want in ref.items():
        have = ours[name]
        if want is None or have is None:
            continue
        if any(kind in ("VAR_POSITIONAL", "VAR_KEYWORD") for _, kind, _ in want) and len(want) <= 3 and want[-1][0] in ("args", "kwargs"):
            continue                                           # the base class's abstract (*args, **kwargs) stubs
        fixed = [p for p in want if p[1] not in ("VAR_POSITIONAL", "VAR_KEYWORD")]
        ours_fixed = [p for p in have if p[1] not in ("VAR_POSITIONAL", "VAR_KEYWORD")]
        if ours_fixed[:len(fixed)] != fixed:
            problems.append((name, fixed, ours_fixed))
        elif any(extra[2] is None for extra in ours_fixed[len(fixed):]):
            problems.append((name, "extra parameter without a default", ours_fixed[len(fixed):]))
    assert not problems, problems
