"""The inputs of the conv fixtures (tests/golden/a1_neuralop_conv, a4_rno_conv, a6_pino_conv), regenerated, not stored.

tests/golden/make_golden.py draws every input of these three fixtures from torch's CPU generator after one manual_seed
per fixture: the module's parameters as the reference initialises them, the input x and the output gradient gy, case
after case.  Stored, they pushed single fixtures past 1 MB; replayed in the same order they come back bit for bit.  So
the files keep the reference's results (y, dx, parameter gradients), the seed and each case's shapes, plus a strided
sample of every replayed tensor, which restore() checks before a test sees the case.  Storing each case in a file of its
own would not do: a4's cfg3_small (1.61 MB) and a6's cfg4_small (1.51 MB) are each over 1 MB alone.

If restore() raises, torch's CPU generator no longer gives the same draws: regenerate the three fixtures with
tests/golden/make_golden.py from a checkout of the reference (strip() checks the new replay bit for bit when it writes
them), or run the suite with a torch version that still reproduces them.
"""
import math

import torch

# the fixtures whose inputs are replayed; restore() leaves every other fixture as it was loaded
FAMILIES = ("a1_neuralop_conv", "a4_rno_conv", "a6_pino_conv")
CHECK_STRIDE = 97
INPUTS = ("x", "gy", "params")


def _draw_params(family, shapes):
    """The reference modules' initialisation, in their order of draws (make_golden.py builds the module first)."""
    if family == "a1_neuralop_conv":
        # neuralop FactorizedSpectralConv: init_std = 1 / (ci * co); the complex weights first, then the bias
        ci, co = shapes["weight.0.tensor"][:2]
        std = 1.0 / (ci * co)
        p = {n: torch.zeros(s, dtype=torch.cfloat).normal_(0, std) for n, s in shapes.items() if n != "bias"}
        p["bias"] = std * torch.randn(shapes["bias"])
        return p
    if family == "a4_rno_conv":
        ci, co, m1, m2, _ = shapes["fourier_weight.0"]
        std = 1.0 / (ci * co * math.sqrt(m1 * m2))
        return {n: torch.empty(s).normal_(0, std) for n, s in shapes.items()}
    if family == "a6_pino_conv":
        ci, co = shapes["weights1"][:2]
        scale = 1.0 / (ci * co)
        return {n: scale * torch.rand(*s, dtype=torch.cfloat) for n, s in shapes.items()}
    raise KeyError(family)


def _replay(family, seed, cases):
    """Yields (name, inputs) in the order make_golden.py drew them."""
    torch.manual_seed(seed)
    for name, c in cases.items():
        inputs = {"params": _draw_params(family, c["param_shapes"])}
        inputs["x"] = torch.randn(c["x_shape"])
        if "y" in c and "dx" in c:                   # fwd + bwd cases; the layer-index case is forward only
            inputs["gy"] = torch.randn(c["y"].shape)
        yield name, inputs


def _samples(inputs):
    out = {k: v.flatten()[::CHECK_STRIDE].clone() for k, v in inputs.items() if k != "params"}
    out.update({f"params.{n}": v.flatten()[::CHECK_STRIDE].clone() for n, v in inputs["params"].items()})
    return out


def strip(family, seed, cases):
    """Full cases (as make_golden.py builds them) -> what the fixture file stores.  Raises if the replay does not give
    back every input bit for bit."""
    stored = {}
    for name, c in cases.items():
        s = {k: v for k, v in c.items() if k not in INPUTS}
        s["x_shape"] = tuple(c["x"].shape)
        s["param_shapes"] = {n: tuple(p.shape) for n, p in c["params"].items()}
        stored[name] = s
    for name, inputs in _replay(family, seed, stored):
        for k in inputs:
            want, got = cases[name][k], inputs[k]
            same = (all(torch.equal(want[n], got[n]) for n in want) and want.keys() == got.keys()) if k == "params" \
                else torch.equal(want, got)
            if not same:
                raise ValueError(f"{family}/{name}: the seeded replay does not reproduce {k}")
        stored[name]["check"] = _samples(inputs)
    return {"seed": seed, "cases": stored}


def restore(family, data):
    """What a fixture file stores -> the full cases the tests read (x, gy and params filled in)."""
    if family not in FAMILIES:
        return data
    cases = {name: dict(c) for name, c in data["cases"].items()}
    for name, inputs in _replay(family, data["seed"], cases):
        c = cases[name]
        check = c.pop("check")
        got = _samples(inputs)
        if got.keys() != check.keys() or not all(torch.equal(got[k], check[k]) for k in check):
            raise RuntimeError(f"{family}/{name}: torch's CPU generator no longer reproduces the fixture's inputs "
                               "(regenerate them with tests/golden/make_golden.py; see tests/seeded_inputs.py)")
        params = inputs.pop("params")
        c["params"] = {n: params[n] for n in c.pop("param_shapes")}
        del c["x_shape"]
        c.update(inputs)
    return cases
