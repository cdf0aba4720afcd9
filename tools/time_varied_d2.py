"""Per-instance physical parameters for second derivatives (trepb_deriv2_varied_batch_dev) against the plain entry
point, same inputs, alternating in one process; CUDA events around each call (the varied call's map upload included,
and the linearize launch that every deriv2 call makes).  Same method as tools/time_varied.py.

  pend_on_cart z:     pend-on-cart deriv2, 2^18 instances, z-contracted fdxdx / fdxdu / fdudu only; both sides on
                      the run-time-parameter kernels (literal=False), not the all-literal kernel a default handle runs
  pend_on_cart full:  the same with all 30 tensors written
  fourbar d2jac:      fourbar on the table-driven kernels (per-parameter scheme, passes A and B), 16384 instances
  marionette:         varied on a TREPB_FLAG_NO_COOP handle against plain on the default cooperative handle,
                      1024 instances, z-contracted (what a robust-optimisation Newton step pays)

Usage: python tools/time_varied_d2.py [--reps 5] [--small]     (--small: 1/16 of every size)
Prints one JSON line per workload: plain and varied ms (median of reps), their ratio, the card and its power limit."""
import argparse
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tests"))
sys.path.insert(0, HERE)
import golden_util as G  # noqa: E402
from test_varied_params import variable_refs  # noqa: E402
from time_varied import card, params, report, timed, up  # noqa: E402
from trep_b200 import lib  # noqa: E402


def refs_of(d):
    """Every entry that may vary except the frame_se3 rotations, as the tests draw them."""
    return [r for r in variable_refs(d) if r[0] != 1]


def case(name, B, tensors, rng, plain_kw, varied_kw):
    d, g = G.desc(name), G.golden(name)
    idx = np.arange(B) % len(g["case_iters"])
    c = lambda k: np.ascontiguousarray(g["case_" + k][idx])
    refs = refs_of(d)
    vals = params(d, refs, B, rng, spread=0.2)
    sp = lib.System(d, **plain_kw)
    sv = lib.System(d, **varied_kw) if varied_kw is not None else sp
    ins = dict(q1=up(c("q1")), p1=up(c("p1")), u1=up(c("u1")) if d.nu else None, k2=up(c("k2")) if d.nk else None,
               t1=up(np.zeros(B)), t2=up(np.full(B, 0.01)), q2g=up(c("q2_guess")),
               lam=up(c("lambda_guess")) if d.nc else None, z=up(rng.normal(0, 1, (B, d.nX))), vals=up(vals))
    outs = dict(status=lib.DeviceBuffer(0, (B,), np.int32), fdxdx=lib.DeviceBuffer(0, (B, d.nX, d.nX)),
                fdxdu=lib.DeviceBuffer(0, (B, d.nX, max(d.nU, 1))), fdudu=lib.DeviceBuffer(0, (B, max(d.nU, 1), max(d.nU, 1))))
    tens = {n: lib.DeviceBuffer(0, sh) for n, sh in sp.d2_shapes(B).items() if np.prod(sh)} if tensors else {}

    def run(varied):
        s = sv if varied else sp
        s.deriv2_raw(True, B, ins["q1"], ins["p1"], ins["u1"], ins["k2"], outs["status"], tens, z=ins["z"],
                     fdxdx=outs["fdxdx"], fdxdu=outs["fdxdu"] if d.nU else None,
                     fdudu=outs["fdudu"] if d.nU else None, t1=ins["t1"], t2=ins["t2"], q2_guess=ins["q2g"],
                     lambda_guess=ins["lam"], params=(refs, ins["vals"]) if varied else None)
    return run, dict(batch=B, entries=len(refs), tensors=bool(tensors), plain_kernel=sp.kernel_name,
                     varied_kernel=sv.kernel_name)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--small", action="store_true")
    a = ap.parse_args()
    f = 16 if a.small else 1
    gpu = card()
    rng = np.random.default_rng(0)
    todo = [("pend_on_cart z", "pend_on_cart1", (1 << 18) // f, False, dict(literal=False), None),
            ("pend_on_cart full", "pend_on_cart1", (1 << 18) // f, True, dict(literal=False), None),
            ("fourbar d2jac", "fourbar", 16384 // f, False, dict(specialize=False, cooperative=False), None),
            ("marionette", "puppet", 1024 // f, False, {}, dict(cooperative=False))]
    for label, name, B, tensors, pkw, vkw in todo:
        run, extra = case(name, B, tensors, rng, pkw, vkw)
        plain, varied = timed(run, a.reps)
        report(label, plain, varied, extra, gpu)


if __name__ == "__main__":
    main()
