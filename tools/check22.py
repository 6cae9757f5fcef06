"""Debug: 2^lg product sumcheck through the native engine, final-claim identity, resident vs per-round launches."""
import os, sys, pathlib
import numpy as np
ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import jolt_b200
from jolt_b200 import BatchMember, LOW_TO_HIGH, HIGH_TO_LOW, Polynomial, ProductMember
from jolt_b200 import field as F
from oracle.coracle import rand_limbs

lg = int(sys.argv[1]) if len(sys.argv) > 1 else 22
order = LOW_TO_HIGH
tabs = [rand_limbs(1 + j, 1 << lg) for j in range(2)]

def run(env):
    os.environ.pop("JB_NO_TAIL", None)
    for k in env:
        os.environ[k] = "1"
    sess = jolt_b200.Session(0)
    probe = ProductMember(sess, [Polynomial.new(sess, t) for t in tabs], order)
    ev = probe.prove_round_evals(None, 0)
    claim = (ev[0] + ev[1]) % F.R_MOD
    probe.close()
    outs = []
    for rep in range(3):
        mem = ProductMember(sess, [Polynomial.new(sess, t) for t in tabs], order)
        res = jolt_b200.prove_batch_native([BatchMember(claim, 1, lg, 0)], [mem], lg, 2, claim, seed=7)
        fe = mem.final_evals()
        mem.close()
        ok = fe[0] * fe[1] % F.R_MOD == res.final_claim
        outs.append((ok, res.final_claim, fe, [p.coefficients for p in res.round_polynomials]))
    sess.close()
    return outs

a = run(["JB_NO_TAIL"])
c = run([])
print("launched ok:", [o[0] for o in a])
print("resident ok:", [o[0] for o in c], "== launched:", [o[1:] == a[0][1:] for o in c])
for o in c:
    if o[1:] != a[0][1:]:
        diff = [i for i, (p, q) in enumerate(zip(o[3], a[0][3])) if p != q]
        print("first differing round polys:", diff[:5], "final evals equal:", o[2] == a[0][2])
        break
