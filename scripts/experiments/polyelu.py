"""Exhaustive CPU emulation of the packed-fp16 ELU of the batched kernel (kernels_tc.cuh: elu_neg_poly_f16x2, elu_pack16).

Both exponential paths take x = -|z'| and the result is max.NaN(z', c*2^x - c) (kEluMax, 0 <= alpha <= 1) or the
z' < 0 select (kEluSelect).  Every fp16 input is checked against the fp64 ELU: finite negatives (the error bound),
non-negatives (must pass through bit-exactly), NaN (must stay NaN).  The last part is the local search over
fp16-representable neighbours of the polynomial's coefficients that chose them."""
import itertools
import numpy as np

f16 = np.float16
def h(x): return np.asarray(x, dtype=np.float32).astype(f16)
def fma16(a, b, c): return h(a.astype(np.float32) * b.astype(np.float32) + c.astype(np.float32))  # single rounding approx (f32 exact product of 11-bit; sum rounding in f32 then f16)
def add16(a, b): return h(a.astype(np.float32) + b.astype(np.float32))
def negabs(z16): return (z16.view(np.uint16) | np.uint16(0x8000)).view(f16)
BASE = [0.1103433, 0.4852223, 1.3865219, 1.9998561]

def poly_exp_branch(z16, c, coef=BASE):
    """c*2^x - c for x = -|z16| on the FMA pipe (elu_neg_poly_f16x2)."""
    M = h(1536.0)
    xc = np.maximum(negabs(z16), h(-13.0))           # max.f16x2: a NaN operand yields the other one
    xc = np.where(np.isnan(z16), h(-13.0), xc)
    u = add16(M, -xc)
    kf = add16(u, -M)
    r = add16(xc, kf)
    a3, a2, a1, a0 = [h(v) for v in coef]
    p = fma16(np.broadcast_to(a3, r.shape), r, np.broadcast_to(a2, r.shape))
    p = fma16(p, r, np.broadcast_to(a1, r.shape))
    p = fma16(p, r, np.broadcast_to(a0, r.shape))
    km = (u.view(np.uint16) & 0xF).astype(np.uint16)
    res = (p.view(np.uint16) - (km << 10)).astype(np.uint16).view(f16)
    return fma16(res, np.broadcast_to(h(c / 2), r.shape), np.broadcast_to(h(-c), r.shape))

def mufu_exp_branch(z16, c):
    """the same with a correctly rounded fp16 2^x standing in for ex2.approx.f16x2"""
    e16 = h(np.exp2(negabs(z16).astype(np.float64)))
    return fma16(e16, np.broadcast_to(h(c), z16.shape), np.broadcast_to(h(-c), z16.shape))

def select_max(z16, e): return np.maximum(z16, e)            # max.NaN: NaN if either operand is NaN
def select_neg(z16, e): return np.where(z16 < 0, e, z16)     # HSET2.LT + LOP3

every = np.arange(0, 0x10000, dtype=np.uint32).astype(np.uint16).view(f16)
every = every[~np.isinf(every)]
neg, nonneg, nan = every < 0, every >= 0, np.isnan(every)

def check(name, alpha, exp_branch, select):
    c = alpha * 1.4426950408889634
    out = select(every, exp_branch(every, c))
    z = every.astype(np.float64)
    with np.errstate(over="ignore", invalid="ignore"):    # the discarded branch of large positive inputs
        ref = np.where(z < 0, c * (np.exp2(z) - 1), z)
    err = np.abs(out.astype(np.float64)[neg] - ref[neg]).max()
    passthru = np.array_equal(out[nonneg].view(np.uint16), every[nonneg].view(np.uint16))
    print(f"{name:28s} alpha {alpha:4}: max abs err over negative inputs {err:.2e}, non-negative inputs pass through "
          f"bit-exactly: {passthru}, NaN stays NaN: {bool(np.isnan(out[nan]).all())}")
    return err

for alpha in (1.0, 0.5, 0.0):
    check("polynomial + max.NaN", alpha, poly_exp_branch, select_max)
    check("polynomial + select", alpha, poly_exp_branch, select_neg)
    check("ideal 2^x + max.NaN", alpha, mufu_exp_branch, select_max)
    check("ideal 2^x + select", alpha, mufu_exp_branch, select_neg)
# alpha > 1: c*(2^z - 1) < z just below 0, the max picks z -- such layers keep the select (kEluSelect)
check("polynomial + max.NaN", 1.5, poly_exp_branch, select_max)
check("polynomial + select", 1.5, poly_exp_branch, select_neg)

# local search over fp16-representable coefficient neighbours (alpha = 1)
def err(coef):
    c = 1.4426950408889634
    z = every[neg]
    return np.abs(select_max(z, poly_exp_branch(z, c, coef)).astype(np.float64) - c * (np.exp2(z.astype(np.float64)) - 1)).max()
best = (err(BASE), BASE)
cands = []
for b in BASE:
    bits = int(h(b).view(np.uint16))
    cands.append([float(np.uint16(bits + d).view(f16)) for d in (-2, -1, 0, 1, 2)])
for co in itertools.product(*cands):
    e = err(list(co))
    if e < best[0]:
        best = (e, list(co))
print("coefficient search: shipped", BASE, f"{err(BASE):.2e}", "best neighbour", best[1], f"{best[0]:.2e}")
