"""K3 projections checked directly against fp64 (kernel_ref.gemm_ref) in every kernel variant, epilogue class and instance
layout the update and the rollout launch, through sgrl_gemm_desc (include/sgrl_b200.h).

Every case
  - fills C with NaN (random values for accumulate cases) and leaves columns past N (ldc > N) and two rows past M of every
    instance as sentinels that must come back bit-identical, likewise rowsum / gram_f / gram_g past what the call writes;
  - gives every instance its own data in every operand (z-stride 0 only where a case broadcasts A or B);
  - asserts the plan the library reports (kernel variant, split kind, epilogue class, TMA store), so that a change of the
    planner cannot turn it into a test of another variant;
  - bounds the error of every element by its own scale: |C - ref| <= tol * (|alpha| |A| |B|^T + |bias| + |res| (+ |C0|)),
    divided by |rowdiv| and scaled by |colscale| like the value, and reports the worst element as (z, row, column).

Tolerances: 4x the worst ratio measured per path on a B200 (power limit 1000 W), rounded up to two digits:
    path      worst measured   tolerance
    simt      1.76e-07         7.1e-07     fp32 SIMT tile and skinny kernels
    deep      4.09e-07         1.7e-06     3xTF32 tile kernel: BN 64 / 128, every layout, GRAM, atomic split-K, groups
    sm2       1.33e-06         5.4e-06     two CTAs per SM: one accumulator for all three product terms
    csk       2.08e-07         8.4e-07     cluster split-K, 2 and 3 ranks
    persist   1.35e-06         5.4e-06     persistent plain and GRAM kernels (one accumulator)
    bf16      2.61e-07         1.1e-06     BF16-input mode, against the bf16-rounded operands
test_plan_coverage pins the set of (variant, split kind, epilogue class, TMA store) the cases reach.
"""
import pytest
import torch

import kernel_ref as R
from sgrl_b200.packing import GP_K

pytestmark = pytest.mark.gpu

TOL = {"simt": 7.1e-07, "deep": 1.7e-06, "sm2": 5.4e-06, "csk": 8.4e-07, "persist": 5.4e-06, "bf16": 1.1e-06}
PLAN = ("path", "bn", "amn", "bmn", "bpre", "sm2", "gram", "persist", "split", "sk_x", "cluster", "tma_c", "epi")


def r4(n):
    return (n + 3) // 4 * 4


# ------------------------------------------------------------------------------------------------ problems
def problem(seed, M, N, K, nb=1, ta=0, tb=0, pre=True, epi=(), acc=0, splitk=1, bcast=(), gram=False, gram_g=False, gd=False,
            alpha=0.75, colscale_n=256, ldc=None):
    """One SgrlGemmProblem as a dict of flat CUDA buffers (kernel_ref.gemm_ref's format).  epi: any of bias, relu, rowdiv,
    colscale, mask, res1, res2, rowsum.  bcast: "A" / "B" get z-stride 0."""
    g = torch.Generator(device="cuda").manual_seed(seed)

    def rnd(n, scale=1.0):
        return torch.randn(r4(n) + 16, device="cuda", generator=g) * scale

    def nan(n):
        return torch.full((r4(n) + 16,), float("nan"), device="cuda")
    pr = dict(M=M, N=N, K=K, nb=nb, trans_a=ta, trans_b=tb, alpha=alpha, accumulate=acc, splitk=splitk, relu=int("relu" in epi),
              colscale=0.37, colscale_n=colscale_n if "colscale" in epi else 0)
    if gram:
        zs = r4(M * GP_K) + 8
        pr.update(A=None, lda=0, zs_a=0, gram_z=rnd(nb * zs, 0.5), zs_gram_z=zs, gram_f=nan(nb * zs), gram_g=nan(nb * zs) if gram_g else None)
    else:
        rows, cols = (K, M) if ta else (M, K)
        pr["lda"] = r4(cols) + 4
        pr["zs_a"] = 0 if "A" in bcast else rows * pr["lda"] + 4
        pr["A"] = rnd(max(nb * pr["zs_a"], rows * pr["lda"]))
    rows, cols = (K, N) if tb else (N, K)
    pr["ldb"] = r4(cols) + 4
    pr["zs_b"] = 0 if "B" in bcast else rows * pr["ldb"] + 4
    pr["B"] = rnd(max(nb * pr["zs_b"], rows * pr["ldb"]), K ** -0.5)
    pr["B_hi"] = pr["B_lo"] = None
    if pre:
        from sgrl_b200._lib import lib, ptr, stream, check
        pr["B_hi"], pr["B_lo"] = torch.empty_like(pr["B"]), torch.empty_like(pr["B"])
        check(lib.sgrl_split_tf32(ptr(pr["B"]), ptr(pr["B_hi"]), ptr(pr["B_lo"]), pr["B"].numel(), stream()), "split")
    pr["ldc"] = ldc or r4(N) + 4
    pr["zs_c"] = (M + 2) * pr["ldc"]                           # two sentinel rows per instance
    if acc:
        C = rnd(nb * pr["zs_c"])
        C.view(-1)[:nb * pr["zs_c"]].view(nb, M + 2, pr["ldc"])[:, M:, :] = float("nan")
        C.view(-1)[:nb * pr["zs_c"]].view(nb, M + 2, pr["ldc"])[:, :, N:] = float("nan")
        pr["C"] = C
    else:
        pr["C"] = nan(nb * pr["zs_c"])
    if "bias" in epi:
        pr["zs_bias"] = r4(N) + 4
        pr["bias"] = rnd(nb * pr["zs_bias"])
    if "rowdiv" in epi:
        pr["zs_rowdiv"] = r4(M) + 4
        pr["rowdiv"] = rnd(nb * pr["zs_rowdiv"]).abs() * 3 + 0.5
    for k in ("mask", "res1", "res2"):
        if k in epi:
            ld = r4(N) + 8
            pr["ld" + k] = ld
            pr["zs_" + k] = M * ld + 4
            pr[k] = rnd(nb * pr["zs_" + k])
    if "rowsum" in epi:
        pr["zs_rowsum"] = r4(M) + 4
        rs = rnd(nb * pr["zs_rowsum"])
        for z in range(nb):
            rs[z * pr["zs_rowsum"] + M:(z + 1) * pr["zs_rowsum"]] = float("nan")
        pr["rowsum"] = rs
    if gd:
        pr["zs_gd"] = r4(2 * M) + 4
        pr["gd"] = rnd(nb * pr["zs_gd"])
    return pr


def _fill(dst, pr):
    from sgrl_b200._lib import ptr
    for f, _ in dst._fields_:
        if f in pr and pr[f] is not None:
            v = pr[f]
            setattr(dst, f, ptr(v) if torch.is_tensor(v) else v)


def run(prs, use_tc=1, sm2_ok=0, **over):
    """sgrl_gemm_desc on 1..4 problems; returns (list of plan dicts, launches)."""
    import ctypes as C
    from sgrl_b200._lib import GemmDesc, GemmPlanInfo, lib, stream, check
    d = GemmDesc()
    d.n, d.use_tc, d.sm2_ok = len(prs), use_tc, sm2_ok
    for f in ("bn", "split", "csk", "sm2", "persist", "tma_store", "group"):
        setattr(d, f, over.pop(f, -1))
    assert not over, over
    for i, pr in enumerate(prs):
        _fill(d.pr[i], pr)
    info = GemmPlanInfo()
    check(lib.sgrl_gemm_desc(C.byref(d), C.byref(info), stream()), "sgrl_gemm_desc")
    torch.cuda.synchronize()
    return [{f: getattr(info.pr[i], f) for f in PLAN} for i in range(len(prs))], info.launches


def compare(pr, outs, ref):
    """Worst error ratio over every output of one problem; asserts the sentinels and that no written element is NaN."""
    worst = (0.0, None)
    for name, (val, bound, written) in ref.items():
        got = outs[name]
        n = val.numel()
        gw, orig = got[:n], pr[name][:n]
        assert torch.equal(gw[~written].view(torch.int32), orig[~written].view(torch.int32)), f"{name}: an entry it must not write changed"
        g64 = gw.double()
        assert not torch.isnan(g64[written]).any(), f"{name}: NaN in the written entries"
        ratio = torch.zeros_like(val)
        ratio[written] = (g64[written] - val[written]).abs() / (bound[written] + 1e-30)
        i = int(ratio.argmax())
        if ratio[i].item() > worst[0]:
            zs = {"C": pr["zs_c"], "rowsum": pr.get("zs_rowsum"), "gram_f": pr.get("zs_gram_z"), "gram_g": pr.get("zs_gram_z")}[name]
            ld = {"C": pr["ldc"], "rowsum": 1, "gram_f": 1, "gram_g": GP_K}[name]
            z, r = divmod(i, zs)
            worst = (ratio[i].item(), f"{name}[z={z}, row={r // ld}, col={r % ld}] = {g64[i].item():.9g} vs {val[i].item():.9g}")
    return worst


def path_of(p, use_tc):
    if p["path"] != 2:
        return "simt"
    if use_tc == 2:
        return "bf16"
    return "persist" if p["persist"] else "sm2" if p["sm2"] else "csk" if p["cluster"] > 1 else "deep"


def coverage_key(p):
    if p["path"] != 2:
        v = "simt" if p["path"] == 0 else "skinny"
    else:
        v = f"bn{p['bn']}" + "".join(f"-{k}" for k in ("amn", "bmn", "bpre", "sm2", "gram", "persist") if p[k])
    sk = f"csk{p['cluster']}" if p["cluster"] > 1 else ("atomic" if p["split"] > 1 else "none")
    return (v, sk, p["epi"], p["tma_c"])


def execute(c):
    """Run one case of CASES: returns (plans, launches, [(path, worst ratio, where)] per problem)."""
    prs = [problem(**a) for a in c["probs"]]
    before = [{k: v.clone() for k, v in pr.items() if torch.is_tensor(v)} for pr in prs]
    use_tc = c.get("call", {}).get("use_tc", 1)
    refs = [R.gemm_ref({**pr, **b}, bf16=use_tc == 2) for pr, b in zip(prs, before)]
    plans, launches = run(prs, **c.get("call", {}))
    res = []
    for pr, b, ref, p in zip(prs, before, refs, plans):
        w, where = compare({**pr, **b}, {k: pr[k] for k in ref}, ref)
        res.append((path_of(p, use_tc), w, where))
    return plans, launches, res


# ------------------------------------------------------------------------------------------------ the matrix
CASES = {}


def case(cid, probs, expect, launches=None, **call):
    """probs: problem() keyword dicts; expect: per problem, the plan fields that must hold (dict) or one dict for all."""
    probs = probs if isinstance(probs, list) else [probs]
    expect = expect if isinstance(expect, list) else [expect] * len(probs)
    CASES[cid] = dict(probs=probs, expect=expect, launches=launches, call=call)


def P(seed, M, N, K, **kw):
    return dict(seed=seed, M=M, N=N, K=K, **kw)


DEEP = dict(sm2=0, persist=0, csk=0)
# every instantiation of tc_go_deep64 / tc_go_deep128: BN x {K-major, B MN-major, both MN-major, A MN-major} x {pre-split, on the fly}
for bn in (64, 128):
    for ta, tb in ((0, 0), (0, 1), (1, 1), (1, 0)):
        for pre in (True, False):
            tma = (ta + tb + pre) % 2          # half of them through the TMA store, the others with residuals or st.global
            epi = ("bias", "relu") if tma or not ta else ("mask", "res1", "res2")
            case(f"deep-bn{bn}-a{ta}b{tb}-pre{int(pre)}", P(100 + bn + 4 * ta + 2 * tb + pre, 300, 192, 256, ta=ta, tb=tb, pre=pre, epi=epi),
                 dict(path=2, bn=bn, amn=ta, bmn=tb, bpre=int(pre), sm2=0, persist=0, cluster=1, split=1, tma_c=tma,
                      epi=-1 if tma else 0 if "bias" in epi else 6),
                 bn=bn, tma_store=tma, **DEEP)

# two CTAs per SM (inference passes): reciprocal row division, through the TMA store and through st.global
for bn in (64, 128):
    for tb in (0, 1):
        tma = (bn == 64) ^ tb
        case(f"sm2-bn{bn}-b{tb}-tma{int(tma)}", P(200 + bn + tb, 2304, 256, 256, tb=tb, epi=("bias", "relu", "rowdiv", "colscale")),
             dict(path=2, bn=bn, sm2=1, bmn=tb, tma_c=int(tma), epi=-1 if tma else 1), bn=bn, sm2=1, tma_store=int(tma), persist=0, csk=0, sm2_ok=1)

# GRAM (A rows generated from Z), with and without keeping the rows; the persistent GRAM kernel
for bn in (64, 128):
    for keep in (0, 1):
        case(f"gram-bn{bn}-G{keep}", P(300 + bn + keep, 300, 256, GP_K, gram=True, gram_g=bool(keep), epi=("bias", "relu"), nb=2),
             dict(path=2, bn=bn, gram=1, persist=0, epi=0, tma_c=0), bn=bn, persist=0, tma_store=0)
case("gram-persist", P(310, 1000, 256, GP_K, gram=True, epi=("bias", "relu"), nb=2), dict(path=2, gram=1, persist=1, epi=-1), persist=1, sm2_ok=1)

# persistent plain and [X P^T | gd]; the gd epilogue of the tile kernel (vector, class 7) and the generic one (ragged ldc)
case("persist-plain", P(320, 1000, 384, 256, epi=("bias", "rowdiv", "colscale"), colscale_n=100, nb=2), dict(path=2, bn=128, persist=1, epi=-1),
     persist=1, sm2_ok=1)
case("persist-gd", P(321, 3 * 1000, 32, 128, gd=True, ldc=32), dict(path=2, persist=1, tma_c=0, epi=-1), persist=1, sm2_ok=1)
case("gd-tile", P(322, 3 * 700, 32, 256, gd=True, ldc=32, nb=2), dict(path=2, persist=0, epi=7), persist=0)
case("gd-generic", P(323, 3 * 700, 32, 256, gd=True, ldc=33), dict(path=2, persist=0, epi=6), persist=0)

# cluster split-K: 2 and 3 ranks under every epilogue class that may not use atomics
CSK_EPI = {1: dict(epi=("bias", "relu", "rowdiv", "colscale"), colscale_n=100), 2: dict(epi=("mask",)), 3: dict(epi=("res1", "res2")),
           4: dict(acc=1), 6: dict(epi=("bias", "mask", "relu"))}
for ranks in (2, 3):
    for ek, kw in CSK_EPI.items():
        case(f"csk{ranks}-epi{ek}", P(400 + 10 * ranks + ek, 300, 256, 1024, **kw), dict(path=2, cluster=ranks, split=1, epi=ek, tma_c=0),
             csk=ranks, sm2=0, persist=0)
case("csk-model", P(420, 900, 256, 1152, epi=("rowdiv", "colscale")), dict(path=2, bn=128, cluster=3, epi=1))     # 16 tiles, 36 k-blocks

# atomic split-K folded into blockIdx.x (weight gradients dW += alpha dY^T X), with the fused bias gradient
WG = dict(ta=1, tb=1, pre=False, acc=1, splitk=8)
case("split-rowsum", P(500, 256, 128, 2304, epi=("rowsum",), **WG), dict(path=2, bn=128, split=4, sk_x=1, epi=5, amn=1, bmn=1), split=4, bn=128)
case("split-rowsum-4tiles", P(505, 256, 256, 2304, epi=("rowsum",), **WG), dict(path=2, bn=64, split=2, epi=5), split=2, bn=64)     # row sums from n0 = 0 only
case("split-empty-slice", P(501, 256, 128, 288, epi=("rowsum",), **WG), dict(path=2, split=4, sk_x=1, epi=5), split=4)     # 9 k-blocks: 3,3,3,0
case("split-bn128", P(502, 256, 256, 2304, **WG), dict(path=2, bn=128, split=6, epi=5), split=6, bn=128)
case("split-model", P(503, 30, 128, 2304, **WG), dict(path=2, sk_x=1, epi=5))            # the model splits small weight gradients
case("rowsum-kmajor", P(504, 256, 128, 2304, ta=0, tb=1, pre=False, acc=1, epi=("rowsum",)), dict(path=2, split=1, epi=4), csk=0)

# grouped launches (one launch for problems of one variant, unequal M; re-planned to BN = 128; disagreeing variants)
G = dict(pre=True, epi=("bias", "relu"))
case("group2", [P(600, 300, 128, 256, **G), P(601, 700, 128, 256, epi=("rowdiv", "colscale"))], dict(path=2, bn=128), launches=1)
case("group3-bn128", [P(602, 300, 64, 256, **G), P(603, 130, 128, 256, **G), P(604, 900, 256, 256, pre=True, epi=("rowdiv",))],
     dict(path=2, bn=128), launches=1)
case("group4-nb2", [P(605 + i, M, 128, 256, nb=2, **G) for i, M in enumerate((129, 300, 511, 64))], dict(path=2, bn=128), launches=1)
case("group-disagree", [P(610, 300, 128, 256, **G), P(611, 300, 128, 256, tb=1, pre=True), P(612, 200, 128, 256, **G)],
     [dict(bmn=0), dict(bmn=1), dict(bmn=0)], launches=3)
case("group-empty-first", [P(613, 0, 128, 256, **G), P(614, 300, 64, 256, **G), P(615, 300, 256, 256, **G)],
     [dict(), dict(bn=128), dict(bn=128)], launches=1)
case("group-off", [P(616, 300, 128, 256, **G), P(617, 400, 128, 256, **G)], dict(path=2), launches=2, group=0)

# every epilogue class of the tile kernel, with the TMA store on and off where it applies
E = dict(bn=64, **DEEP)
for tma in (0, 1):
    case(f"epi0-tma{tma}", P(700 + tma, 700, 256, 256, epi=("bias", "relu")), dict(epi=-1 if tma else 0, tma_c=tma), tma_store=tma, **E)
    for cn in (256, 100):
        case(f"epi1-cs{cn}-tma{tma}", P(702 + tma + cn, 700, 768, 256, epi=("bias", "rowdiv", "colscale"), colscale_n=cn),
             dict(epi=-1 if tma else 1, tma_c=tma), tma_store=tma, **E)
case("epi2-mask", P(710, 700, 256, 256, epi=("mask",)), dict(epi=2), **E)
case("epi3-res1", P(711, 700, 256, 256, epi=("res1",)), dict(epi=3), **E)
case("epi3-res12", P(712, 700, 256, 256, epi=("res1", "res2")), dict(epi=3), **E)
case("epi4-acc", P(713, 700, 256, 256, acc=1), dict(epi=4), **E)
case("epi6-acc-bias", P(714, 700, 256, 256, acc=1, epi=("bias", "relu")), dict(epi=6), **E)
case("epi6-colscale", P(715, 700, 256, 256, epi=("colscale",), colscale_n=100), dict(epi=6), **E)
case("epi6-all", P(716, 700, 256, 256, epi=("bias", "relu", "rowdiv", "colscale", "mask", "res1", "res2"), colscale_n=40, acc=1),
     dict(epi=6), **E)

# shape edges: M tails of 1 and 127 rows, N % 4 != 0, N = 30 / 252, K = 16 and K % 32 != 0
for M in (129, 255):
    case(f"mtail{M}", P(800 + M, M, 256, 512, epi=("bias", "relu")), dict(path=2, epi=0), tma_store=0, **E)
for N in (130, 30, 252):
    case(f"ntail{N}", P(810 + N, 1000, N, 256, epi=("bias", "rowdiv"), ldc=r4(N) + 4), dict(path=2, tma_c=0 if N % 4 else 1), **DEEP)
case("ntail-acc", P(815, 1000, 130, 256, acc=1), dict(path=2, epi=4), **DEEP)
case("k16", P(820, 2304, 64, 16, epi=("bias",)), dict(path=2), **DEEP)
case("k100", P(821, 1000, 256, 100, epi=("mask", "res1")), dict(path=2, epi=6), **DEEP)
case("threshold", P(822, 64, 128, 256, epi=("bias",)), dict(path=2))                  # M N K = 2^21: the smallest tcgen05 problem

# SIMT and skinny kernels (use_tc = 0), the rollout sizes of B = 1..3 and below the tcgen05 threshold
for M in (1, 9, 32):
    case(f"skinny{M}", P(830 + M, M, 252, 128, pre=False, epi=("bias", "relu", "rowdiv", "colscale", "res1", "res2"), colscale_n=100, nb=2),
         dict(path=1), use_tc=0)
case("simt-33", P(833, 33, 252, 128, pre=False, epi=("bias", "relu", "mask")), dict(path=0), use_tc=0)
case("simt-all", P(834, 300, 130, 145, ta=1, tb=1, pre=False, nb=2, acc=1, epi=("bias", "relu", "rowdiv", "colscale", "mask", "res1", "res2")),
     dict(path=0), use_tc=0)
case("simt-split", P(835, 256, 128, 900, ta=1, tb=1, pre=False, acc=1, splitk=3), dict(path=0, split=3), use_tc=0)
case("simt-below-threshold", P(836, 64, 128, 255, pre=False, epi=("bias",)), dict(path=0), use_tc=0)

# instances: nb = 2, 5, 16 with every operand per instance; A or B shared (z-stride 0)
case("nb2-acc-res", P(900, 300, 256, 256, nb=2, acc=1, epi=("res1", "res2")), dict(path=2, epi=6), **E)
case("nb5-generic", P(901, 300, 256, 256, nb=5, epi=("bias", "relu", "rowdiv", "colscale", "mask", "res1", "res2")), dict(epi=6), **E)
case("nb5-mask", P(902, 300, 256, 256, nb=5, epi=("mask",)), dict(epi=2), **E)
case("nb16-rowdiv", P(903, 130, 64, 256, nb=16, epi=("bias", "rowdiv", "colscale"), colscale_n=32), dict(epi=1), tma_store=0, **E)
case("nb16-tma", P(904, 130, 64, 256, nb=16, epi=("bias", "rowdiv")), dict(tma_c=1), tma_store=1, **E)
case("nb2-rowsum-split", P(905, 256, 128, 1152, nb=2, epi=("rowsum",), **WG), dict(split=3, epi=5), split=3)
case("bcast-A", P(906, 300, 256, 256, nb=5, bcast=("A",), epi=("bias", "res1")), dict(path=2), tma_store=0, **E)
case("bcast-B", P(907, 300, 256, 256, nb=5, bcast=("B",), epi=("bias", "relu")), dict(path=2), **E)
case("csk3-nb2", P(908, 130, 256, 1024, nb=2, epi=("mask",)), dict(cluster=3, epi=2), csk=3, sm2=0, persist=0)

# BF16-input mode (against the bf16-rounded operands)
case("bf16-fwd", P(950, 1000, 256, 256, epi=("bias", "relu")), dict(path=2), use_tc=2, **DEEP)
case("bf16-fly-dgrad", P(951, 1000, 256, 256, tb=1, pre=False, acc=1), dict(path=2, bpre=0, epi=4), use_tc=2, **DEEP)
case("bf16-wgrad", P(952, 256, 128, 2304, epi=("rowsum",), **WG), dict(path=2, split=4), split=4, use_tc=2)
case("bf16-sm2", P(953, 2304, 256, 256, epi=("bias", "rowdiv")), dict(path=2, sm2=1), sm2=1, persist=0, use_tc=2, sm2_ok=1)
case("bf16-persist", P(954, 1000, 256, 256, epi=("bias",)), dict(path=2, persist=1), persist=1, use_tc=2, sm2_ok=1)


# ------------------------------------------------------------------------------------------------ tests
@pytest.fixture(scope="module")
def results():
    return {cid: execute(c) for cid, c in CASES.items()}


@pytest.mark.parametrize("cid", list(CASES))
def test_gemm_variant(results, cid):
    plans, launches, res = results[cid]
    c = CASES[cid]
    for i, (p, exp) in enumerate(zip(plans, c["expect"])):
        if c["probs"][i]["M"] == 0:
            continue
        bad = {k: (p[k], v) for k, v in exp.items() if p[k] != v}
        assert not bad, f"problem {i}: plan {p} differs from the expected {bad} (got, expected)"
    if c["launches"] is not None:
        assert launches == c["launches"]
    for i, (path, w, where) in enumerate(res):
        assert w <= TOL[path], f"problem {i} ({path}): error {w:.3g} x bound at {where} (tolerance {TOL[path]:.1g})"


COVERAGE = [      # (variant, split kind, epilogue class, TMA store) of every case; epilogue class -1: TMA-store or persistent epilogue
    ('bn128', 'none', 0, 0),
    ('bn128-amn', 'none', -1, 1),
    ('bn128-amn-bmn', 'atomic', 5, 0),
    ('bn128-amn-bmn', 'none', 6, 0),
    ('bn128-amn-bmn-bpre', 'none', -1, 1),
    ('bn128-amn-bpre', 'none', 6, 0),
    ('bn128-bmn', 'none', -1, 1),
    ('bn128-bmn', 'none', 4, 0),
    ('bn128-bmn-bpre', 'none', 0, 0),
    ('bn128-bmn-bpre-sm2', 'none', -1, 1),
    ('bn128-bpre', 'csk2', 1, 0),
    ('bn128-bpre', 'csk2', 2, 0),
    ('bn128-bpre', 'csk2', 3, 0),
    ('bn128-bpre', 'csk2', 4, 0),
    ('bn128-bpre', 'csk2', 6, 0),
    ('bn128-bpre', 'csk3', 1, 0),
    ('bn128-bpre', 'csk3', 2, 0),
    ('bn128-bpre', 'csk3', 3, 0),
    ('bn128-bpre', 'csk3', 4, 0),
    ('bn128-bpre', 'csk3', 6, 0),
    ('bn128-bpre', 'none', -1, 1),
    ('bn128-bpre', 'none', 1, 0),
    ('bn128-bpre', 'none', 4, 0),
    ('bn128-bpre', 'none', 6, 0),
    ('bn128-bpre-gram', 'none', 0, 0),
    ('bn128-bpre-persist', 'none', -1, 0),
    ('bn128-bpre-persist', 'none', -1, 1),
    ('bn128-bpre-sm2', 'none', -1, 1),
    ('bn128-bpre-sm2', 'none', 1, 0),
    ('bn256-bpre-gram-persist', 'none', -1, 1),
    ('bn64', 'none', 0, 0),
    ('bn64-amn', 'none', -1, 1),
    ('bn64-amn-bmn', 'atomic', 5, 0),
    ('bn64-amn-bmn', 'none', 6, 0),
    ('bn64-amn-bmn-bpre', 'none', -1, 1),
    ('bn64-amn-bpre', 'none', 6, 0),
    ('bn64-bmn', 'none', -1, 1),
    ('bn64-bmn', 'none', 4, 0),
    ('bn64-bmn-bpre', 'none', -1, 1),
    ('bn64-bmn-bpre', 'none', 0, 0),
    ('bn64-bmn-bpre-sm2', 'none', 1, 0),
    ('bn64-bpre', 'none', -1, 1),
    ('bn64-bpre', 'none', 0, 0),
    ('bn64-bpre', 'none', 1, 0),
    ('bn64-bpre', 'none', 2, 0),
    ('bn64-bpre', 'none', 3, 0),
    ('bn64-bpre', 'none', 4, 0),
    ('bn64-bpre', 'none', 6, 0),
    ('bn64-bpre', 'none', 7, 0),
    ('bn64-bpre-gram', 'none', 0, 0),
    ('bn64-bpre-sm2', 'none', -1, 1),
    ('simt', 'atomic', -1, 0),
    ('simt', 'none', -1, 0),
    ('skinny', 'none', -1, 0),
]


def test_plan_coverage(results):
    """The cases reach exactly this set of kernel variants, split kinds, epilogue classes and store paths: a planner change
    that moves a case onto another variant fails here instead of leaving the variant untested."""
    got = sorted({coverage_key(p) for cid, (plans, _, _) in results.items() for p, a in zip(plans, CASES[cid]["probs"]) if a["M"] > 0})
    assert got == sorted(COVERAGE), got


def test_deterministic_mode_is_bit_reproducible():
    """Deterministic mode: no atomic split-K and no cluster split-K, and two runs give bit-identical C and rowsum."""
    from sgrl_b200._lib import lib
    prev = lib.sgrl_deterministic(1)
    try:
        outs = []
        for _ in range(2):
            a = P(960, 256, 128, 2304, epi=("rowsum",), **WG)
            b = P(961, 300, 256, 1024, epi=("bias", "relu", "rowdiv"))
            pa, pb = problem(**a), problem(**b)
            (plan_a,), _ = run([pa])
            (plan_b,), _ = run([pb])
            assert plan_a["split"] == 1 and plan_a["cluster"] == 1 and plan_b["cluster"] == 1, (plan_a, plan_b)
            outs.append((pa["C"].clone(), pa["rowsum"].clone(), pb["C"].clone()))
        for x, y in zip(*outs):
            assert torch.equal(x.view(torch.int32), y.view(torch.int32))
    finally:
        lib.sgrl_deterministic(prev)


def test_split_k_bias_is_refused_on_both_paths():
    """Regression: the tcgen05 atomic split-K epilogue dropped the bias (the SIMT kernel added it once), so the same
    sgrl_gemm call gave shape-dependent results.  splitk > 1 with a bias, or without accumulate, is now refused."""
    from sgrl_b200._lib import lib, ptr, stream
    pr = problem(**P(970, 30, 128, 2304, ta=1, tb=1, pre=False, acc=1, epi=("bias",)))
    for use_tc in (0, 1):
        rc = lib.sgrl_gemm(ptr(pr["A"]), pr["lda"], 1, ptr(pr["B"]), pr["ldb"], 1, ptr(pr["C"]), pr["ldc"], 30, 128, 2304, 1.0,
                           ptr(pr["bias"]), None, 0, 1, 8, use_tc, stream())
        assert rc < 0 and b"no bias" in lib.sgrl_last_error()

