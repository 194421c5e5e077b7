"""GPU: the embedding lookup and the row-update backward of a LookupPlan at every width, optimiser and decomposition edge, against
float64 references (oracle/embedding_ref.py, optim_ref.py, ftrl_ref.py).

Backward (hrb_lookup_bwd_update).  Every case runs two steps on different ids from tables and optimiser slots initialised on the
device by init_uniform (nonzero slots: Adam at steps 5 and 6), with one dense-gradient table in most plans.  The host forms only
the touched rows' initial values (hash_uniform_rows) and their float64 updates; every untouched row and slot must keep its bits.
Each case runs twice (bit-equal) and once under torch.profiler, which must show the kernels of the path the unit-decomposition
restatement predicts: bwd_unit_kernel<MODE, G> for every width of the plan, bwd_unit_combine_kernel when a row is split over
slices, split_kernel only on that path; bwd_chunk_kernel / bwd_merge_kernel, bwd_hot_slice_kernel for tables of <= 128 rows and
bwd_long_detect_kernel on the sorted one.  Tolerances follow test_gpu_parity.py (atol = tol * max|ref|).

Forward (hrb_lookup_fwd / hrb_lookup_fm_fwd): each of lookup_tile_kernel, lookup_rows_kernel and lookup_items_kernel at every width
it admits, gathers bit-exact, pooled and FM outputs within 1e-5, and check_ids raising from each kernel."""
import re

import numpy as np
import pytest
import torch

import oracle
from oracle.embedding_ref import plan_grad_sums, table_units, unit_counts, unit_path_taken
from oracle.ftrl_ref import ftrl_dense, ftrl_sparse
from oracle.optim_ref import adagrad_dense, adagrad_sparse, adam_lazy_sparse
from tests.test_gpu_parity import _zipf_ids, close, rnd

pytestmark = pytest.mark.gpu

MODES = ("sgd", "adam", "adagrad", "ftrl")
MODE_ID = {"sgd": 0, "adam": 1, "adagrad": 3, "ftrl": 4}  # UpdMode, the first template argument of the backward kernels
ALGOS = ("units", "sort")
TOL = {"sgd": 1e-4, "adam": 2e-4, "adagrad": 1e-4, "ftrl": 1e-4}
GRAD_TOL = 1e-4  # gradient sums of dense-gradient tables
LR = {"sgd": 0.1, "adam": 0.01, "adagrad": 0.1, "ftrl": 0.1}
FTRL = dict(l1=0.01, l2=0.01, lr_power=-0.5, l2_shrinkage=0.0)
SLOTS = {"sgd": [], "adam": [(-1e-2, 1e-2), (1e-4, 1e-3)], "adagrad": [(0.05, 0.5)], "ftrl": [(0.05, 0.5), (-0.2, 0.2)]}
ADAM_STEP0 = 5
DSCALE = 1e-2


def K():
    from handyrec_b200 import kernels

    return kernels


# ------------------------------------------------------------------------------------------------------------------------------
# cases: tables (rows, dim), fields (table, seq_len, pool, ids_col, out_col), dense-gradient tables, the ids of the two steps
# ------------------------------------------------------------------------------------------------------------------------------
def _case(shapes, fields, steps, dense=()):
    return {"shapes": shapes, "fields": fields, "steps": steps, "dense": set(dense)}


def _hist(g, B, L, rows, empty=True):
    """Pooled ids with front padding; with `empty`, ~10 % all-padding rows."""
    ids = torch.randint(1, rows, (B, L), generator=g, dtype=torch.int32)
    lens = torch.randint(0 if empty else 1, L + 1, (B,), generator=g)
    if empty:
        lens[torch.rand(B, generator=g) < 0.1] = 0
    return torch.where(torch.arange(L)[None] >= (L - lens)[:, None], ids, torch.zeros_like(ids))


def base_case(D, B, seed=0):
    """A tiny table (units: slices + combine; sort: hot rows), a 6-row table (single-row units), a large table under a plain and a
    mean-pooled field (id rows-1 in its short last unit, negative and out-of-range ids in both fields), and a dense-gradient
    table under a sum-pooled field with all-padding rows."""
    big = 100003 if D <= 128 else 20011
    shapes = [(2, D), (6, D), (big, D), (1000, D)]
    fields = [(0, 1, "none", 0, 0), (1, 1, "none", 1, D), (2, 1, "none", 2, 2 * D), (2, 5, "mean", 3, 3 * D), (3, 4, "sum", 8, 4 * D)]
    steps = []
    for s in range(2):
        g = torch.Generator().manual_seed(1000 * seed + 17 * s + D)
        c0 = torch.randint(0, 2, (B, 1), generator=g, dtype=torch.int32)
        c1 = torch.randint(0, 6, (B, 1), generator=g, dtype=torch.int32)
        c2 = torch.randint(0, big, (B, 1), generator=g, dtype=torch.int32)
        h = _hist(g, B, 5, big)
        q = _hist(g, B, 4, 1000)
        q[::5] = 0
        for i, (col, v) in enumerate(((c2, big - 1), (c2, -5), (c2, big), (h, -1), (h, big + 3), (h, big - 1))):
            if B > i + s:
                col[i + s, -1] = v
        steps.append(torch.cat([c0, c1, c2, h, q], 1).contiguous())
    return _case(shapes, fields, steps, dense=[3])


def cap64_case(D):
    """A 2-row table under a 10-long mean-pooled field whose ids are all 1 at B = 65536: 655360 positions on row 1, 64 slices."""
    B = 65536
    steps = []
    for s in range(2):
        ids = torch.ones(B, 11, dtype=torch.int32)
        if s:
            ids[::19, :3] = 0  # some padding in the second step
        ids[:, 10] = torch.randint(0, 5000, (B,), generator=torch.Generator().manual_seed(s), dtype=torch.int32)
        steps.append(ids)
    return _case([(2, D), (5000, D)], [(0, 10, "mean", 0, 0), (1, 1, "none", 10, D)], steps, dense=[1])


def zipf_case(D):
    """Zipf ids in a 2 M-row table: the first unit overflows (histogram split over the helper CTAs, single hot rows)."""
    B, V = 65536, 2_000_000
    steps = [torch.stack([_zipf_ids(B, V, 1.05, 40 + s), torch.randint(0, 1000, (B,), generator=torch.Generator().manual_seed(s),
                                                                        dtype=torch.int32)], 1) for s in range(2)]
    return _case([(V, D), (1000, D)], [(0, 1, "none", 0, 0), (1, 1, "none", 1, D)], steps, dense=[1])


def unit_list_case(D, n_first, hot_row=None):
    """A 2^20-row table at B = 65536 (32 units of 2^15 rows): exactly n_first positions land in the first unit's list; with hot_row,
    4097 of them name that one row."""
    B, V = 65536, 1 << 20
    rng = 1 << table_units(V, 1, B)[0]["shift"]
    steps = []
    for s in range(2):
        g = torch.Generator().manual_seed(7 + s)
        ids = torch.randint(rng, V, (B,), generator=g, dtype=torch.int32)
        ids[:n_first] = torch.randint(0, rng, (n_first,), generator=g, dtype=torch.int32)
        if hot_row is not None:
            ids[:4097] = hot_row
        ids = ids[torch.randperm(B, generator=g)]
        steps.append(torch.stack([ids, torch.randint(0, 1000, (B,), generator=g, dtype=torch.int32)], 1))
    return _case([(V, D), (1000, D)], [(0, 1, "none", 0, 0), (1, 1, "none", 1, D)], steps, dense=[1])


def long_runs_case(D):
    """Runs of 256, 257, 511, 512 and 513 positions (around the 256-position sampling of the long-run classification) between
    short ones."""
    B, V = 65536, 50000
    steps = []
    for s in range(2):
        g = torch.Generator().manual_seed(70 + s)
        ids = torch.randint(100, V, (B,), generator=g, dtype=torch.int32)
        o = 0
        for r, n in zip((11 + s, 12, 13, 14, 15), (256, 257, 511, 512, 513)):
            ids[o: o + n] = r
            o += n
        steps.append(ids[torch.randperm(B, generator=g)].reshape(B, 1))
    return _case([(V, D)], [(0, 1, "none", 0, 0)], steps)


def tiny33_case(D):
    """33 tables of 100 rows: the first 32 are the sorted path's host-known hot tables, the 33rd is not."""
    B = 4097
    steps = [torch.randint(0, 100, (B, 33), generator=torch.Generator().manual_seed(s), dtype=torch.int32) for s in range(2)]
    return _case([(100, D)] * 33, [(t, 1, "none", t, t * D) for t in range(33)], steps)


def bins_case(rows):
    """8 columns at B = 65536: 256 rows are 256 one-row units, 257 rows exceed the 256-unit limit."""
    B = 65536
    steps = [torch.randint(0, rows, (B, 8), generator=torch.Generator().manual_seed(s), dtype=torch.int32) for s in range(2)]
    return _case([(rows, 16)], [(0, 8, "sum", 0, 0)], steps)


def cols_case(L):
    """One mean-pooled field of L positions: 256 position columns per table is the unit path's limit."""
    B = 2048
    return _case([(5000, 16)], [(0, L, "mean", 0, 0)], [_hist(torch.Generator().manual_seed(s), B, L, 5000) for s in range(2)])


def mixed_case():
    """All six unit widths in one plan (six launch groups), a mean-pooled field on the 32-wide table."""
    B = 4097
    dims = [4, 8, 16, 32, 64, 128]
    shapes = [(3000 + 7 * i, d) for i, d in enumerate(dims)]
    fields, col = [], 0
    for t, d in enumerate(dims):
        fields.append((t, 1, "none", t, col))
        col += d
    fields.append((3, 3, "mean", 6, col))
    steps = []
    for s in range(2):
        g = torch.Generator().manual_seed(90 + s)
        steps.append(torch.cat([torch.randint(0, 3000, (B, 6), generator=g, dtype=torch.int32), _hist(g, B, 3, 3021)], 1))
    return _case(shapes, fields, steps)


# ------------------------------------------------------------------------------------------------------------------------------
# running a case
# ------------------------------------------------------------------------------------------------------------------------------
def _out_cols(case):
    return max(f[4] + case["shapes"][f[0]][1] for f in case["fields"])


def _douts(case):
    return [rnd(ids.shape[0], _out_cols(case), seed=300 + s, scale=DSCALE) for s, ids in enumerate(case["steps"])]


def _init(dev, case, mode):
    k = K()
    w, slots = [], [[] for _ in SLOTS[mode]]
    for t, (rows, d) in enumerate(case["shapes"]):
        w.append(k.init_uniform(torch.empty(rows, d, device=dev), 1000 + t))
        for j, (lo, hi) in enumerate(SLOTS[mode]):
            slots[j].append(k.init_uniform(torch.empty(rows, d, device=dev), 2000 + 10 * t + j, lo, hi))
    return w, slots


def _touched(case, mode, sums_per_step):
    """Per table: the rows any step changes (Ftrl: row 0 too where a pooled field's padding named it, unless dense-updated)."""
    out = []
    for t in range(len(case["shapes"])):
        r = [s[t]["rows"] for s in sums_per_step]
        if mode == "ftrl" and t not in case["dense"] and any(s[t]["pad"] for s in sums_per_step):
            r.append(torch.zeros(1, dtype=torch.long))
        out.append(torch.unique(torch.cat(r)))
    return out


def _reference(case, mode, l2_scale, douts, sums_per_step, touched):
    """float64 state of the touched rows after the case's steps: (weights, [slots], dense gradient or None) per table, plus the
    Ftrl elements whose |linear| came within rounding of l1 (the select may go either way there)."""
    lr = LR[mode]
    res = []
    for t, (rows, d) in enumerate(case["shapes"]):
        rr = touched[t].numpy()
        W = torch.from_numpy(oracle.hash_uniform_rows(rr, d, 1000 + t)).double()
        S = [torch.from_numpy(oracle.hash_uniform_rows(rr, d, 2000 + 10 * t + j, lo, hi)).double() for j, (lo, hi) in enumerate(SLOTS[mode])]
        amb = torch.zeros(len(rr), d, dtype=torch.bool)
        if t in case["dense"]:
            G = torch.zeros(len(rr), d, dtype=torch.float64)
            for sums in sums_per_step:
                G[np.searchsorted(rr, sums[t]["rows"].numpy())] += sums[t]["grad"]
            res.append((W, S, G, amb))
            continue
        for i, sums in enumerate(sums_per_step):
            rows_s, g = sums[t]["rows"], sums[t]["grad"]
            if mode == "ftrl" and sums[t]["pad"] and not bool((rows_s == 0).any()):
                rows_s = torch.cat([torch.zeros(1, dtype=torch.long), rows_s])
                g = torch.cat([torch.zeros(1, d, dtype=torch.float64), g])
            if len(rows_s) == 0:
                continue
            p = torch.from_numpy(np.searchsorted(rr, rows_s.numpy()))
            ar = torch.arange(len(p))
            if mode == "sgd":
                W[p] = W[p] - lr * (g + l2_scale * W[p])
            elif mode == "adam":
                W[p], S[0][p], S[1][p] = adam_lazy_sparse(W[p], S[0][p], S[1][p], ar, g, lr, step=ADAM_STEP0 + i, l2_scale=l2_scale)
            elif mode == "adagrad":
                if l2_scale:
                    W[p], S[0][p] = adagrad_dense(W[p], S[0][p], g, lr, l2_scale=l2_scale)
                else:
                    W[p], S[0][p] = adagrad_sparse(W[p], S[0][p], ar, g, lr)
            else:
                if l2_scale:
                    W[p], S[0][p], S[1][p] = ftrl_dense(W[p], S[0][p], S[1][p], g, lr, l2_scale=l2_scale, **FTRL)
                else:
                    W[p], S[0][p], S[1][p] = ftrl_sparse(W[p], S[0][p], S[1][p], ar, g, lr, **FTRL)
                amb[p] |= ((S[1][p].abs() - FTRL["l1"]).abs() <= 1e-5)
        res.append((W, S, None, amb))
    return res


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.key for e in prof.key_averages()}


def _has(names, pat):
    return any(re.search(pat, n) for n in names)


def _check_path(case, mode, algo, names):
    """The kernels seen are those of the path the restatement of build_units / unit_path_supported predicts."""
    shapes, fields = case["shapes"], case["fields"]
    B = case["steps"][0].shape[0]
    m = MODE_ID[mode]
    units = algo == "units" and unit_path_taken(shapes, fields, B)
    where = f"{algo} / {mode} / kernels seen: {sorted(n for n in names if 'bwd' in n or 'split' in n)}"
    if units:
        assert _has(names, r"split_kernel") and not _has(names, r"bwd_chunk_kernel"), where
        for G in sorted({d // 4 for _, d in shapes}):
            assert _has(names, rf"bwd_unit_kernel<{m}, {G}>"), f"no bwd_unit_kernel<{m}, {G}>: {where}"
        sliced = any(u["slices"] > 1 for t, (rows, d) in enumerate(shapes)
                     for u in table_units(rows, sum(f[1] for f in fields if f[0] == t), B))
        assert _has(names, rf"bwd_unit_combine_kernel<{m}, ") == sliced, where
    else:
        assert not _has(names, r"split_kernel") and not _has(names, r"bwd_unit_kernel"), where
        assert _has(names, rf"bwd_chunk_kernel<{m}, ") and _has(names, rf"bwd_merge_kernel<{m}>"), where
        G = max(d for _, d in shapes) // 4
        pow2 = G & (G - 1) == 0 and G <= 128
        hot = pow2 and any(rows <= 128 for rows, _ in shapes)  # the host-known hot rows: tables of <= 128 rows (the first 32 such)
        assert _has(names, r"bwd_hot_slice_kernel") == (hot or (pow2 and B * sum(f[1] for f in fields) >= 1024)), where
        assert _has(names, r"bwd_long_detect_kernel") == (pow2 and B * sum(f[1] for f in fields) >= 1024), where
        if hot:
            assert _has(names, rf"bwd_hot_apply_kernel<{m}>"), where
    return units


def run_case(dev, case, mode, algo, l2_scale=0.0):
    from handyrec_b200 import _lib

    k = K()
    douts = _douts(case)
    sums = [plan_grad_sums(case["shapes"], case["fields"], ids, dout) for ids, dout in zip(case["steps"], douts)]
    touched = _touched(case, mode, sums)
    tdev = [t.to(dev) for t in touched]
    hyper = dict(FTRL) if mode == "ftrl" else {}

    def one_run(profile):
        w, slots = _init(dev, case, mode)
        kw = {}
        if mode == "adam":
            kw = dict(adam_m=slots[0], adam_v=slots[1])
        elif mode == "adagrad":
            kw = dict(accum=slots[0])
        elif mode == "ftrl":
            kw = dict(accum=slots[0], linear=slots[1])
        plan = k.LookupPlan(w, case["fields"], **kw)
        grads = [torch.zeros_like(w[t]) if t in case["dense"] else None for t in range(len(w))]
        if case["dense"]:
            plan.set_dense_grads(grads)
        _lib.call("hrb_plan_set_bwd_algo", plan._h, _lib.BWD_UNITS if algo == "units" else _lib.BWD_SORT)

        def steps():
            for i, (ids, dout) in enumerate(zip(case["steps"], douts)):
                plan.backward_update(ids.to(dev), dout.to(dev), opt=mode, lr=LR[mode], l2_scale=l2_scale, step=ADAM_STEP0 + i, **hyper)

        names = _kernel_names(steps) if profile else None
        if not profile:
            steps()
        torch.cuda.synchronize()
        # untouched rows keep their bits: compare with a fresh initialisation (the hash is a pure function of seed and index)
        w0, s0 = _init(dev, case, mode)
        for t in range(len(w)):
            keep = torch.ones(w[t].shape[0], dtype=torch.bool, device=dev)
            keep[tdev[t]] = False
            for a, b in [(w[t], w0[t])] + [(s[t], z[t]) for s, z in zip(slots, s0)]:
                assert not bool(((a != b).any(1) & keep).any()), f"table {t}: an untouched row changed"
            if grads[t] is not None:
                assert not bool(((grads[t] != 0).any(1) & keep).any()), f"table {t}: a dense gradient row outside the touched rows"
        got = [(w[t][tdev[t]].cpu(), [s[t][tdev[t]].cpu() for s in slots], None if grads[t] is None else grads[t][tdev[t]].cpu())
               for t in range(len(w))]
        return got, names

    got, names = one_run(profile=True)
    got2, _ = one_run(profile=False)
    for t, (a, b) in enumerate(zip(got, got2)):  # deterministic, bit for bit
        assert torch.equal(a[0], b[0]) and all(torch.equal(x, y) for x, y in zip(a[1], b[1])), f"table {t}: not deterministic"
        assert (a[2] is None) or torch.equal(a[2], b[2]), f"table {t}: dense gradient not deterministic"
    units = _check_path(case, mode, algo, names)
    ref = _reference(case, mode, l2_scale, douts, sums, touched)
    tol = TOL[mode]
    for t, ((gw, gs, gg), (W, S, G, amb)) in enumerate(zip(got, ref)):
        what = f"table {t} {case['shapes'][t]} ({'units' if units else 'sort'} path, {mode})"
        if G is not None:
            close(gg, G, GRAD_TOL)
            continue
        ok = ~amb
        try:
            close(gw[ok], W[ok], tol)
            for a, b in zip(gs, S):
                close(a[ok], b[ok], tol)
        except AssertionError as e:
            raise AssertionError(f"{what}: {e}") from None
    return units


# ------------------------------------------------------------------------------------------------------------------------------
# backward matrix
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("D", [4, 8, 16, 32, 64, 128])
def test_bwd_unit_widths(dev, D, mode, algo):
    assert run_case(dev, base_case(D, 20000), mode, algo) == (algo == "units")


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("D", [12, 24, 96, 256, 1024])
def test_bwd_sort_only_widths(dev, D, mode):
    """G not a power of two (no hot or long passes), G = 64 (4 groups per CTA), G = 256 (one group per CTA): the unit path is not
    available, a UNITS preference falls back to the sorted path."""
    B = 20000 if D <= 128 else 4097
    assert run_case(dev, base_case(D, B), mode, "units") is False


@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("mode", MODES)
def test_bwd_l2_scale(dev, mode, algo):
    run_case(dev, base_case(16, 20000, seed=1), mode, algo, l2_scale=1e-2)


ROUTES = {
    "cap64": cap64_case,
    "zipf_2m": zipf_case,
    "list_4096": lambda D: unit_list_case(D, 4096),
    "list_4097": lambda D: unit_list_case(D, 4097),
    "row_4097": lambda D: unit_list_case(D, 5000, hot_row=5),
    "long_runs": long_runs_case,
    "tiny_33": tiny33_case,
}


# the unit-list boundaries are routes of the unit path; on the sorted path they would be one more uniform case
ROUTE_ALGOS = [(r, a) for r in ROUTES for a in ALGOS if a == "units" or not r.startswith(("list", "row"))]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("D", [4, 16, 128])
@pytest.mark.parametrize("route,algo", ROUTE_ALGOS)
def test_bwd_routes(dev, route, algo, D, mode):
    case = ROUTES[route](D)
    B = case["steps"][0].shape[0]
    if route.startswith(("list", "row")):  # the ids land where the case says: the first unit's list holds exactly n positions
        u = table_units(1 << 20, 1, B)
        want = {"list_4096": 4096, "list_4097": 4097, "row_4097": 5000}[route]
        assert all(unit_counts(u, ids[:, 0].numpy())[0] == want for ids in case["steps"])
    if route == "zipf_2m":
        u = table_units(2_000_000, 1, B)
        assert all(unit_counts(u, ids[:, 0].numpy())[0] > 4 * 4096 for ids in case["steps"])  # overflow, all helpers busy
    if route == "cap64":
        assert [x["slices"] for x in table_units(2, 10, B)] == [64, 64]
    assert run_case(dev, case, mode, algo) == (algo == "units")


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("which", ["bins_256", "bins_257", "cols_256", "cols_257"])
def test_bwd_units_sort_boundary(dev, which, mode):
    """Both sides of each limit of the unit path under a UNITS preference: 256 vs 257 units in one table, 256 vs 257 position
    columns.  The last one over the limit silently takes the sorted path (the profiler shows which)."""
    kind, n = which.split("_")
    case = bins_case(int(n)) if kind == "bins" else cols_case(int(n))
    assert run_case(dev, case, mode, "units") == (n == "256")


@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("mode", ["sgd", "adam"])
@pytest.mark.parametrize("B", [1, 15, 16, 17, 4095, 4096, 4097, 65537])
def test_bwd_batch_sizes(dev, B, mode, algo):
    run_case(dev, base_case(16, B, seed=2), mode, algo)


@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("mode", MODES)
def test_bwd_six_widths_in_one_plan(dev, mode, algo):
    assert run_case(dev, mixed_case(), mode, algo) == (algo == "units")


def test_bwd_autotune_matches_the_reference(dev):
    """backward_update(autotune=True): calls 3..6 alternate the two algorithms, then the faster is kept; 8 lazy Adam steps on
    different ids match the float64 reference whichever one the timing keeps."""
    k = K()
    D, B, n = 16, 20000, 8
    case = base_case(D, B, seed=3)
    case["steps"] = [base_case(D, B, seed=10 + i)["steps"][0] for i in range(n)]
    douts = _douts(case)
    sums = [plan_grad_sums(case["shapes"], case["fields"], ids, dout) for ids, dout in zip(case["steps"], douts)]
    touched = _touched(case, "adam", sums)
    w, slots = _init(dev, case, "adam")
    plan = k.LookupPlan(w, case["fields"], adam_m=slots[0], adam_v=slots[1])
    grads = [torch.zeros_like(w[t]) if t in case["dense"] else None for t in range(len(w))]
    plan.set_dense_grads(grads)
    for i, (ids, dout) in enumerate(zip(case["steps"], douts)):
        plan.backward_update(ids.to(dev), dout.to(dev), opt="adam", lr=LR["adam"], step=ADAM_STEP0 + i, autotune=True)
    torch.cuda.synchronize()
    assert plan.bwd_algo in ("units", "sort") and set(plan.bwd_algo_ms) == {"units", "sort"}
    ref = _reference(case, "adam", 0.0, douts, sums, touched)
    for t, (W, S, G, _) in enumerate(ref):
        idx = touched[t].to(dev)
        if G is not None:
            close(grads[t][idx], G, GRAD_TOL)
            continue
        close(w[t][idx], W, TOL["adam"])
        close(slots[0][t][idx], S[0], TOL["adam"])
        close(slots[1][t][idx], S[1], TOL["adam"])


# ------------------------------------------------------------------------------------------------------------------------------
# forward matrix
# ------------------------------------------------------------------------------------------------------------------------------
def _fwd_reference(tabs, fields, ids, out_cols):
    """float64 pooled output (B, out_cols) of the plan; max pooling follows sequence.py: padded positions offer W[0] - 1e9 in fp32."""
    ids = ids.long()
    B = ids.shape[0]
    out = torch.zeros(B, out_cols, dtype=torch.float64)
    for ti, L, pool, ids_col, out_col in fields:
        T = torch.from_numpy(tabs[ti]).double()
        rows, d = T.shape
        c = ids[:, ids_col: ids_col + L]
        valid = (c >= 0) & (c < rows) & ((c != 0) if pool != "none" else True)
        x = T[c.clamp(0, rows - 1)] * valid[..., None]
        if pool in ("none", "sum"):
            r = x.sum(1)
        elif pool == "mean":
            n = valid.sum(1, keepdim=True).double()
            r = torch.where(n > 0, x.sum(1) / n.clamp(min=1), torch.zeros_like(x[:, 0]))
        else:
            pad = torch.from_numpy((tabs[ti][0] - np.float32(1e9)).astype(np.float32)).double()
            x = torch.where(valid[..., None], x, pad.expand_as(x))
            r = x.max(1).values
        out[:, out_col: out_col + d] = r
    return out


def _fwd_tables(dev, shapes, seed=0):
    k = K()
    host = [oracle.hash_uniform_table(rows, d, 500 + seed + t) for t, (rows, d) in enumerate(shapes)]
    devt = [k.init_uniform(torch.empty(rows, d, device=dev), 500 + seed + t) for t, (rows, d) in enumerate(shapes)]
    return host, devt


def _fwd_check(dev, shapes, fields, ids, kernel, fm=False, inv=False, fm_sum=False, out_pad=0):
    k = K()
    host, devt = _fwd_tables(dev, shapes)
    plan = k.LookupPlan(devt, fields)
    B = ids.shape[0]
    oc = plan.out_cols
    buf = torch.full((B, oc + 2 * out_pad), float("nan"), device=dev)
    out = buf[:, out_pad: out_pad + oc] if out_pad else None
    D = shapes[0][1]
    w, w0 = rnd(D, 1, seed=D, scale=0.1), torch.tensor([0.2])
    res = {}

    def go():
        res.update(plan.forward(ids.to(dev), out=out, want_inv_count=inv, fm=(w.to(dev), w0.to(dev)) if fm else None, want_fm_sum=fm_sum))

    names = _kernel_names(go)
    assert _has(names, kernel), f"{kernel} did not run: {sorted(n for n in names if 'lookup' in n)}"
    want = _fwd_reference(host, fields, ids, oc)
    got = res["out"].cpu()
    if out_pad:
        assert bool(buf[:, :out_pad].isnan().all()) and bool(buf[:, out_pad + oc:].isnan().all())  # nothing outside `out` written
    for ti, L, pool, ids_col, out_col in fields:
        d = shapes[ti][1]
        g, r = got[:, out_col: out_col + d], want[:, out_col: out_col + d]
        if pool == "none":
            assert torch.equal(g, r.float()), f"field at column {out_col}: gather not bit-exact"
        else:  # an all-padding max-pooled row is fl(W[0] - 1e9) on both sides: exact; the rest within 1e-5
            big = r.abs() > 1e8
            assert torch.equal(g[big], r[big].float())
            close(g[~big], r[~big], 1e-5)
    if inv:
        n = torch.stack([((ids[:, f[3]: f[3] + f[1]] != 0) & (ids[:, f[3]: f[3] + f[1]] < shapes[f[0]][0])).sum(1) if f[2] == "mean"
                         else torch.full((B,), -1) for f in fields], 1).double()
        winv = torch.where(n > 0, 1.0 / n.clamp(min=1), torch.where(n == 0, torch.zeros_like(n), torch.ones_like(n)))
        close(res["inv_count"].cpu(), winv, 1e-6)
    if fm:
        x = want.reshape(B, len(fields), D)
        close(res["fm_out"].cpu(), oracle.fm(x, w.double(), w0.double())[:, 0], 1e-5)
        if fm_sum:
            close(res["fm_sum"].cpu(), x.sum(1), 1e-5)
    return plan


def _plain_ids(B, vocabs, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.stack([torch.randint(0, v, (B,), generator=g, dtype=torch.int32) for v in vocabs], 1)


@pytest.mark.parametrize("fm", [False, True])
@pytest.mark.parametrize("D,F,kernel", [(8, 8, "lookup_tile_kernel<2, "), (16, 26, "lookup_tile_kernel<4, "), (32, 8, "lookup_tile_kernel<8, "),
                                        (64, 8, "lookup_tile_kernel<16, "), (32, 20, "lookup_tile_kernel<8, "),
                                        (32, 30, "lookup_rows_kernel<8, true, "), (64, 26, "lookup_rows_kernel<16, true, ")])
def test_fwd_plain_groups_tile_and_rows(dev, D, F, kernel, fm):
    """Plain contiguous groups: the 32-sample tile fits 100 KB of shared memory up to 20 fields at D = 32 (not 30) and up to 8 at
    D = 64 (not the Criteo shape's 26), beyond which the rows kernel takes them."""
    kernel += ("true" if fm else "false") + ("" if kernel.startswith("lookup_tile") else ">")
    vocabs = [7 + 1000 * f for f in range(F)]
    _fwd_check(dev, [(v, D) for v in vocabs], [(f, 1, "none", f, f * D) for f in range(F)], _plain_ids(1000, vocabs, D + F), kernel,
               fm=fm, fm_sum=fm)


@pytest.mark.parametrize("D", [4, 128])
def test_fwd_fm_rows_kernel_at_the_edge_widths(dev, D):
    """FM at D = 4 and 128 (no tile kernel there) through the rows kernel; the same groups without FM through the items kernel."""
    vocabs = [10, 1000, 100000, 5]
    shapes, fields = [(v, D) for v in vocabs], [(f, 1, "none", f, f * D) for f in range(4)]
    ids = _plain_ids(4099, vocabs, D)
    _fwd_check(dev, shapes, fields, ids, rf"lookup_rows_kernel<{D // 4}, true, true>", fm=True, fm_sum=True)
    _fwd_check(dev, shapes, fields, ids, r"lookup_items_kernel")


def _pooled_group(D, pool, B=1031, seed=0, empty=True):
    shapes = [(50, D), (3000, D), (20, D)]
    fields = [(0, 1, "none", 0, 0), (1, 6, pool, 1, D), (1, 1, "none", 7, 2 * D), (2, 3, pool, 8, 3 * D)]
    g = torch.Generator().manual_seed(seed + D)
    ids = torch.cat([torch.randint(0, 50, (B, 1), generator=g, dtype=torch.int32), _hist(g, B, 6, 3000, empty),
                     torch.randint(0, 3000, (B, 1), generator=g, dtype=torch.int32), _hist(g, B, 3, 20, empty)], 1)
    if empty:
        ids[::4, 8:11] = 0  # all-padding rows
    return shapes, fields, ids


@pytest.mark.parametrize("pool", ["mean", "sum", "max"])
@pytest.mark.parametrize("D", [4, 8, 16, 32, 64, 128])
def test_fwd_fm_with_pooled_fields(dev, D, pool):
    # an all-padding max-pooled row is ~-1e9 (sequence.py), which leaves nothing of the FM interaction to compare: none here
    shapes, fields, ids = _pooled_group(D, pool, empty=pool != "max")
    _fwd_check(dev, shapes, fields, ids, rf"lookup_rows_kernel<{D // 4}, false, true>", fm=True, inv=True, fm_sum=True)


@pytest.mark.parametrize("D", [4, 16, 128])
def test_fwd_fm_plain_with_inv_count(dev, D):
    vocabs = [10, 1000, 77]
    _fwd_check(dev, [(v, D) for v in vocabs], [(f, 1, "none", f, f * D) for f in range(3)], _plain_ids(513, vocabs, 1),
               rf"lookup_rows_kernel<{D // 4}, true, true>", fm=True, inv=True)


@pytest.mark.parametrize("pool", ["mean", "sum", "max"])
@pytest.mark.parametrize("D", [4, 8, 12, 16, 32, 64, 128, 256])
def test_fwd_items_pooled(dev, D, pool):
    """Pooled groups without FM (max pooling with all-padding rows included), with inv_count, written into a column slice of a wider
    buffer (nothing outside it changes)."""
    shapes, fields, ids = _pooled_group(D, pool, seed=1)
    _fwd_check(dev, shapes, fields, ids, r"lookup_items_kernel", inv=True, out_pad=4)


@pytest.mark.parametrize("D", [4, 12, 128, 256])
def test_fwd_items_plain(dev, D):
    vocabs = [3, 999, 100003]
    _fwd_check(dev, [(v, D) for v in vocabs], [(f, 1, "none", f, f * D) for f in range(3)], _plain_ids(4097, vocabs, D),
               r"lookup_items_kernel")


def test_fwd_items_mixed_widths(dev):
    shapes = [(100, 4), (2000, 32), (30, 128), (500, 12)]
    fields = [(0, 1, "none", 0, 0), (1, 5, "mean", 1, 4), (2, 1, "none", 6, 36), (3, 2, "max", 7, 164), (1, 1, "none", 9, 176)]
    g = torch.Generator().manual_seed(3)
    ids = torch.cat([torch.randint(0, 100, (777, 1), generator=g, dtype=torch.int32), _hist(g, 777, 5, 2000),
                     torch.randint(0, 30, (777, 1), generator=g, dtype=torch.int32), _hist(g, 777, 2, 500),
                     torch.randint(0, 2000, (777, 1), generator=g, dtype=torch.int32)], 1)
    _fwd_check(dev, shapes, fields, ids, r"lookup_items_kernel", inv=True, out_pad=8)


@pytest.mark.parametrize("kind", ["tile", "rows", "items"])
@pytest.mark.parametrize("where", ["negative", "past_end"])
def test_fwd_check_ids_reports_from_every_kernel(dev, kind, where):
    k = K()
    D = 16 if kind != "items" else 128
    vocabs = [50, 60, 70]
    host, devt = _fwd_tables(dev, [(v, D) for v in vocabs])
    plan = k.LookupPlan(devt, [(f, 1, "none", f, f * D) for f in range(3)])
    ids = _plain_ids(300, vocabs, 5)
    plan.forward(ids.to(dev), check_ids=True)  # in range: no error
    ids[123, 1] = -2 if where == "negative" else 60
    fm = (rnd(D, 1).to(dev), torch.zeros(1, device=dev)) if kind == "rows" else None
    names = set()
    with pytest.raises(IndexError, match="sample index 123"):
        names = _kernel_names(lambda: plan.forward(ids.to(dev), check_ids=True, fm=fm, want_inv_count=kind == "rows"))
    names = _kernel_names(lambda: plan.forward(ids.to(dev), check_ids=False, fm=fm, want_inv_count=kind == "rows"))
    assert _has(names, {"tile": "lookup_tile_kernel", "rows": "lookup_rows_kernel", "items": "lookup_items_kernel"}[kind])
