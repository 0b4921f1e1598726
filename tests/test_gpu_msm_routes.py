"""Every entry point that runs one MSM over the resident generators, on the same seeded scalars, against each other and
against the oracle.

halo_msm_gens, _resident, the submit / collect pair over host and device scalars, halo_msm_multi without bases and
halo_msm_gens_many with one output each choose FIXED or variable base, build the plan and finish the window partials through
the MSM engine.  For every size, with the quad and with the one-lane bucket reduction (the reduce_quad knob, which is part of
the plan that the host finish reads), each entry point must report the same route through halo_test_msm_route and return the
oracle's point.  A segmented halo_msm_gens_many of eight outputs runs under the one-lane reduction as well."""
import numpy as np
import pytest

gpu = pytest.mark.gpu

N_GENS = (1 << 17) + 4096
OFF = 777
# 4000: within halo_msm_multi's 4096 points; 5000: variable base beyond it; 2^17 + 1234 with tables: FIXED base
SIZES = (4000, 5000, (1 << 17) + 1234)
ROUTE_KEYS = ("c", "fixed", "P", "acc", "reduce_quad")


@pytest.fixture(scope="module")
def rt(ctx, oracle):
    """The session context with N_GENS derived generators, the oracle holding the same parameters, and per size the scalars
    with the expected points at OFF and at 0 (halo_msm_gens_many has no offset)."""
    import torch

    O = oracle
    ctx.derive_generators(N_GENS)
    S, H = ctx.get_SH()
    O.set_params(S, H, ctx.get_generators(0, N_GENS))
    cases = {}
    for n in SIZES:
        sc = np.ascontiguousarray(O.random_scalars(n, 40 + n), dtype=np.uint64)
        cases[n] = (sc, O.msm_derived_by_dlog(OFF, sc, threads=8), O.msm_derived_by_dlog(0, sc, threads=8))
    yield dict(ctx=ctx, O=O, cases=cases, torch=torch)
    ctx.set_tuning("reduce_quad", 1)
    ctx.derive_generators(1 << 16)
    S, H = ctx.get_SH()
    O.set_params(S, H, ctx.get_generators(0, 1 << 16))


def _entry_points(rt, n):
    """name -> (function returning the point, whether it runs at OFF)"""
    ctx, torch = rt["ctx"], rt["torch"]
    sc = rt["cases"][n][0]
    d = torch.from_numpy(sc.view(np.int64).copy()).cuda()
    torch.cuda.synchronize()
    eps = {
        "msm_gens": (lambda: ctx.msm_gens(sc, off=OFF), True),
        "msm_gens_resident": (lambda: ctx.msm_gens_resident(d.data_ptr(), n, off=OFF), True),
        "submit_collect": (lambda: ctx.msm_gens_collect(ctx.msm_gens_submit(sc, off=OFF)), True),
        "submit_resident_collect": (lambda: ctx.msm_gens_collect(ctx.msm_gens_submit_resident(d.data_ptr(), n, off=OFF)), True),
        "msm_gens_many": (lambda: ctx.msm_gens_many([sc])[0], False),
    }
    if n <= 4096:
        eps["msm_multi"] = (lambda: ctx.msm_multi([(None, sc, None, OFF)])[0], True)
    return eps, d


@gpu
@pytest.mark.parametrize("n", SIZES)
def test_generator_msm_entry_points_agree(rt, n):
    ctx, O = rt["ctx"], rt["O"]
    _, exp_off, exp_0 = rt["cases"][n]
    if n >= 1 << 17:
        ctx.precompute_generators(0)
    try:
        for quad in (1, 0):
            ctx.set_tuning("reduce_quad", quad)
            eps, _keep = _entry_points(rt, n)
            routes = {}
            for name, (run, at_off) in eps.items():
                p = run()
                r = ctx.test_msm_route(0)
                routes[name] = {k: r[k] for k in ROUTE_KEYS}
                assert O.pt_eq(p, exp_off if at_off else exp_0), (name, n, quad, r)
            first = routes["msm_gens"]
            assert (first["fixed"], first["reduce_quad"]) == (int(n >= 1 << 17), quad), first
            bad = {name: r for name, r in routes.items() if r != first}
            assert not bad, (n, quad, first, bad)
    finally:
        ctx.set_tuning("reduce_quad", 1)


@gpu
def test_segmented_many_one_lane_reduction(rt):
    """Eight outputs of 2049 .. 4096 points: one segmented MSM (the narrowed window 8) with the one-lane bucket reduction."""
    ctx, O = rt["ctx"], rt["O"]
    lens = [4096, 2049, 3000, 4095, 2500, 3333, 4000, 2222]
    vecs = [np.ascontiguousarray(O.random_scalars(m, 90 + j), dtype=np.uint64) for j, m in enumerate(lens)]
    try:
        ctx.set_tuning("reduce_quad", 0)
        got = ctx.msm_gens_many(vecs)
        r = ctx.test_msm_route(0)
        assert (r["c"], r["fixed"], r["reduce_quad"]) == (8, 0, 0), r
        for j, v in enumerate(vecs):
            assert O.pt_eq(got[j], O.msm_derived_by_dlog(0, v, threads=8)), j
    finally:
        ctx.set_tuning("reduce_quad", 1)
