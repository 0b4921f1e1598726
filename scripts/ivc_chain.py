"""BASELINE config 4: ASDL IVC chain -- k accumulation steps (random_instance + prover, benches/acc.rs:76-98) followed
by the fast path (k verifiers + one decider, benches/acc.rs:64-74) at n = 2^lg.  Times each phase on the GPU path, then
(outside the timed regions) hands the chain to the CPU oracle: acc_verifier on three spot steps (first, middle, last) and
acc_decider on the final accumulator.  `all_accept` is the conjunction of the GPU path's own k verifiers + decider (they
raise on a rejection) and of the oracle's decisions."""
import json, sys, time
import numpy as np
sys.path.insert(0, ".")
import halo_accumulation_b200 as H
from halo_accumulation_b200 import acc, group, pcdl

lg = int(sys.argv[1]) if len(sys.argv) > 1 else 20
k = int(sys.argv[2]) if len(sys.argv) > 2 else 64
n, d = 1 << lg, (1 << lg) - 1
ctx = H.Context(0, n)
t0 = time.perf_counter(); ctx.derive_generators(n); ctx.precompute_generators(0); setup_s = time.perf_counter() - t0
rng = np.random.Generator(np.random.PCG64(3))
def rs(m):
    a = rng.integers(0, 1 << 64, size=(m, 4), dtype=np.uint64); a[:, 3] &= np.uint64((1 << 62) - 1); return a

def draw_instance():
    """The random draws of random_instance (benches/acc.rs:15-29), made before the clock starts: numpy's generator and the
    pageable arrays it returns are harness, not the path being measured."""
    dp = int(rng.integers(d // 2, d))            # benches/acc.rs:16
    return dp, rs(dp + 1), rs(1)[0], rs(1)[0], rs(1)[0], rs(dp)

def random_instance(draws):
    dp, p, w, z, wb, q = draws
    Cm = pcdl.commit(ctx, p, d, w)
    v = group.scalar_dot(ctx, p, group.construct_powers(ctx, z, dp + 1))
    pi = pcdl.open(ctx, p, Cm, d, z, w, q, wb)
    return acc.new_instance(Cm, d, z, v, pi)

t_inst = t_prov = t_ver = 0.0
inst_ms, prov_ms = [], []
a, qss, accs = None, [], []
for s in range(k):
    draws = draw_instance()
    h0, w, q, wb = rs(2), rs(1)[0], rs(n - 1), rs(1)[0]
    t = time.perf_counter(); q_new = random_instance(draws); t_inst += time.perf_counter() - t; inst_ms.append((time.perf_counter() - t) * 1e3)
    qs = [acc.to_instance(a), q_new] if a is not None else [q_new]
    t = time.perf_counter(); a = acc.prover(ctx, d, qs, h0, w, q, wb); t_prov += time.perf_counter() - t; prov_ms.append((time.perf_counter() - t) * 1e3)
    qss.append(qs); accs.append(a)
t = time.perf_counter()
for qs, ac in zip(qss, accs):
    acc.verifier(ctx, d, qs, ac)
t_ver = time.perf_counter() - t
t = time.perf_counter(); acc.decider(ctx, accs[-1]); t_dec = time.perf_counter() - t
# the same fast path with ONE batch verifier over the k steps (rho drawn after the steps are fixed)
rho = rs(1)[0]
t = time.perf_counter(); acc.verifier_batch(ctx, d, list(zip(qss, accs)), rho); acc.decider(ctx, accs[-1]); t_fast_batch = time.perf_counter() - t
# and with ONE fused call: the steps verified and the last accumulator decided together (DESIGN.md K5d)
t = time.perf_counter(); acc.verify_decide_batch(ctx, d, list(zip(qss, accs)), [accs[-1]], rho); t_fast_fused = time.perf_counter() - t
# ---- the oracle's view of the same chain (checker only, untimed) ----
from oracle import oracle as O
S, Hh = ctx.get_SH()
O.set_params(S, Hh, ctx.get_generators(0, n))
T = max(1, O.lib().orc_num_threads())
as_o = lambda x, cls: cls.from_buffer_copy(bytes(x))
spots = sorted({0, k // 2, k - 1})
oracle_verifier = {s: O.acc_verifier(d, [as_o(q, O.Instance) for q in qss[s]], as_o(accs[s], O.Accumulator)) for s in spots}
t = time.perf_counter(); oracle_decider = O.acc_decider(as_o(accs[-1], O.Accumulator), threads=T); t_odec = time.perf_counter() - t
all_accept = all(rc == 0 for rc in oracle_verifier.values()) and oracle_decider == 0
print(json.dumps({"config": f"ivc_chain_2^{lg}_k{k}", "setup_s": setup_s, "random_instance_ms": t_inst / k * 1e3, "prover_ms": t_prov / k * 1e3,
                  "random_instance_ms_median": float(np.median(inst_ms)), "prover_ms_median": float(np.median(prov_ms)),
                  "random_instance_ms_first3": inst_ms[:3], "verifier_ms": t_ver / k * 1e3, "decider_ms": t_dec * 1e3, "fast_path_total_s": t_ver + t_dec,
                  "fast_path_batch_s": t_fast_batch, "fast_path_fused_s": t_fast_fused,
                  "chain_total_s": t_inst + t_prov, "kernel_launches": ctx.kernel_launches(), "all_accept": all_accept,
                  "oracle": {"acc_verifier_rc_at_steps": {str(s): rc for s, rc in oracle_verifier.items()}, "acc_decider_rc": oracle_decider,
                             "acc_decider_cpu_ms": t_odec * 1e3, "threads": T}}))
assert all_accept, "the oracle rejects the GPU chain"
