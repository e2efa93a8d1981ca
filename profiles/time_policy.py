"""Where the policy-in-the-loop step goes (BASELINE configs[3]): python profiles/time_policy.py [envs]"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import marl_mass_b200 as mm
from bench import WORKLOADS
from marl_mass_b200.rollout import BatchedMAPPORollout

E = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
cfg = dict(mm.DEFAULT_CONFIG, **WORKLOADS["mass_td3_srew"]["cfg"])
env = mm.MergeEnvBatched(E, cfg)
env.reset(seed=1)
pol = BatchedMAPPORollout(env, roll_out_n_steps=1)
v = env.buffers()


def timed(fn, n=20):
    for _ in range(3):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); a.record()
    for _ in range(n):
        fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / n


acts, _ = pol._act(v["obs"], v["n_agents"])
obs = v["obs"]
with torch.no_grad():
    logp = pol.actor(obs.view(-1, mm.NS))
    print("actor forward      %.3f ms" % timed(lambda: pol.actor(obs.view(-1, mm.NS))))
    print("exp + multinomial  %.3f ms" % timed(lambda: torch.multinomial(logp.exp(), 1)))
print("act_torch (all)    %.3f ms" % timed(lambda: pol.act_torch(v["obs"], v["n_agents"])))
print("env.step           %.3f ms" % timed(lambda: env.step(acts, auto_reset=True)))
print("act + step         %.3f ms" % timed(lambda: env.step(pol._act(v["obs"], v["n_agents"])[0], auto_reset=True)))
print("act_fused          %.3f ms" % timed(lambda: pol.act_fused(v["obs"], v["n_agents"])))
print("act_fused + step   %.3f ms" % timed(lambda: env.step(pol.act_fused(v["obs"], v["n_agents"])[0], auto_reset=True)))
lp = mm.rollout.actor_sample(pol.actor, obs, v["n_agents"], seed=1, step=1, want_logp=True)[1]
with torch.no_grad():
    logp = pol.actor(obs.view(-1, mm.NS))          # the env has stepped since the first evaluation: same rows again
print("max |logp_fused - logp_torch| = %.3e" % float((lp.view(-1, 5) - logp).abs().max()))
# the two actor kernels and the MAPPO_GI shared network on the same rows
from marl_mass_b200 import rollout
for name in ("tcgen05", "mma"):
    rollout.set_actor_impl(name)
    print("actor_sample %-13s %.4f ms" % (name, timed(lambda: rollout.actor_sample(pol.actor, obs, v["n_agents"], seed=1, step=1), n=50)))
rollout.set_actor_impl("tcgen05")
gi = rollout.ActorCriticNetwork().cuda()
with torch.no_grad():
    print("GI torch forward+draw      %.4f ms" % timed(lambda: torch.multinomial(gi(obs.view(-1, mm.NS)).exp(), 1)))
print("GI policy_sample (h1=160)  %.4f ms" % timed(lambda: rollout.policy_sample(gi, obs, v["n_agents"], seed=1, step=1), n=50))
print("GI policy_sample + value   %.4f ms" % timed(lambda: rollout.policy_sample(gi, obs, v["n_agents"], seed=1, step=1, want_value=True), n=50))
