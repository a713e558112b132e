"""Helper of tests/test_reference_driver_cpu.py (own process): the reference's UNCHANGED ``train_off_policy.py`` and THIS
package's restatement of it (``agilerl_b200/training/train_off_policy.py`` — the driver the GPU box runs, where the reference
does not exist) train the same seeded population on the same environment with the same stand-in kernels.  Stand-in outputs
are deterministic functions of their inputs, so a faithful restatement yields IDENTICAL fitnesses, step counts, mutations,
indices, call counts, exploration schedules and replay contents.

The reference's run is stored in tests/golden/driver_equivalence.json; by default only our driver runs and is compared with
it.  ``--record`` (tests/golden/make_golden.py, where the reference exists) runs both drivers, checks them against each other
and prints the reference's run."""
import json
import math
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODE = sys.argv[1] if len(sys.argv) > 1 else "DQN"
RECORD = "--record" in sys.argv
helper = {"RAINBOW": "_reference_driver_rainbow_standin.py", "MADDPG": "_reference_ma_driver_standin.py"}.get(MODE, "_reference_driver_standin.py")
src = open(os.path.join(ROOT, "tests", helper)).read()
cut = {"RAINBOW": 'pop = create_population("Rainbow DQN"', "MADDPG": 'pop = create_population("MADDPG"'}.get(MODE, "import glob  # noqa: E402")
sys.argv = [sys.argv[0], MODE] + ([] if RECORD else ["--without-reference"])
exec(compile(src[:src.index(cut)].replace("os.path.abspath(__file__)", repr(os.path.join(ROOT, "tests", helper))), helper, "exec"))
from agilerl_b200.training import train_multi_agent_off_policy as ours_ma_driver  # noqa: E402
from agilerl_b200.training import train_off_policy as ours_driver  # noqa: E402


def run(driver):
    torch.manual_seed(0); np.random.seed(0); random.seed(0)          # noqa: F821 (names come from the helper's setup)
    for k in calls:                                                   # noqa: F821
        calls[k] = 0                                                  # noqa: F821
    if MODE == "MADDPG":
        pop = create_population("MADDPG", obs_spaces, act_spaces, None, INIT_HP, population_size=3, num_envs=E)   # noqa: F821
        memory = C.MultiAgentReplayBuffer(200, ["obs", "action", "reward", "next_obs", "done"], IDS, device="cuda")  # noqa: F821
        pop, fits = driver(ParallelVecEnv(), "synthetic", "MADDPG", pop, memory, INIT_HP=INIT_HP, MUT_P={}, max_steps=96,  # noqa: F821
                           evo_steps=32, eval_steps=12, eval_loop=1, tournament=H.TournamentSelection(2, True, 3, 1),  # noqa: F821
                           mutation=H.Mutations(0.5, 0, 0.2, 0.5, 0, 0, rand_seed=0, device="cuda"), wb=False, verbose=False)  # noqa: F821
        return dict(fits=[[float(x) for x in f] for f in fits], steps=[int(a.steps[-1]) for a in pop], muts=[str(a.mut) for a in pop],
                    calls=dict(calls), idx=[a.index for a in pop], scores=[[float(x) for x in a.scores] for a in pop],  # noqa: F821
                    replay=[float(torch.nan_to_num(r.double(), nan=-3.0).sum()) for r in memory._rings], mem=len(memory),  # noqa: F821
                    counter=memory.counter, noise=[float(sum(v.abs().sum() for v in a.current_noise.values())) for a in pop])
    if MODE == "RAINBOW":
        pop = create_population("Rainbow DQN", obs_space, act_space, dict(NET), INIT_HP, population_size=2)       # noqa: F821
        memory, nm = C.PrioritizedReplayBuffer(256, 0.6, device="cuda"), C.MultiStepReplayBuffer(256, 3, 0.99, device="cuda")  # noqa: F821
        kw = dict(max_steps=80, evo_steps=40, n_step=True, per=True, n_step_memory=nm, tournament=H.TournamentSelection(2, True, 2, 1),  # noqa: F821
                  mutation=H.Mutations(0.6, 0, 0.2, 0.4, 0, 0, rand_seed=0, device="cuda"))                       # noqa: F821
        name = "Rainbow DQN"
    else:
        pop = create_population(ALGO, obs_space, act_space, None, INIT_HP, population_size=4, num_envs=2)         # noqa: F821
        memory, nm = C.ReplayBuffer(512, device="cuda"), None                                                     # noqa: F821
        kw = dict(max_steps=120, evo_steps=40, tournament=H.TournamentSelection(2, True, 4, 1),                  # noqa: F821
                  mutation=H.Mutations(0.5, 0, 0.2, 0.25, 0, 0.25, rand_seed=0, device="cuda"))                   # noqa: F821
        name = ALGO                                                                                               # noqa: F821
    pop, fits = driver(VecEnv(), "synthetic", name, pop, memory, INIT_HP=INIT_HP, MUT_P={}, eval_steps=10, eval_loop=1, wb=False,  # noqa: F821
                       verbose=False, **kw)
    out = dict(fits=[[float(x) for x in f] for f in fits], steps=[int(a.steps[-1]) for a in pop], muts=[str(a.mut) for a in pop],
               calls=dict(calls), idx=[a.index for a in pop], scores=[[float(x) for x in a.scores] for a in pop],          # noqa: F821
               replay={str(k): t.double().sum().item() for k, t in memory._fields.items()}, mem=len(memory))
    if MODE == "RAINBOW":
        out.update(beta=[a.beta for a in pop], tree_sum=float(_f64(memory.sum_tree.data_ptr, 2)[1]), max_priority=memory.max_priority,  # noqa: F821
                   nstep={str(k): t.double().sum().item() for k, t in nm._fields.items()})
    return out


def same(x, y):
    """Equal, floats to 1e-12 relative: the stored run comes from another process, maybe on another CPU, where a float sum over
    a tensor may round its last bit differently."""
    if isinstance(x, float) or isinstance(y, float):
        return math.isclose(x, y, rel_tol=1e-12, abs_tol=1e-300)
    if isinstance(x, dict):
        return isinstance(y, dict) and x.keys() == y.keys() and all(same(x[k], y[k]) for k in x)
    if isinstance(x, list):
        return isinstance(y, list) and len(x) == len(y) and all(same(u, v) for u, v in zip(x, y))
    return x == y


if RECORD:
    a = run(T.train_multi_agent_off_policy if MODE == "MADDPG" else T.train_off_policy)  # noqa: F821
    print("REFERENCE " + json.dumps(a))
else:
    with open(os.path.join(ROOT, "tests", "golden", "driver_equivalence.json")) as f:
        a = json.load(f)[MODE]
b = json.loads(json.dumps(run(ours_ma_driver if MODE == "MADDPG" else ours_driver)))
print("RESULT " + json.dumps({"equal": same(a, b), "diff": [k for k in a if not same(a[k], b.get(k))],
                              "learn_calls": a["calls"].get("learn", a["calls"].get("loss")), "generations": len(a["fits"])}))
