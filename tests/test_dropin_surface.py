"""The drop-in contract of SURVEY.md section 8(b): every method / buffer name the reference's callers use exists on the mirrors
with a compatible signature (the reference's positional parameters are stored in tests/golden/dropin_signatures.json by
tests/golden/make_golden.py:gen_dropin), and phc_b200.dropin rebinds the classes in the reference's modules (both import
spellings run_hydra.py uses).  The rebinding is checked on stand-in modules with the reference's module names, package layout
and class hierarchy, written to a temporary directory.  CPU only: nothing is instantiated."""
import importlib
import inspect
import json
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

TASK_METHODS = ["step", "reset", "_compute_observations", "_compute_task_obs", "_compute_reward", "_compute_reset", "_compute_humanoid_obs",
                "_compute_amp_observations", "fetch_amp_obs_demo", "get_obs_size", "get_task_obs_size", "get_self_obs_size", "get_num_amp_obs",
                "get_action_size", "resample_motions", "get_task_obs_size_detail", "get_running_mean_size", "post_physics_step"]
AGENT_METHODS = ["train", "train_epoch", "play_steps", "calc_gradients", "discount_values", "_calc_advs", "_preproc_obs", "_disc_loss",
                 "_calc_amp_rewards", "_combine_rewards", "get_stats_weights", "set_stats_weights", "get_full_state_weights",
                 "set_full_state_weights", "restore", "save", "env_reset", "env_step", "get_action_values", "_eval_critic", "prepare_dataset",
                 "pre_epoch", "_update_amp_demos", "_init_amp_demo_buf", "_store_replay_amp_obs", "set_eval", "set_train"]
# the reference defines these itself (not only through rl_games / Isaac Gym bases): positional parameters must line up
SIGNATURE_METHODS = {
    "HumanoidIm": ["__init__", "_compute_task_obs", "_compute_reward", "_compute_reset", "resample_motions", "get_task_obs_size",
                   "get_task_obs_size_detail", "post_physics_step"],
    "AMPAgent": ["__init__", "play_steps", "calc_gradients", "train_epoch", "_calc_amp_rewards", "_combine_rewards", "_disc_loss",
                 "get_stats_weights", "set_stats_weights", "_preproc_obs"],
}

# The reference's modules as the drop-in sees them: phc/ is a package (parse_task.py imports phc.env.tasks.*) and also
# sys.path[0] of run_hydra.py (short names learning.*, env.tasks.*); the subclasses import their base module by its long name.
STAND_INS = {
    "phc/__init__.py": "",
    "phc/env/__init__.py": "",
    "phc/env/tasks/__init__.py": "",
    "phc/env/tasks/humanoid_im.py": "class HumanoidIm:\n    pass\n",
    "phc/env/tasks/humanoid_im_mcp.py": "import phc.env.tasks.humanoid_im as humanoid_im\n\n\n"
                                        "class HumanoidImMCP(humanoid_im.HumanoidIm):\n    pass\n",
    "phc/learning/__init__.py": "",
    "phc/learning/amp_agent.py": "class AMPAgent:\n    pass\n",
    "phc/learning/im_amp.py": "import phc.learning.amp_agent as amp_agent\n\n\nclass IMAmpAgent(amp_agent.AMPAgent):\n    pass\n",
}
_TOP_LEVEL = ("phc", "env", "learning")


def _write_stand_ins(root):
    for rel, src in STAND_INS.items():
        p = root / rel
        p.parent.mkdir(parents=True, exist_ok=True)
        p.write_text(src)
    return str(root), str(root / "phc")


@pytest.fixture
def stand_in_modules(tmp_path, monkeypatch):
    """Imports the stand-ins under both spellings; afterwards drops them from sys.modules and restores the backend factory that
    dropin.install() registers."""
    from phc_b200.env import backends
    pkg_parent, script_dir = _write_stand_ins(tmp_path)
    monkeypatch.syspath_prepend(script_dir)
    monkeypatch.syspath_prepend(pkg_parent)
    importlib.invalidate_caches()
    factory = backends._FACTORY
    try:
        yield (importlib.import_module("phc.env.tasks.humanoid_im"), importlib.import_module("phc.learning.amp_agent"),
               importlib.import_module("learning.amp_agent"), importlib.import_module("phc.env.tasks.humanoid_im_mcp"))
    finally:
        backends.register_backend_factory(factory)
        for name in [m for m in sys.modules if m.split(".")[0] in _TOP_LEVEL]:
            del sys.modules[name]


def test_mirror_surface_is_complete():
    from phc_b200.env.humanoid_im import HumanoidIm
    from phc_b200.env.humanoid_im_mcp import HumanoidImMCP
    from phc_b200.learning.amp_agent import AMPAgent
    assert [m for m in TASK_METHODS if not callable(getattr(HumanoidIm, m, None))] == []
    assert [m for m in AGENT_METHODS if not callable(getattr(AMPAgent, m, None))] == []
    assert issubclass(HumanoidImMCP, HumanoidIm)
    assert list(inspect.signature(HumanoidIm.__init__).parameters)[1:] == ["cfg", "sim_params", "physics_engine", "device_type", "device_id", "headless"]
    assert list(inspect.signature(AMPAgent.__init__).parameters)[1:] == ["base_name", "config"]


def test_signatures_match_the_reference():
    from phc_b200.env.humanoid_im import HumanoidIm
    from phc_b200.learning.amp_agent import AMPAgent
    with open(os.path.join(HERE, "golden", "dropin_signatures.json")) as f:
        ref = json.load(f)
    for cname, ours in (("HumanoidIm", HumanoidIm), ("AMPAgent", AMPAgent)):
        assert sorted(ref[cname]) == sorted(SIGNATURE_METHODS[cname]), f"reference signatures of {cname} incomplete"
        for n in SIGNATURE_METHODS[cname]:
            rp = ref[cname][n]                           # [[name, required], ...] of the positional parameters
            op = [p for p in inspect.signature(getattr(ours, n)).parameters.values()]
            r_req = [name for name, required in rp if required]
            o_names = [p.name for p in op if p.kind in (p.POSITIONAL_ONLY, p.POSITIONAL_OR_KEYWORD)]
            assert o_names[:len(r_req)] == r_req or len(o_names) >= len(r_req), f"{cname}.{n}: reference {r_req} vs ours {o_names}"
            o_req = [p.name for p in op if p.default is p.empty and p.kind in (p.POSITIONAL_ONLY, p.POSITIONAL_OR_KEYWORD)]
            assert len(o_req) <= len(rp), f"{cname}.{n}: ours requires {o_req}, the reference passes at most {[name for name, _ in rp]}"


def test_dropin_rebinds_both_import_spellings(stand_in_modules):
    from phc_b200 import dropin
    from phc_b200.env.humanoid_im import HumanoidIm
    from phc_b200.env.humanoid_im_mcp import HumanoidImMCP
    from phc_b200.learning.amp_agent import AMPAgent
    ref_env, ref_agent, ref_agent_short, ref_mcp = stand_in_modules
    assert dropin.install() >= 4
    assert ref_env.HumanoidIm is HumanoidIm and ref_mcp.HumanoidImMCP is HumanoidImMCP
    assert ref_agent.AMPAgent is AMPAgent and ref_agent_short.AMPAgent is AMPAgent
    assert eval("HumanoidIm", vars(ref_env)) is HumanoidIm          # what parse_task.py:60 does


def test_install_on_import_rebinds_when_the_reference_modules_load_later(tmp_path):
    """The sitecustomize route: the hook is registered BEFORE the reference modules are imported (as when `python
    phc/run_hydra.py` starts) and rebinds the classes right after each module body ran -- checked in a fresh interpreter."""
    pkg_parent, script_dir = _write_stand_ins(tmp_path)
    code = r'''
import sys
sys.path.insert(0, %r); sys.path.insert(0, %r); sys.path.insert(0, %r)
import phc_b200.dropin as d
d.install_on_import()                                     # what sitecustomize.py does
assert not any(m in sys.modules for m in ("phc.env.tasks.humanoid_im", "learning.amp_agent"))
import phc.env.tasks.humanoid_im as ref_env              # parse_task.py:29-38 spelling
import learning.amp_agent as ref_agent                   # run_hydra.py:57-64 spelling
import learning.im_amp as im_amp                          # class IMAmpAgent(amp_agent.AMPAgent)
from phc_b200.env.humanoid_im import HumanoidIm
from phc_b200.learning.amp_agent import AMPAgent
assert ref_env.HumanoidIm is HumanoidIm and eval("HumanoidIm", vars(ref_env)) is HumanoidIm
assert ref_agent.AMPAgent is AMPAgent
assert AMPAgent in im_amp.IMAmpAgent.__mro__, im_amp.IMAmpAgent.__mro__
print("OK")
''' % (script_dir, pkg_parent, ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
