"""Reference-facing façades: `RailEnv` and `TreeObsForRailEnv` with the API surface that
solution/eval_env.py, solution/demo.py and solution/plfActor.py of the reference use
(SURVEY.md §8b), backed by a `BatchedRailEnv` on the GPU.

  RailEnv.reset() -> (obs, info)                     rail_env.py:260-357
  RailEnv.step(action_dict) -> (obs, rewards, dones, info)   rail_env.py:501-634
  RailEnv.agents[i].state / .position / .speed_counter.is_cell_entry ...   eval_env.py:27-31,86-88
  RailEnv.action_required(agent), .dones, .rewards_dict, ._max_episode_steps, .number_of_agents
  TreeObsForRailEnv(max_nodes, max_pred_depth).set_env/reset/get_many/get_properties   main.cpp:17-22

World generation stays reference Python (north star): `RailEnv(...)` with generator arguments
imports the reference's `flatland` package for rail/line/timetable generation at reset time and
uploads the result; `RailEnv.from_world(world)` / `RailEnv.view(batch, e)` need no reference.

copy.deepcopy(env) gives an independent environment, as on the reference: it gets its own batch of one environment, a
device copy of env's slot (BatchedRailEnv.fork_of: world, tables, caches, state, schedule position and the current
observation), whether env owns its batch or is a view into a shared one, plus copies of the host attributes (dones,
rewards, observation, elapsed steps, world dict), a new TreeObsForRailEnv bound to the copy and a deep copy of the
reference environment that generates its worlds, if any.  Given the same action dicts, the copy then returns what env
returns, across episode ends too; stepping one leaves the other unchanged.
"""
import copy
from enum import IntEnum

import numpy as np
import torch

from . import _lib
from .batch import BatchedRailEnv
from .worlds import world_from_reference_env


class TrainState(IntEnum):  # step_utils/states.py:5-25
    WAITING = 0
    READY_TO_DEPART = 1
    MALFUNCTION_OFF_MAP = 2
    MOVING = 3
    STOPPED = 4
    MALFUNCTION = 5
    DONE = 6

    def is_malfunction_state(self):
        return self in (TrainState.MALFUNCTION, TrainState.MALFUNCTION_OFF_MAP)

    def is_off_map_state(self):
        return self in (TrainState.WAITING, TrainState.READY_TO_DEPART, TrainState.MALFUNCTION_OFF_MAP)

    def is_on_map_state(self):
        return self in (TrainState.MOVING, TrainState.STOPPED, TrainState.MALFUNCTION)

    def __str__(self):
        return "TrainState." + self.name


class _SpeedCounter:  # step_utils/speed_counter.py
    def __init__(self, speed, counter):
        self.speed, self.counter = speed, counter

    @property
    def max_count(self):
        return int(1 / self.speed) - 1

    @property
    def is_cell_entry(self):
        return self.counter == 0

    @property
    def is_cell_exit(self):
        return self.counter == self.max_count


class _MalfunctionHandler:  # step_utils/malfunction_handler.py
    def __init__(self, down, num):
        self.malfunction_down_counter, self.num_malfunctions = down, num

    @property
    def in_malfunction(self):
        return self.malfunction_down_counter > 0

    @property
    def malfunction_counter_complete(self):
        return self.malfunction_down_counter == 0


class _ActionSaver:
    def __init__(self, saved):
        self.saved_action = saved or None

    @property
    def is_action_saved(self):
        return self.saved_action is not None


class AgentView:
    """Read-only host mirror of one agent (the attributes of flatland.envs.agent_utils.EnvAgent that
    consumers of the hot path read)."""

    def __init__(self, handle, world, s):
        i = handle
        self.handle = i
        self.initial_position = tuple(int(x) for x in world["init_pos"][i])
        self.initial_direction = int(world["init_dir"][i])
        self.target = tuple(int(x) for x in world["target"][i])
        self.earliest_departure = int(world["earliest"][i])
        self.latest_arrival = int(world["latest"][i])
        self.state = TrainState(int(s["state"][i]))
        self.position = None if s["pos"][i][0] < 0 else tuple(int(x) for x in s["pos"][i])
        self.direction = int(s["dir"][i])
        self.old_position = None if s["old_pos"][i][0] < 0 else tuple(int(x) for x in s["old_pos"][i])
        self.old_direction = None if s["old_dir"][i] < 0 else int(s["old_dir"][i])
        self.arrival_time = None if s["arrival"][i] < 0 else int(s["arrival"][i])
        self.speed_counter = _SpeedCounter(float(world["speed"][i]), int(s["ctr"][i]))
        self.malfunction_handler = _MalfunctionHandler(int(s["mal"][i]), int(s["nmal"][i]))
        self.action_saver = _ActionSaver(int(s["saved"][i]))
        self.moving = False


class TreeObsForRailEnv:
    """flatland_cutils.TreeObsForRailEnv façade (flatland_cutils/src/treeobs.h:133-169).  The tree is
    built on the GPU for the whole batch by fl_observe; this object hands out the rows of one env."""

    def __init__(self, max_nodes=31, max_pred_depth=500):
        if (max_nodes, max_pred_depth) != (_lib.MAX_NODES, _lib.PRED_DEPTH):
            raise ValueError("the CUDA tree observation is built for max_nodes=31, max_pred_depth=500 "
                             "(solution/impl_config.py:17-18)")
        self.max_nodes, self.max_pred_depth = max_nodes, max_pred_depth
        self.env = None

    def set_env(self, env):
        self.env = env

    def reset(self):
        pass  # deadlock flags are cleared by fl_reset together with the agents

    def get_many(self, handles=None):
        env = self.env
        o = env._obs_host()
        n = env.get_num_agents()
        handles = list(range(n)) if handles is None else list(handles)
        if handles != list(range(n)):
            raise ValueError("flatland_cutils builds observations for all handles in order (treeobs.cpp:94-102)")
        return (o["agent_attr"].tolist(),
                (o["forest"].tolist(), o["adjacency"].tolist(), o["node_order"].tolist(), o["edge_order"].tolist()))

    def get_properties(self):
        env = self.env
        o = env._obs_host()
        w = env.world
        s = env._state_host()
        env_config = {"curr_step": int(env._elapsed_steps), "n_agents": env.get_num_agents(),
                      "max_timesteps": int(w["T"]), "height": int(w["H"]), "width": int(w["W"])}
        props = {
            "dist_target": [float(x) for x in o["dist_target"]],
            "deadlocked": [float(x) for x in s["deadlocked"]],
            "ready_not_depart": [float(x == TrainState.READY_TO_DEPART) for x in s["state"]],
            "earliest_departure": [float(x) for x in w["earliest"]],
            "latest_arrival": [float(x) for x in w["latest"]],
            "speed": [float(np.float32(x)) for x in w["speed"]],
        }
        valid = [[bool(v) for v in row] for row in o["valid_actions"]]
        return env_config, props, valid


class RailEnv:
    """Drop-in for flatland.envs.rail_env.RailEnv on the hot path (one environment = one row of a
    BatchedRailEnv)."""

    def __init__(self, width=None, height=None, rail_generator=None, line_generator=None, number_of_agents=2,
                 obs_builder_object=None, malfunction_generator=None, remove_agents_at_target=True,
                 random_seed=None, record_steps=False, *, world=None, batch=None, index=0, device="cuda:0"):
        if not remove_agents_at_target:
            raise ValueError("remove_agents_at_target=False is not supported (reference default is True)")
        self.width, self.height, self.number_of_agents = width, height, number_of_agents
        self.device = device
        self.world = world
        self._batch, self._e = batch, index
        self._ref_env = None
        self._gen_args = None
        if world is None and batch is None:
            self._gen_args = dict(width=width, height=height, rail_generator=rail_generator,
                                  line_generator=line_generator, number_of_agents=number_of_agents,
                                  malfunction_generator=malfunction_generator, random_seed=random_seed)
        self.obs_builder = obs_builder_object or TreeObsForRailEnv()
        self.obs_builder.set_env(self)
        self.dones, self.rewards_dict, self.obs_dict = {}, {}, None
        self._max_episode_steps = None if world is None else int(world["T"])
        self._elapsed_steps = 0
        self._cache = {}
        self._was_reset = False

    # -- constructors ----------------------------------------------------------------------------
    @classmethod
    def from_world(cls, world, device="cuda:0"):
        return cls(width=int(world["W"]), height=int(world["H"]), number_of_agents=int(world["N"]), world=world,
                   device=device)

    @classmethod
    def view(cls, batch, worlds, e):
        """A reference-API view of environment e of an existing batch (stepping is done on the batch).  The view goes stale
        when its slot gets another environment (BatchedRailEnv.replace_worlds, copy_from, restore): build a new one."""
        w = worlds[e]
        return cls(width=int(w["W"]), height=int(w["H"]), number_of_agents=int(w["N"]), world=w, batch=batch, index=e)

    def __deepcopy__(self, memo):
        """An independent environment with its own batch of one (see the module docstring)."""
        new = RailEnv.__new__(RailEnv)
        memo[id(self)] = new
        new.width, new.height, new.number_of_agents, new.device = self.width, self.height, self.number_of_agents, self.device
        new.world = copy.deepcopy(self.world, memo)
        new._batch = None if self._batch is None else BatchedRailEnv.fork_of(self._batch, [self._e])
        new._e = 0
        new._ref_env = copy.deepcopy(self._ref_env, memo)
        new._gen_args = copy.deepcopy(self._gen_args, memo)
        new.obs_builder = TreeObsForRailEnv()
        new.obs_builder.set_env(new)
        new.dones, new.rewards_dict = dict(self.dones), dict(self.rewards_dict)
        new.obs_dict = copy.deepcopy(self.obs_dict, memo)
        new._max_episode_steps, new._elapsed_steps, new._was_reset = self._max_episode_steps, self._elapsed_steps, self._was_reset
        new._cache = {}
        return new

    # -- host mirrors ----------------------------------------------------------------------------
    def _state_host(self):
        if "state" not in self._cache:
            self._cache["state"] = self._batch.state_numpy(self._e)
        return self._cache["state"]

    def _obs_host(self):
        if "obs" not in self._cache:
            self._cache["obs"] = {k: v[self._e].cpu().numpy() for k, v in self._batch.obs.items()}
        return self._cache["obs"]

    @property
    def agents(self):
        if "agents" not in self._cache:
            s = self._state_host()
            self._cache["agents"] = [AgentView(i, self.world, s) for i in range(int(self.world["N"]))]
        return self._cache["agents"]

    def get_num_agents(self):
        return 0 if self.world is None else int(self.world["N"])

    def get_agent_handles(self):
        return range(self.get_num_agents())

    def action_required(self, agent):  # rail_env.py:243-258
        return agent.state == TrainState.READY_TO_DEPART or \
            (agent.state.is_on_map_state() and agent.speed_counter.is_cell_entry)

    def get_info_dict(self):  # rail_env.py:452-468
        ags = self.agents
        return {"action_required": {i: self.action_required(a) for i, a in enumerate(ags)},
                "malfunction": {i: a.malfunction_handler.malfunction_down_counter for i, a in enumerate(ags)},
                "speed": {i: a.speed_counter.speed for i, a in enumerate(ags)},
                "state": {i: a.state for i, a in enumerate(ags)}}

    # -- reset / step ----------------------------------------------------------------------------
    def _generate_world(self, regenerate_rail, regenerate_schedule, random_seed):
        """Runs the reference's generators (out of scope for the GPU path) and extracts the world."""
        try:
            from flatland.envs.rail_env import RailEnv as RefRailEnv
            from flatland.core.env_observation_builder import DummyObservationBuilder
        except ImportError as e:
            raise _lib.FlatlandB200Error(
                "world generation uses the reference's Python generators; `flatland` is not importable (%s). "
                "Use RailEnv.from_world(...) with a pre-generated world instead." % e)
        if self._ref_env is None:
            a = self._gen_args
            self._ref_env = RefRailEnv(width=a["width"], height=a["height"], rail_generator=a["rail_generator"],
                                       line_generator=a["line_generator"], number_of_agents=a["number_of_agents"],
                                       obs_builder_object=DummyObservationBuilder(),
                                       malfunction_generator=a["malfunction_generator"], random_seed=a["random_seed"])
        self._ref_env.reset(regenerate_rail, regenerate_schedule, random_seed=random_seed)
        return world_from_reference_env(self._ref_env)

    def reset(self, regenerate_rail=True, regenerate_schedule=True, *, random_seed=None):
        own_batch = self._gen_args is not None or self._batch is None
        if self._gen_args is not None:
            self.world = self._generate_world(regenerate_rail, regenerate_schedule, random_seed)
            self._batch = None
        # reset(False, False) on a world that is already resident keeps the agent objects and the malfunction generator of
        # the reference (rail_env.py:260-357: nothing regenerated, no RNG consumed): the schedule carries on and
        # arrival_time survives.  Every other reset builds fresh agents.
        same_agents = self._batch is not None and self._was_reset and not regenerate_rail and not regenerate_schedule
        if own_batch:
            if self._batch is None:
                self._batch, self._e = BatchedRailEnv([self.world], device=self.device), 0
            self._batch.reset(same_agents=same_agents)
        else:
            mask = np.zeros(self._batch.E, np.uint8)
            mask[self._e] = 1
            self._batch.reset(env_mask=mask, same_agents=same_agents)
        self._was_reset = True
        w = self.world
        self.height, self.width, self.number_of_agents = int(w["H"]), int(w["W"]), int(w["N"])
        self._max_episode_steps, self._elapsed_steps = int(w["T"]), 0
        self._cache = {}
        n = self.get_num_agents()
        self.dones = dict.fromkeys(list(range(n)) + ["__all__"], False)
        self.rewards_dict = {}
        self.obs_builder.set_env(self)
        self.obs_builder.reset()
        self.obs_dict = self.obs_builder.get_many(list(range(n)))
        return self.obs_dict, self.get_info_dict()

    def step(self, action_dict_):
        n = self.get_num_agents()
        if self.dones.get("__all__"):
            raise Exception("Episode is done, cannot call step()")  # rail_env.py:508-509
        b = self._batch
        if b.E != 1:
            raise _lib.FlatlandB200Error("RailEnv.step drives a batch of one env; step a shared batch with "
                                         "BatchedRailEnv.step and refresh the views with after_batch_step()")
        acts = np.full((1, n), _lib.ACTION_ABSENT, np.uint8)
        for i, a in action_dict_.items():
            if 0 <= int(i) < n:
                a = int(a)
                acts[0, int(i)] = a if 0 <= a <= 4 else 5  # any invalid value -> DO_NOTHING on the device
        b.step(torch.from_numpy(acts).to(b.device))
        return self.after_batch_step()

    def after_batch_step(self):
        """Refreshes the host mirrors after the batch was stepped; returns what step() returns."""
        n = self.get_num_agents()
        b = self._batch
        self._cache = {}
        self._elapsed_steps = int(b.t["elapsed"][self._e].item())
        rew = b.rewards[self._e].cpu().numpy()
        don = b.dones[self._e].cpu().numpy()
        self.rewards_dict = {i: int(rew[i]) for i in range(n)}
        self.dones = {i: bool(don[i]) for i in range(n)}
        self.dones["__all__"] = bool(don[n])
        self.obs_dict = self.obs_builder.get_many(list(range(n)))
        return self.obs_dict, self.rewards_dict, self.dones, self.get_info_dict()
