"""Base env specs: the tables of PogostickV1Env / BowV1Env, batched.

These classes hold the SAME attribute names the reference's base envs expose through the wrapper
chain (pogostick_v1_env.py:26-84, bow_v1_env.py:26-82) because the reference's wrapper
constructors — and user scripts — read and mutate them by name.  They do not implement `step`:
`_resolve` reports, for one action id, which branch of the reference's if/elif chain
(pogostick_v1_env.py:244-347, bow_v1_env.py:242-320) would run, and the compiler turns that into a
per-config table for the CUDA kernels.
"""
from . import spaces
from .core import Env, ActionEntry, ResetProgram, _Invalid
from . import opcodes as oc


class NovelGridworldBatchEnv(Env):
    """Common skeleton of the two v1 envs (they differ in items, recipes, one manipulation action and
    the craft reward — `diff pogostick_v1_env.py bow_v1_env.py`)."""

    env_id = None
    _ITEMS = ()
    _GOAL = None
    _ITEMS_QUANTITY = ()
    _MANIPULATION = ()
    _RECIPES = ()
    # name -> cost tables of craft() (pogostick_v1_env.py:433-436,447-450,463-470 / bow_v1_env.py:406,418,432-437)
    _COST_MISSING = {}
    _COST_NO_TABLE = {}
    _COST_OK = {}
    _CRAFT_REWARD_IS_DONE = False      # bow_v1_env.py:424 uses reward_done, pogostick_v1_env.py:455 reward_intermediate
    _BREAK_REWARD_ITEMS = ('tree_log',)  # base Break rewards these (pogostick_v1_env.py:288; v0: pogostick_v0_env.py:312)
    _PLACES_TREE_TAP = False           # pogostick_v0_env.py:155-178

    def __init__(self, env=None, num_envs=1, device=None, seed=0, first_env_gid=0, auto_reset=False,
                 max_episode_steps=0, messages=False, strict_actions=False, obs_format='i32', episode_end_info=False,
                 reset_rng='philox'):
        self.env = env                                  # env to restore in reset (pogostick_v1_env.py:29,89-109)
        self.num_envs = int(num_envs)
        self.device = device
        self.rng_seed = int(seed)
        self.first_env_gid = int(first_env_gid)
        # batch extensions (not in the reference): regenerate finished episodes inside step(), optional truncation cap,
        # info['message'] for batched envs (always on when num_envs == 1)
        self.auto_reset = bool(auto_reset)
        self.max_episode_steps = int(max_episode_steps)
        self.messages = bool(messages)
        # strict_actions: a batched step raises like the reference (wrappers.py:76, pogostick_v1_env.py:236) when any env
        # was given an id its chain rejects — one device-to-host read per step; off, the step is a no-op for that env,
        # info['invalid'] marks it and the sticky error flag / NGW_STAT_INVALID count it.  obs_format: 'i32' | 'u8' | 'hits'
        # rows (runtime.obs_to_vector turns the narrow ones back into the reference's vector).
        self.strict_actions = bool(strict_actions)
        self.obs_format = obs_format
        # episode_end_info: a batched step's info also carries 'TimeLimit.truncated' (the step hit max_episode_steps and
        # the env did not end the episode itself) and 'terminal_observation' (with auto_reset, the last observation of
        # each finished episode, valid where done) — what a learner needs to bootstrap at a time limit
        self.episode_end_info = bool(episode_end_info)
        # reset_rng: 'philox' (default) draws maps from the counter-based generator keyed by (seed, env id, episode) — the
        # reference's distribution, not its stream.  'numpy' draws them from the reference's own legacy np.random stream:
        # env i starts from np.random.seed(seed + first_env_gid + i) and continues it episode after episode; with
        # num_envs == 1, reset() instead draws from (and advances) the process's global np.random, as the reference does.
        if reset_rng not in ('philox', 'numpy'):
            raise ValueError("reset_rng must be 'philox' or 'numpy'")
        self.reset_rng = reset_rng

        self.map_size = 10
        self.direction_id = {'NORTH': 0, 'SOUTH': 1, 'WEST': 2, 'EAST': 3}
        self.items = set(self._ITEMS)
        self.items_id = self.set_items_id(self.items)
        self.unbreakable_items = {'air', 'wall'}
        self.goal_item_to_craft = self._GOAL
        self.items_quantity = dict(self._ITEMS_QUANTITY)
        self.inventory_items_quantity = {item: 0 for item in self.items}
        self.selected_item = ''
        self.entities = set()

        # action ids: manipulation, then Craft_<sorted recipes>, then Select_<sorted breakable items>
        self.actions_id = dict()
        self.manipulation_actions_id = {name: i for i, name in enumerate(self._MANIPULATION)}
        self.actions_id.update(self.manipulation_actions_id)
        self.recipes = {out: {'input': dict(inp), 'output': {out: qty}} for out, inp, qty in self._RECIPES}
        base = len(self.actions_id)
        self.craft_actions_id = {'Craft_' + item: base + i for i, item in enumerate(sorted(self.recipes))}
        self.actions_id.update(self.craft_actions_id)
        base = len(self.actions_id)
        selectable = sorted(self.items ^ self.unbreakable_items)
        self.select_actions_id = {'Select_' + item: base + i for i, item in enumerate(selectable)}
        self.actions_id.update(self.select_actions_id)
        self.action_space = spaces.Discrete(len(self.actions_id))

        self.max_items = 20
        # the reference declares this (stale) space and never updates it (pogostick_v1_env.py:76-77)
        self.observation_space = spaces.Dict(
            {'map': spaces.Box(low=0, high=self.max_items, shape=(self.map_size, self.map_size, 1))})

        self.reward_intermediate = 10
        self.reward_done = 50

        # mirrors of the per-step bookkeeping attributes; refreshed by the runtime for num_envs == 1
        self.map = None
        self.agent_location = (1, 1)
        self.agent_facing_str = 'NORTH'
        self.agent_facing_id = 0
        self.block_in_front_str = 'air'
        self.block_in_front_id = 0
        self.block_in_front_location = (0, 0)
        self.last_action = 'Forward'
        self.step_count = 0
        self.last_step_cost = 0
        self.last_reward = 0
        self.last_done = False

        self._top = self
        self._runtime = None

    # ------------------------------------------------------------------ reference helper surface
    def set_items_id(self, items):
        """air -> 0, every other name by sorted order (pogostick_v1_env.py:200-212)."""
        ids = {}
        offset = 0 if 'air' in items else 1
        if 'air' in items:
            ids['air'] = 0
        for name in sorted(items):
            if name != 'air':
                ids[name] = len(ids) + offset
        return ids

    def add_new_items(self, new_items_quantity):
        """pogostick_v1_env.py:495-501.  The reference also calls reset() here.  A batched reset at wrapper-construction
        time would be thrown away by the user's own reset(), so it is skipped, except for one env on the numpy stream:
        there the reference's reset consumes draws of the global np.random, which a seeded script's later maps depend on."""
        for item in new_items_quantity:
            self.items.add(item)
            self.items_id.setdefault(item, len(self.items_id))
            self.items_quantity.update({item: new_items_quantity[item]})
        self.inventory_items_quantity = {item: 0 for item in self.items}
        if self.reset_rng == 'numpy' and self.num_envs == 1:
            self._construction_reset()

    def _construction_reset(self):
        """The base env's reset() with its tables as they are now, on a one-env numpy-stream batch: it advances the global
        np.random exactly as the reference's reset does, and raises where that raises."""
        import torch
        from .compiler import compile_chain
        from .runtime import BatchHandle, global_stream_reset
        h = BatchHandle([compile_chain(self)], 1, self.device, self.rng_seed, self.first_env_gid, reset_rng='numpy')
        try:
            global_stream_reset(h, want_obs=False)
            torch.cuda.current_stream(h.device).synchronize()
            if int(h.error_flags[0].item()) & oc.ERR_PLACEMENT:
                raise AssertionError("Cannot place items, increase map size!")      # pogostick_v1_env.py:167
        finally:
            h.close()

    def remap_action(self, actions_id, start_action_id):
        """Shuffle names until the mapping changes (pogostick_v1_env.py:476-493); draws from the global
        legacy np.random stream exactly as the reference does, so a seeded script remaps identically."""
        import numpy as np
        while True:
            names = list(actions_id.keys())
            np.random.shuffle(names)
            remapped = {names[i - start_action_id]: i
                        for i in range(start_action_id, start_action_id + len(names))}
            if actions_id != remapped:
                return remapped

    # ------------------------------------------------------------------ flattening hooks
    def _recipe_descriptor(self, item, cost_missing, cost_no_table, cost_ok, reward_ok):
        rec = self.recipes[item]
        return {
            'inputs': [(self.items_id[name], qty) if name in self.items_id else (oc.NONE, qty)
                       for name, qty in rec['input'].items()],
            'out_item': self.items_id[item], 'out_qty': rec['output'][item],
            'needs_table': len(rec['input']) > 1,
            'cost_missing': float(cost_missing), 'cost_no_table': float(cost_no_table),
            'cost_ok': float(cost_ok), 'reward_ok': int(reward_ok),
        }

    def _base_craft_entry(self, item):
        if item not in self.recipes:
            raise _Invalid("KeyError: recipes[%r]" % item)
        reward_ok = self.reward_done if self._CRAFT_REWARD_IS_DONE else self.reward_intermediate
        desc = self._recipe_descriptor(item, self._COST_MISSING.get(item, 0), self._COST_NO_TABLE.get(item, 0),
                                       self._COST_OK.get(item, 0), reward_ok)
        return ActionEntry(oc.OP_CRAFT, recipe=desc)

    def _manipulation_entry(self, name):
        raise NotImplementedError

    def _resolve(self, action_id):
        # pogostick_v1_env.py:236 — unknown id raises ValueError before anything happens
        if action_id not in self.actions_id.values():
            raise _Invalid("ValueError: %r is not in actions_id" % (action_id,))
        # the if/elif chain compares by id in this fixed order (pogostick_v1_env.py:244-347)
        for name in self._MANIPULATION:
            if action_id == self.actions_id[name]:
                return self._manipulation_entry(name)
        for name, idx in self.craft_actions_id.items():
            if idx == action_id:
                return self._base_craft_entry('_'.join(name.split('_')[1:]))
        for name, idx in self.select_actions_id.items():
            if idx == action_id:
                item = '_'.join(name.split('_')[1:])
                return ActionEntry(oc.OP_SELECT, arg=self.items_id.get(item, oc.NONE) if item in self.items else oc.NONE)
        return ActionEntry(oc.OP_NOOP)

    def _reset_program(self):
        prog = ResetProgram([(self.items_id[name], qty) for name, qty in self.items_quantity.items()])
        if self._PLACES_TREE_TAP:
            prog.ops.append((oc.RESET_TREETAP, self.items_id['tree_tap'], self.items_id['tree_log'], 0, 0))
        return prog

    def _lidar(self):
        return None

    def _external_action_ids(self):
        return sorted(set(self.actions_id.values()))

    # ------------------------------------------------------------------ gym API -> runtime
    def _runtime_for(self, entry):
        from .runtime import ChainRuntime
        if entry is not self._top:
            raise NotImplementedError(
                "reset()/step() must be called on the outermost wrapper of the chain (the batched runtime "
                "is compiled from it); got %s, outermost is %s" % (type(entry).__name__, type(self._top).__name__))
        if self._runtime is None:
            self._runtime = ChainRuntime(self)
        return self._runtime

    def reset(self, map_size=None, items_id=None, items_quantity=None):
        # pogostick_v1_env.py:111-116
        if map_size is not None:
            self.map_size = map_size
        if items_id is not None:
            self.items_id = items_id
        if items_quantity is not None:
            self.items_quantity = items_quantity
        return self._runtime_for(self).reset()

    def step(self, action_id):
        return self._runtime_for(self).step(action_id)

    def get_observation(self):
        """Dict of LIVE views of the state tensors (pogostick_v1_env.py:214-228)."""
        return self._runtime_for(self._top).dict_observation()

    def render(self, mode='human', title=None, env_index=0):
        """Host visualisation of ONE env of the batch from the exported state: the picture of pogostick_v1_env.py:556-620
        (grid, facing arrow, info panel, win banner, inventory legend).  mode 'human' draws it with matplotlib when that is
        installed and falls back to text; 'ansi' prints and returns the text form; 'spec' returns the drawing list."""
        from . import render as R
        rt = self._runtime_for(self._top)
        if rt.handle is None:
            raise RuntimeError("render() before reset()")
        h, names = rt.handle, rt.compiled.item_names
        grid = h.map[env_index].cpu().numpy()
        r, c, facing, sel = [int(x) for x in h.pose[env_index].cpu().numpy()]
        inv = h.inventory[env_index].cpu().numpy()
        if self.num_envs == 1:
            last = dict(step_count=self.step_count, last_action=self.last_action, last_reward=self.last_reward,
                        last_step_cost=self.last_step_cost, last_done=self.last_done)
        else:                                                   # batched: the latest outputs of that env
            last = dict(step_count=int(h.ep_len[env_index].item()), last_action=self.last_action,
                        last_reward=int(h.reward[env_index].item()), last_step_cost=float(h.step_cost[env_index].item()),
                        last_done=bool(h.done[env_index].item()))
        spec = R.render_spec(self.env_id, grid, (r, c), R.FACING[facing], dict(self.items_id),
                             {n: int(inv[i]) for i, n in enumerate(names) if n in self.items}, self.goal_item_to_craft,
                             selected_item=names[sel] if sel else '', title=title, **last)
        if mode == 'spec':
            return spec
        if mode != 'ansi':
            try:
                R.draw(spec)
                return None
            except ImportError:
                pass
        text = R.to_text(spec)
        print(text)
        return text

    def seed(self, seed=None):
        """The reference has no seed() (it draws from the global np.random).  Here it re-keys the Philox generator, or on
        the numpy stream re-seeds env gid with np.random.seed(seed + gid) (one env: reset() follows the global
        np.random instead, see reset_rng)."""
        if seed is not None:
            self.rng_seed = int(seed)
            self.close()                       # the next reset() builds a handle with the new key
        return [self.rng_seed]

    def close(self):
        if self._runtime is not None:
            self._runtime.close()
            self._runtime = None


class PogostickV1Env(NovelGridworldBatchEnv):
    """Goal: craft 1 pogo_stick (pogostick_v1_env.py:17-84)."""
    env_id = 'NovelGridworld-Pogostick-v1'
    _ITEMS = ('air', 'crafting_table', 'plank', 'pogo_stick', 'rubber', 'stick', 'tree_log', 'tree_tap', 'wall')
    _GOAL = 'pogo_stick'
    _ITEMS_QUANTITY = (('crafting_table', 1), ('tree_log', 5))
    _MANIPULATION = ('Forward', 'Left', 'Right', 'Break', 'Place_tree_tap', 'Extract_rubber')
    _RECIPES = (('pogo_stick', (('stick', 4), ('plank', 2), ('rubber', 1)), 1),
                ('stick', (('plank', 2),), 4),
                ('plank', (('tree_log', 1),), 4),
                ('tree_tap', (('plank', 5), ('stick', 1)), 1))
    _COST_MISSING = {'tree_tap': 360.0, 'pogo_stick': 480.0}
    _COST_NO_TABLE = {'tree_tap': 720.0, 'pogo_stick': 840.0}
    _COST_OK = {'plank': 1200.0, 'stick': 2400.0, 'tree_tap': 7200.0, 'pogo_stick': 8400.0}

    def _manipulation_entry(self, name):
        if name == 'Extract_rubber':
            return ActionEntry(oc.OP_EXTRACT_RUBBER, arg=1)          # pogostick_v1_env.py:323
        return ActionEntry({'Forward': oc.OP_FORWARD, 'Left': oc.OP_LEFT, 'Right': oc.OP_RIGHT,
                            'Break': oc.OP_BREAK, 'Place_tree_tap': oc.OP_PLACE_TREE_TAP}[name])


class BowV1Env(NovelGridworldBatchEnv):
    """Goal: craft 1 bow (bow_v1_env.py:17-82)."""
    env_id = 'NovelGridworld-Bow-v1'
    _ITEMS = ('air', 'bow', 'crafting_table', 'plank', 'stick', 'string', 'tree_log', 'wall', 'wool')
    _GOAL = 'bow'
    _ITEMS_QUANTITY = (('crafting_table', 1), ('tree_log', 3), ('wool', 2))
    _MANIPULATION = ('Forward', 'Left', 'Right', 'Break', 'Extract_string')
    _RECIPES = (('bow', (('stick', 3), ('string', 3)), 1),
                ('stick', (('plank', 2),), 4),
                ('plank', (('tree_log', 1),), 4))
    _COST_MISSING = {'bow': 480.0}
    _COST_NO_TABLE = {'bow': 840.0}
    _COST_OK = {'plank': 1200.0, 'stick': 2400.0, 'bow': 8400.0}
    _CRAFT_REWARD_IS_DONE = True

    def _manipulation_entry(self, name):
        if name == 'Extract_string':
            return ActionEntry(oc.OP_EXTRACT_STRING, arg=4)          # bow_v1_env.py:297
        return ActionEntry({'Forward': oc.OP_FORWARD, 'Left': oc.OP_LEFT, 'Right': oc.OP_RIGHT,
                            'Break': oc.OP_BREAK}[name])


class PogostickV0Env(PogostickV1Env):
    """Ingredients pre-placed, one tree_tap next to a random tree_log, rewards for breaking stick / plank, craft reward
    = reward_done (pogostick_v0_env.py:44,155-178,312,479)."""
    env_id = 'NovelGridworld-Pogostick-v0'
    _ITEMS_QUANTITY = (('crafting_table', 1), ('stick', 4), ('plank', 2), ('tree_log', 2))
    _BREAK_REWARD_ITEMS = ('stick', 'plank')
    _CRAFT_REWARD_IS_DONE = True
    _PLACES_TREE_TAP = True


class BowV0Env(BowV1Env):
    """Ingredients pre-placed, rewards for breaking stick / string, craft reward = reward_intermediate
    (bow_v0_env.py:44,286,424)."""
    env_id = 'NovelGridworld-Bow-v0'
    _ITEMS_QUANTITY = (('crafting_table', 1), ('stick', 3), ('string', 3))
    _BREAK_REWARD_ITEMS = ('stick', 'string')
    _CRAFT_REWARD_IS_DONE = False
