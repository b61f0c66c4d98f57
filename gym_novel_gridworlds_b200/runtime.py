"""Runtime: torch tensors for device memory and streams, libngw_b200.so for everything that computes.

`BatchHandle`  — thin owner of one `ngw_handle` (a batch of envs sharing a map size, 1..255 configs).
`ChainRuntime` — what `reset()` / `step()` of the outermost wrapper talk to: compiles the chain, (re)creates the
                 handle when a table changed, and shapes results like the reference does (Dict views or the lidar
                 vector; python scalars when num_envs == 1, tensors otherwise).
`MixedBatch`   — several wrapper chains in ONE batch / one launch (per-env config ids).
"""
import ctypes as C

import numpy as np
import torch

from . import capi
from . import opcodes as oc
from .capi import ConfigC, StateViewC
from .compiler import compile_chain


class _DeviceArray(object):
    """Zero-copy torch view of library-owned device memory (numba-style __cuda_array_interface__)."""

    def __init__(self, ptr, shape, typestr, owner):
        self.__cuda_array_interface__ = {'shape': tuple(shape), 'typestr': typestr, 'data': (int(ptr), False),
                                         'version': 2, 'strides': None}
        self._owner = owner


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


_OBS_FORMATS = {'i32': capi.OBS_I32, 'u8': capi.OBS_U8, 'hits': capi.OBS_HITS}
_RESET_RNGS = {'philox': capi.RNG_PHILOX, 'numpy': capi.RNG_NUMPY}


def _tail_offset(c, obs_format):
    """Byte offset of the int32 inventory tail in a narrow row of config `c` (include/ngw.h, NGW_OBS_U8 / NGW_OBS_HITS)."""
    n = c.n_lidar_items * c.n_beams if obs_format == 'u8' else 2 * c.n_beams
    return (n + 3) & ~3


def _split_rows(rows, c, obs_format):
    nl, ni = c.n_lidar_items * c.n_beams, c.n_inv_obs
    if obs_format == 'i32':
        return rows[:, :nl], rows[:, nl:nl + ni]
    off = _tail_offset(c, obs_format)
    tail = rows[:, off:off + 4 * ni]
    tail = tail.view(torch.int32) if isinstance(tail, torch.Tensor) else tail.view(np.int32)
    if obs_format == 'u8':
        return rows[:, :nl], tail
    return rows[:, :2 * c.n_beams].reshape(rows.shape[0], c.n_beams, 2), tail


def _rows_to_vector(rows, c, obs_format, width):
    """int32 [n, width] vector of config `c` from rows (torch) laid out for that config.  Only bounded index arithmetic:
    rows of another config (mixed batches, discarded by the caller) decode to garbage but never index out of range."""
    n, L, B = rows.shape[0], c.n_lidar_items, c.n_beams
    lidar, tail = _split_rows(rows, c, obs_format)
    out = torch.zeros((n, width), dtype=torch.int32, device=rows.device)
    if obs_format == 'hits':
        item = lidar[:, :, 0].to(torch.int64)
        rng = torch.where((item > 0) & (item <= L), lidar[:, :, 1].to(torch.int32), 0)
        vec = torch.zeros((n, B, L), dtype=torch.int32, device=rows.device)
        vec.scatter_(2, (item - 1).clamp(0, L - 1).unsqueeze(2), rng.unsqueeze(2))
        out[:, :L * B] = vec.view(n, L * B)
    else:
        out[:, :L * B] = lidar.to(torch.int32)
    out[:, L * B:L * B + c.n_inv_obs] = tail
    return out


def obs_to_vector(rows, compiled, obs_format, cfg_ids=None):
    """The reference's observation vector (observation_wrappers.py:70-80), int32 [n, obs_dim], from observation rows
    of any layout ('i32', 'u8', 'hits'; include/ngw.h).  obs_dim is the widest config's; an env's entries beyond its own
    config's L*B + I_obs are 0, as in an 'i32' row.  `compiled`: the batch's compiled chain(s); `cfg_ids` [n]: each
    row's config index (None = config 0).  A CUDA tensor is decoded with torch ops only (no host synchronisation, so
    the call can be captured in a CUDA graph) and gives a tensor; a numpy array gives a numpy array.  Needs no library."""
    compiled = list(compiled) if isinstance(compiled, (list, tuple)) else [compiled]
    if obs_format not in _OBS_FORMATS:
        raise ValueError("unknown obs_format %r" % (obs_format,))
    as_numpy = not isinstance(rows, torch.Tensor)
    if as_numpy:
        rows = np.ascontiguousarray(rows)
        rows = torch.from_numpy(rows if rows.flags.writeable else rows.copy())
        if cfg_ids is not None:
            cfg_ids = torch.from_numpy(np.asarray(cfg_ids, dtype=np.int64))
    width = max([cc.c.n_lidar_items * cc.c.n_beams + cc.c.n_inv_obs for cc in compiled if cc.c.n_beams > 0] or [0])
    if rows.shape[0] == 0:
        # no rows, e.g. the terminal observations of a step that ended no episode (an empty NumPy selection has strides
        # (0, 0), which a narrow row's int32 tail view cannot take)
        out = torch.zeros((0, width), dtype=torch.int32, device=rows.device)
    elif obs_format == 'i32':
        out = rows[:, :width].to(torch.int32).clone()
    else:
        out = torch.zeros((rows.shape[0], width), dtype=torch.int32, device=rows.device)
        for k, cc in enumerate(compiled):
            if cc.c.n_beams <= 0:
                continue
            vec = _rows_to_vector(rows, cc.c, obs_format, width)
            if cfg_ids is None:
                out = vec
                break
            out = torch.where((cfg_ids.to(rows.device) == k).unsqueeze(1), vec, out)
    return out.numpy() if as_numpy else out


class RolloutRecord(object):
    """Reusable per-step buffers of a K-step rollout (BatchHandle.rollout_record, include/ngw.h ngw_set_rollout_record).
    Padded device tensors [max_steps, n_envs_padded, ...] hold the steps; the attributes below are their [:, :n] views,
    element [t][e] being what the t-th of as many single steps would report for env e:
        obs        observation rows (the handle's format) after step t and its auto-reset: what the rollout's policy acts
                   on at step t + 1, and what observe() returns after the t-th single step
        reward, step_cost   float32;  done, result, truncated   uint8
        final_obs  rows like obs, only with final_obs=True: written only where step t's auto-reset regenerated the env
                   (the observation the step produced); other rows keep what they held.
    Flatten with obs.reshape(-1, obs.shape[-1]) to decode narrow rows with BatchHandle.obs_vector / obs_to_vector."""

    def __init__(self, handle, max_steps, final_obs=False):
        if max_steps < 1:
            raise ValueError("max_steps must be >= 1")
        self.handle, self.max_steps = handle, int(max_steps)
        self.obs_format, self.obs_row_bytes = handle.obs_format, handle.obs_row_bytes
        T, npad, n, dev = self.max_steps, handle.n_padded, handle.n, handle.device

        def rows():
            if not handle.obs_dim:
                return None
            if handle.obs_format == 'i32':
                return torch.zeros((T, npad, handle.obs_row_bytes // 4), dtype=torch.int32, device=dev)
            return torch.zeros((T, npad, handle.obs_row_bytes), dtype=torch.uint8, device=dev)

        self.padded = {'obs': rows(), 'final_obs': rows() if final_obs else None}
        for k, dt in (('reward', torch.float32), ('step_cost', torch.float32), ('done', torch.uint8),
                      ('result', torch.uint8), ('truncated', torch.uint8)):
            self.padded[k] = torch.zeros((T, npad), dtype=dt, device=dev)
        for k, t in self.padded.items():
            setattr(self, k, None if t is None else t[:, :n])
        self._c = capi.RolloutRecordC(self.max_steps, *[None if self.padded[k] is None else self.padded[k].data_ptr()
                                                        for k in ('obs', 'reward', 'step_cost', 'done', 'result',
                                                                  'truncated', 'final_obs')])


class BatchHandle(object):
    def __init__(self, compiled, n_envs, device=None, seed=0, first_env_gid=0, cfg_id=None, obs_format='i32',
                 reset_rng='philox'):
        if not torch.cuda.is_available():
            raise RuntimeError("gym_novel_gridworlds_b200 needs a CUDA device (B200, sm_100a); there is no CPU path")
        self.lib = capi.load_library()
        self.compiled = list(compiled)
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        self.n = int(n_envs)
        self.map_size = self.compiled[0].map_size
        if any(cc.map_size != self.map_size for cc in self.compiled):
            raise ValueError("all configs of one batch must share map_size")
        cfgs = (ConfigC * len(self.compiled))()
        for i, cc in enumerate(self.compiled):
            C.memmove(C.byref(cfgs, i * C.sizeof(ConfigC)), C.byref(cc.c), C.sizeof(ConfigC))
        self._h = C.c_void_p()
        capi.check(self.lib, self.lib.ngw_create(C.byref(self._h), cfgs, len(self.compiled), self.n, self.map_size,
                                                 self.device.index, int(first_env_gid), int(seed) & (2 ** 64 - 1)))
        if obs_format not in _OBS_FORMATS:
            raise ValueError("obs_format must be 'i32' (the reference's vector as int32), 'u8' (uint8 lidar ranges) or "
                             "'hits' (one (item, range) byte pair per beam)")
        self.obs_format = obs_format
        if obs_format != 'i32':
            capi.check(self.lib, self.lib.ngw_set_obs_format(self._h, _OBS_FORMATS[obs_format]))
        sv = StateViewC()
        capi.check(self.lib, self.lib.ngw_state(self._h, C.byref(sv)))
        self.inv_stride, self.obs_dim, self.n_padded = sv.inv_stride, sv.obs_dim, sv.n_envs_padded
        self.obs_row_bytes = sv.obs_row_bytes
        ms = self.map_size

        def view(ptr, shape, typestr):
            return torch.as_tensor(_DeviceArray(ptr, shape, typestr, self), device=self.device)

        # LIVE views of the state (what get_observation hands out, pogostick_v1_env.py:222-226)
        self.map = view(sv.map, (self.n_padded, ms, ms), '|i1')[:self.n]
        self.pose = view(sv.pose, (self.n_padded, 4), '|u1')[:self.n]
        self.inventory = view(sv.inventory, (self.n_padded, self.inv_stride), '<i4')[:self.n]
        self.cfg_id = view(sv.cfg_id, (self.n_padded,), '|u1')[:self.n]
        self.episode = view(sv.episode, (self.n_padded,), '<i4')[:self.n]
        self.ep_len = view(sv.ep_len, (self.n_padded,), '<i4')[:self.n]
        self.error_flags = view(sv.error_flags, (self.n_padded,), '<i4')[:self.n]
        with torch.cuda.device(self.device):
            d = max(self.obs_dim, 1)
            if obs_format != 'i32':      # rows: uint8 lidar ranges or hits | pad to 4 | int32 inventory tail (see split_obs)
                self.obs = torch.zeros((self.n, max(self.obs_row_bytes, 4)), dtype=torch.uint8, device=self.device)
            else:
                self.obs = torch.zeros((self.n, d), dtype=torch.int32, device=self.device)
            self.reward = torch.zeros(self.n, dtype=torch.float32, device=self.device)
            self.done = torch.zeros(self.n, dtype=torch.uint8, device=self.device)
            self.step_cost = torch.zeros(self.n, dtype=torch.float32, device=self.device)
            self.result = torch.zeros(self.n, dtype=torch.uint8, device=self.device)
            self._stats = torch.zeros(8, dtype=torch.float64, device=self.device)
        # the output tensors live as long as the handle: their pointers are converted once (step() is host-bound)
        self._out_ptrs = (_ptr(self.obs) if self.obs_dim else None, _ptr(self.reward), _ptr(self.done),
                          _ptr(self.step_cost), _ptr(self.result))
        self._host = None
        if cfg_id is not None:
            self.set_env_configs(cfg_id)
        self.reset_rng = 'philox'
        if reset_rng != 'philox':
            self.set_reset_rng(reset_rng)

    # ------------------------------------------------------------------
    def _stream(self):
        try:                                    # raw handle of torch's current stream, without building a Stream object
            return C.c_void_p(torch._C._cuda_getCurrentRawStream(self.device.index))
        except AttributeError:
            return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def close(self):
        if getattr(self, '_h', None) is not None and self._h.value:
            self.lib.ngw_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_env_configs(self, cfg_id):
        t = torch.as_tensor(cfg_id, dtype=torch.int32, device=self.device).contiguous()
        assert t.numel() == self.n
        capi.check(self.lib, self.lib.ngw_set_env_configs(self._h, _ptr(t), self._stream()))

    def load_state(self, map, pose, inventory, first=0):
        """Inject states (the parity harness's entry; also the `env=` restore of pogostick_v1_env.py:89-109)."""
        m = torch.as_tensor(map, device=self.device).to(torch.int8).contiguous()
        count = m.shape[0]
        m = m.reshape(count, -1)
        p = torch.as_tensor(pose, device=self.device).to(torch.uint8).contiguous()
        v = torch.as_tensor(inventory, device=self.device).to(torch.int32)
        if v.shape[1] != self.inv_stride:
            full = torch.zeros((count, self.inv_stride), dtype=torch.int32, device=self.device)
            full[:, :v.shape[1]] = v
            v = full
        v = v.contiguous()
        assert m.shape[1] == self.map_size ** 2 and p.shape == (count, 4)
        capi.check(self.lib, self.lib.ngw_load_state(self._h, _ptr(m), _ptr(p), _ptr(v), first, count, self._stream()))
        torch.cuda.current_stream(self.device).synchronize()      # m/p/v may be temporaries

    def export_state(self, first=0, count=None, host=False):
        """Copy of `count` env states from env `first` through ngw_export_state: (map int8 [count, ms, ms], pose uint8
        [count, 4], inventory int32 [count, inv_stride]); host=True exports straight into pinned host memory."""
        count = self.n - first if count is None else int(count)
        kw = {'device': 'cpu', 'pin_memory': True} if host else {'device': self.device}
        m = torch.empty((count, self.map_size * self.map_size), dtype=torch.int8, **kw)
        p = torch.empty((count, 4), dtype=torch.uint8, **kw)
        v = torch.empty((count, self.inv_stride), dtype=torch.int32, **kw)
        capi.check(self.lib, self.lib.ngw_export_state(self._h, _ptr(m), _ptr(p), _ptr(v), int(first), count,
                                                       self._stream()))
        if host:
            torch.cuda.current_stream(self.device).synchronize()
        return m.view(count, self.map_size, self.map_size), p, v

    def set_reset_rng(self, kind):
        """'philox' (default): the counter-based map generator.  'numpy': the reference's own legacy np.random stream, one
        state per env, env i seeded as np.random.seed(seed + first_env_gid + i) (ngw_set_reset_rng; calling it again
        re-seeds)."""
        if kind not in _RESET_RNGS:
            raise ValueError("reset_rng must be 'philox' or 'numpy'")
        capi.check(self.lib, self.lib.ngw_set_reset_rng(self._h, _RESET_RNGS[kind], self._stream()))
        self.reset_rng = kind

    def rng_state(self, first=0, count=None):
        """(key uint32 [count, 624], pos int32 [count]): the np.random states of envs first .. first + count - 1 in
        np.random.get_state()'s layout (numpy stream only)."""
        count = self.n - first if count is None else int(count)
        key = torch.empty((count, 624), dtype=torch.int32, device=self.device)
        pos = torch.empty(count, dtype=torch.int32, device=self.device)
        capi.check(self.lib, self.lib.ngw_export_rng_state(self._h, _ptr(key), _ptr(pos), int(first), count, self._stream()))
        return key.cpu().numpy().view(np.uint32), pos.cpu().numpy()

    def load_rng_state(self, key, pos, first=0):
        """Set the np.random states of envs first .. first + len(pos) - 1 (numpy stream only): key uint32 [count, 624],
        pos int32 [count] in [0, 624], as np.random.RandomState(s).get_state()[1:3] gives them."""
        k = np.ascontiguousarray(np.asarray(key, dtype=np.uint32).reshape(-1, 624))
        p = np.ascontiguousarray(np.asarray(pos, dtype=np.int32).reshape(-1))
        if k.shape[0] != p.shape[0]:
            raise ValueError("key and pos must describe the same number of envs")
        kt = torch.from_numpy(k.view(np.int32)).to(self.device)
        pt = torch.from_numpy(p).to(self.device)
        capi.check(self.lib, self.lib.ngw_load_rng_state(self._h, _ptr(kt), _ptr(pt), int(first), int(p.shape[0]),
                                                         self._stream()))
        torch.cuda.current_stream(self.device).synchronize()      # kt / pt are temporaries

    def split_obs(self, obs, cfg=0):
        """(lidar part, inventory tail int32 [n, I_obs]) views of an observation buffer of this handle's format (torch
        tensor or numpy array) for config `cfg` — the two halves of observation_wrappers.py:70-80.  The lidar part is the
        ranges [n, L*B] ('i32', 'u8') or the (item, range) pairs uint8 [n, B, 2] ('hits')."""
        return _split_rows(obs, self.compiled[cfg].c, self.obs_format)

    def obs_vector(self, rows=None):
        """The reference's int32 vector [n, obs_dim] of observation rows of this handle (default: self.obs); see
        obs_to_vector."""
        rows = self.obs if rows is None else rows
        cfg_ids = None
        if len(self.compiled) > 1:
            cfg_ids = self.cfg_id if isinstance(rows, torch.Tensor) else self.cfg_id.cpu().numpy()
        return obs_to_vector(rows, self.compiled, self.obs_format, cfg_ids)

    def reset(self, mask=None, want_obs=True):
        mk = None
        if mask is not None:
            mk = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
        obs = self.obs if (want_obs and self.obs_dim > 0) else None
        capi.check(self.lib, self.lib.ngw_reset(self._h, _ptr(mk), _ptr(obs), self._stream()))
        if mk is not None:
            torch.cuda.current_stream(self.device).synchronize()
        return obs

    def step(self, actions, auto_reset=False, max_episode_steps=0):
        """Device path: `actions` is an int32 CUDA tensor [n]; outputs are the handle's reused tensors."""
        if actions.dtype != torch.int32 or not actions.is_cuda or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.int32).contiguous()
        o = self._out_ptrs
        capi.check(self.lib, self.lib.ngw_step(self._h, actions.data_ptr(), o[0], o[1], o[2], o[3], o[4],
                                               1 if auto_reset else 0, int(max_episode_steps), self._stream()))
        return self.obs, self.reward, self.done, self.step_cost, self.result

    def rollout_record(self, max_steps, final_obs=False):
        """A reusable per-step record for rollout(..., record=) of up to max_steps steps (see RolloutRecord).  final_obs is
        opt-in: it is as large as obs.  Preallocated, it keeps a recorded rollout capturable in a CUDA graph."""
        return RolloutRecord(self, max_steps, final_obs)

    def rollout(self, n_steps, actions=None, policy_seed=0, auto_reset=False, max_episode_steps=0,
                record_actions=False, policy=None, record=None):
        """n_steps consecutive steps in ONE launch (tile resident in shared memory).  actions: int32 CUDA tensor
        [n_steps, n]; None = on-device uniform random policy; policy=(W int32 [obs_dim, A], b int32 [A]) = closed loop,
        action = argmax(b + obs @ W) computed on the device from the current observation.  Returns (obs after the last
        step, reward sum, step_cost sum, episodes finished, last done, last result[, actions taken][, record]).
        record: a RolloutRecord of this handle, filled with every step's transition (set for this call only)."""
        if record is None:
            return self._rollout(n_steps, actions, policy_seed, auto_reset, max_episode_steps, record_actions, policy)
        if record.handle is not self or record.obs_row_bytes != self.obs_row_bytes:
            raise ValueError("rollout: the record was built for another handle or observation format "
                             "(rows of %d bytes, this handle's are %d)" % (record.obs_row_bytes, self.obs_row_bytes))
        capi.check(self.lib, self.lib.ngw_set_rollout_record(self._h, C.byref(record._c)))
        try:
            out = self._rollout(n_steps, actions, policy_seed, auto_reset, max_episode_steps, record_actions, policy)
        finally:
            capi.check(self.lib, self.lib.ngw_set_rollout_record(self._h, None))
        return out + (record,)

    def _rollout(self, n_steps, actions, policy_seed, auto_reset, max_episode_steps, record_actions, policy):
        if policy is not None:
            w = torch.as_tensor(policy[0], device=self.device).to(torch.int32).contiguous()
            b = torch.as_tensor(policy[1], device=self.device).to(torch.int32).contiguous()
            assert w.shape == (self.obs_dim, b.numel()) and b.numel() <= 16
            if not hasattr(self, '_done_count'):
                self._done_count = torch.zeros(self.n, dtype=torch.int32, device=self.device)
            taken = torch.empty((n_steps, self.n), dtype=torch.int32, device=self.device) if record_actions else None
            capi.check(self.lib, self.lib.ngw_rollout_policy(
                self._h, _ptr(w), _ptr(b), int(b.numel()), int(n_steps), _ptr(self.obs), _ptr(self.reward),
                _ptr(self.step_cost), _ptr(self._done_count), _ptr(self.done), _ptr(self.result), _ptr(taken),
                int(bool(auto_reset)), int(max_episode_steps), self._stream()))
            out = (self.obs, self.reward, self.step_cost, self._done_count, self.done, self.result)
            return out + (taken,) if record_actions else out
        if actions is not None:
            actions = actions.to(device=self.device, dtype=torch.int32).contiguous()
            assert actions.shape == (n_steps, self.n)
        if not hasattr(self, '_done_count'):
            self._done_count = torch.zeros(self.n, dtype=torch.int32, device=self.device)
        taken = torch.empty((n_steps, self.n), dtype=torch.int32, device=self.device) if record_actions else None
        capi.check(self.lib, self.lib.ngw_rollout(
            self._h, _ptr(actions), int(n_steps), int(policy_seed) & (2 ** 64 - 1),
            _ptr(self.obs) if self.obs_dim else None, _ptr(self.reward), _ptr(self.step_cost), _ptr(self._done_count),
            _ptr(self.done), _ptr(self.result), _ptr(taken), int(bool(auto_reset)), int(max_episode_steps),
            self._stream()))
        out = (self.obs, self.reward, self.step_cost, self._done_count, self.done, self.result)
        return out + (taken,) if record_actions else out

    def capture_policy_rollout(self, policy, n_steps, auto_reset=False, max_episode_steps=0):
        """SURVEY §8f N1, general policy hook: ONE CUDA graph of n_steps x [actions = policy(obs); ngw_step(actions)].
        `policy` is any callable made of torch ops on the current stream mapping the handle's observation tensor
        (int32 [n, obs_dim], or uint8 rows with obs_format 'u8' / 'hits') to an int32 action tensor [n]; observations and actions
        never leave the device and the host is out of the loop (tests/train.py:122-135 is the use case).  Returns
        (graph, record): `graph.replay()` advances every env by n_steps; `record` holds the tensors the graph fills
        (actions [n_steps, n], reward_sum, cost_sum, done_count, and the handle's obs/reward/done/... of the last step)."""
        dev = self.device
        rec = {'actions': torch.zeros((n_steps, self.n), dtype=torch.int32, device=dev),
               'reward_sum': torch.zeros(self.n, dtype=torch.float32, device=dev),
               'cost_sum': torch.zeros(self.n, dtype=torch.float32, device=dev),
               'done_count': torch.zeros(self.n, dtype=torch.int32, device=dev)}
        stream = torch.cuda.Stream(dev)
        stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(stream):
            for _ in range(2):                                  # warm-up outside the capture (lazy torch initialisation)
                a = policy(self.obs).to(torch.int32)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=stream):
                rec['reward_sum'].zero_(); rec['cost_sum'].zero_(); rec['done_count'].zero_()
                for t in range(n_steps):
                    rec['actions'][t].copy_(policy(self.obs))
                    self.step(rec['actions'][t], auto_reset, max_episode_steps)
                    rec['reward_sum'] += self.reward
                    rec['cost_sum'] += self.step_cost
                    rec['done_count'] += self.done
        torch.cuda.current_stream(dev).wait_stream(stream)
        rec.update(obs=self.obs, reward=self.reward, done=self.done, step_cost=self.step_cost, result=self.result)
        return graph, rec

    def enable_messages(self, on=True):
        """Make every following step also write info['message'] codes (uint16 per env) into self.msg."""
        if on and getattr(self, 'msg', None) is None:
            self.msg = torch.zeros(self.n, dtype=torch.int16, device=self.device)
        capi.check(self.lib, self.lib.ngw_set_message_buffer(self._h, _ptr(self.msg) if on else None))
        if not on:
            self.msg = None
        return self.msg

    def enable_episode_end(self, on=True):
        """Make every following one-step call (step, step_host, StepGroup) also write self.truncated (uint8 [n]: 1 where
        the step hit max_episode_steps and the env did not end the episode itself, gym's info['TimeLimit.truncated']) and,
        for the envs its auto-reset regenerated, self.final_obs (rows like self.obs: the observation the step produced,
        before the reset observation replaced it).  on=False switches both off and releases them."""
        if on and getattr(self, 'truncated', None) is None:
            self.truncated = torch.zeros(self.n, dtype=torch.uint8, device=self.device)
            self.final_obs = torch.zeros_like(self.obs)
        if not on:
            self.truncated = self.final_obs = None
        capi.check(self.lib, self.lib.ngw_set_episode_end_buffers(
            self._h, _ptr(self.truncated), _ptr(self.final_obs) if self.obs_dim else None))
        return self.truncated, self.final_obs

    def observe(self):
        if self.obs_dim:
            capi.check(self.lib, self.lib.ngw_observe(self._h, _ptr(self.obs), self._stream()))
        return self.obs

    def _host_buffers(self):
        if self._host is None:
            d = max(self.obs_dim, 1)
            n = self.n
            # ONE pinned block mirroring the library's device staging (observation rows | pad to 16 | reward | step_cost |
            # done | result): ngw_step_host then brings a whole step back with a single device-to-host copy
            row = max(self.obs_row_bytes, 4) if self.obs_format != 'i32' else 4 * d
            obs_bytes = n * row if self.obs_dim else 0
            off = (obs_bytes + 15) & ~15
            block = torch.zeros(off + 10 * n + 64, dtype=torch.uint8).pin_memory()
            small = block[off:off + 10 * n]
            if self.obs_dim == 0:
                host_obs = torch.zeros((n, 1), dtype=torch.int32)
            elif self.obs_format != 'i32':
                host_obs = block[:obs_bytes].view(n, row)
            else:
                host_obs = block[:obs_bytes].view(torch.int32).view(n, d)
            self._host = {
                'actions': torch.zeros(n, dtype=torch.int32).pin_memory(),
                'block': block,
                'obs': host_obs,
                'small': small,
                'reward': small[:4 * n].view(torch.float32),
                'step_cost': small[4 * n:8 * n].view(torch.float32),
                'done': small[8 * n:9 * n],
                'result': small[9 * n:10 * n],
            }
        return self._host

    def step_host(self, actions, auto_reset=False, max_episode_steps=0):
        """Host path: numpy in, numpy views of pinned buffers out; H2D + step + D2H inside libngw_b200."""
        hb = self._host_buffers()
        hb['actions'].numpy()[:] = np.asarray(actions, dtype=np.int32).reshape(self.n)
        capi.check(self.lib, self.lib.ngw_step_host(
            self._h, _ptr(hb['actions']), _ptr(hb['obs']) if self.obs_dim else None, _ptr(hb['reward']),
            _ptr(hb['done']), _ptr(hb['step_cost']), _ptr(hb['result']), int(bool(auto_reset)),
            int(max_episode_steps)))
        return (hb['obs'].numpy(), hb['reward'].numpy(), hb['done'].numpy(), hb['step_cost'].numpy(),
                hb['result'].numpy())

    def step_host_begin(self, actions, auto_reset=False, max_episode_steps=0):
        """Enqueue H2D + step + D2H on the handle's own stream and return at once (pipelining over several batches);
        `step_host_end()` blocks until the pinned output buffers are valid and returns them."""
        hb = self._host_buffers()
        hb['actions'].numpy()[:] = np.asarray(actions, dtype=np.int32).reshape(self.n)
        capi.check(self.lib, self.lib.ngw_step_host_begin(
            self._h, _ptr(hb['actions']), _ptr(hb['obs']) if self.obs_dim else None, _ptr(hb['reward']),
            _ptr(hb['done']), _ptr(hb['step_cost']), _ptr(hb['result']), int(bool(auto_reset)),
            int(max_episode_steps)))

    def step_host_end(self):
        capi.check(self.lib, self.lib.ngw_step_host_end(self._h))
        hb = self._host
        return (hb['obs'].numpy(), hb['reward'].numpy(), hb['done'].numpy(), hb['step_cost'].numpy(),
                hb['result'].numpy())

    def stats_allreduce(self, reset=False):
        """Job-wide episode statistics: the handle's counters summed over all ranks (NCCL when torch.distributed is up)."""
        from .sharding import allreduce_stats
        return allreduce_stats(self.stats(reset).clone())

    def stats(self, reset=False):
        """float64[8] on device, order = opcodes.STAT_NAMES; all-reduce it with NCCL for the job total."""
        capi.check(self.lib, self.lib.ngw_stats(self._h, _ptr(self._stats), int(bool(reset)), self._stream()))
        return self._stats

    def launch_count(self):
        return int(self.lib.ngw_launch_count(self._h))

    def concurrent_launch_count(self):
        """One-step launches that ran overlapped with their predecessor (another handle's step, proven adjacent in a
        stream capture; see include/ngw.h)."""
        return int(self.lib.ngw_concurrent_launch_count(self._h))


class StepGroup(object):
    """ngw_step_many over a fixed list of BatchHandles (env pools): one library call steps them all, in order, on the
    current stream; the launches of different handles overlap (eager mode too).  The ngw_step_item array is built once."""

    def __init__(self, handles):
        import ctypes as C
        assert len(handles) > 0
        self.handles = list(handles)
        self._arr = (capi.StepItem * len(self.handles))()
        for i, h in enumerate(self.handles):
            it = self._arr[i]
            it.h = h._h
            it.obs = _ptr(h.obs) if h.obs_dim else None
            it.reward, it.done = _ptr(h.reward), _ptr(h.done)
            it.step_cost, it.result = _ptr(h.step_cost), _ptr(h.result)
        self._arr_p = C.cast(self._arr, C.c_void_p)
        self._outs = [(h.obs, h.reward, h.done, h.step_cost, h.result) for h in self.handles]

    def step(self, actions, auto_reset=False, max_episode_steps=0):
        """`actions`: one contiguous int32 CUDA tensor per handle.  Returns the handles' output tuples (reused tensors)."""
        hs = self.handles
        assert len(actions) == len(hs)
        keep = []
        for i, a in enumerate(actions):
            if a.dtype != torch.int32 or not a.is_cuda or not a.is_contiguous():
                a = a.to(device=hs[i].device, dtype=torch.int32).contiguous()
                keep.append(a)
            self._arr[i].actions = a.data_ptr()
        h0 = hs[0]
        capi.check(h0.lib, h0.lib.ngw_step_many(self._arr_p, len(hs), int(bool(auto_reset)), int(max_episode_steps),
                                                h0._stream()))
        return self._outs


def step_many(handles, actions, auto_reset=False, max_episode_steps=0):
    """One-off form of StepGroup(handles).step(actions)."""
    return StepGroup(handles).step(actions, auto_reset=auto_reset, max_episode_steps=max_episode_steps)


_MSG_FIXED = {0: '', 1: 'Block in path', 3: 'Block tree_tap placed', 5: 'Item not found in inventory',
              6: 'No tree_log near tree_tap', 7: 'No tree_tap found', 8: 'No wool found',
              10: 'Need to be in front of crafting_table', 14: 'Cannot break due to fence restriction',
              15: 'You died due to fire_wall'}


def decode_message(code, compiled):
    """16-bit message code (enum ngw_msg | arg << 5) -> the reference's info['message'] string."""
    code = int(code) & 0xFFFF
    kind, arg = code & 31, code >> 5
    if kind in _MSG_FIXED:
        return _MSG_FIXED[kind]
    names = compiled.item_names
    if kind == 2:
        return "Cannot break " + names[arg]                                   # pogostick_v1_env.py:292
    if kind == 4:
        return "Block " + names[arg] + " already exists when trying to place block"   # pogostick_v1_env.py:309
    if kind == 9:                                                              # pogostick_v1_env.py:432-440
        rec = compiled.c.recipes[arg & 7]
        parts = [str(rec.in_qty[i]) + ' ' + names[rec.in_item[i]] for i in range(rec.n_inputs) if (arg >> 3) & (1 << i)]
        return "Missing items: " + ', '.join(parts)
    if kind == 11:
        return "Crafted " + names[arg]                                         # pogostick_v1_env.py:472
    if kind == 12:
        return "Cannot break without " + names[arg] + " selected"              # novelty_wrappers.py:501
    if kind == 13:
        return "Cannot chop " + names[arg]                                     # novelty_wrappers.py:1307
    return ''


class LazyInfo(object):
    """info of a batched step: tensors; the reference's strings are formatted only when 'message' is asked for.
    `episode_end` (truncated, terminal observation rows), when given, adds 'TimeLimit.truncated' and
    'terminal_observation'; a host-path step passes a callable that fetches them on first access."""

    def __init__(self, result, step_cost, msg=None, compiled=None, cfg_ids=None, flags=None, episode_end=None):
        self.result, self.step_cost = result, step_cost
        self._msg, self._compiled, self._cfg_ids, self._flags = msg, compiled, cfg_ids, flags
        self._episode_end = episode_end

    def _end(self):
        if callable(self._episode_end):
            self._episode_end = self._episode_end()
        return self._episode_end

    def __getitem__(self, key):
        if key == 'result':
            return self.result
        if key == 'step_cost':
            return self.step_cost
        if key == 'invalid':         # envs whose action id the chain rejects (the reference raises, wrappers.py:76)
            return None if self._flags is None else (self._flags & oc.ERR_INVALID_ACTION) != 0
        if key == 'message':
            if self._msg is None:
                return None      # message codes are off unless the env was made with messages=True
            codes = self._msg.cpu().numpy() if hasattr(self._msg, 'cpu') else self._msg
            if self._cfg_ids is None:
                return [decode_message(c, self._compiled[0]) for c in codes]
            return [decode_message(c, self._compiled[int(i)]) for c, i in zip(codes, self._cfg_ids)]
        if self._episode_end is not None and key == 'TimeLimit.truncated':
            return self._end()[0]
        if self._episode_end is not None and key == 'terminal_observation':
            return self._end()[1]
        raise KeyError(key)

    def __contains__(self, key):
        return key in self.keys()

    def get(self, key, default=None):
        return self[key] if key in self.keys() else default

    def keys(self):
        keys = ['result', 'step_cost', 'message', 'invalid']
        return keys + ['TimeLimit.truncated', 'terminal_observation'] if self._episode_end is not None else keys


def global_stream_reset(h, want_obs=True):
    """Reset env 0 of a numpy-stream handle from the process's global np.random and advance that stream by the draws the
    reset took, as the reference's reset() does: get_state -> load into env 0 -> reset -> export -> set_state (the cached
    Gaussian is kept)."""
    name, key, pos, has_gauss, cached = np.random.get_state()
    h.load_rng_state(np.asarray(key, np.uint32).reshape(1, 624), np.array([pos], np.int32))
    obs = h.reset(want_obs=want_obs)
    k, p = h.rng_state(0, 1)
    np.random.set_state((name, k[0].copy(), int(p[0]), has_gauss, cached))
    return obs


class ChainRuntime(object):
    """Drives one wrapper chain (one config) through a BatchHandle with the reference's return conventions."""

    def __init__(self, base):
        self.base = base
        self.handle = None
        self.compiled = None
        self._fingerprint = None
        self.auto_reset = base.auto_reset
        self.max_episode_steps = base.max_episode_steps
        self.messages = base.messages
        self.episode_end_info = getattr(base, 'episode_end_info', False)

    # ------------------------------------------------------------------
    def _ensure(self):
        cc = compile_chain(self.base._top)
        fp = cc.fingerprint()
        if self.handle is None or fp != self._fingerprint:
            if self.handle is not None:
                self.handle.close()
            self.compiled, self._fingerprint = cc, fp
            self.handle = BatchHandle([cc], self.base.num_envs, self.base.device, self.base.rng_seed,
                                      self.base.first_env_gid,
                                      obs_format='i32' if self.base.num_envs == 1 else self.base.obs_format,
                                      reset_rng=self.base.reset_rng)
            if self.single or self.messages:
                self.handle.enable_messages()
            if self.episode_end_info and not self.single:       # (the reference has no auto-reset: N == 1 is unchanged)
                self.handle.enable_episode_end()
        return self.handle

    def close(self):
        if self.handle is not None:
            self.handle.close()
            self.handle = None

    @property
    def single(self):
        return self.base.num_envs == 1


    @property
    def global_stream(self):
        """num_envs == 1 on the numpy stream: reset() draws from the process's global np.random, as the reference does."""
        return self.single and self.base.reset_rng == 'numpy'

    def dict_observation(self):
        h = self.handle
        names = self.compiled.item_names
        if self.single:                                 # the env's own live objects, as get_observation hands them out
            b = self.base
            self._sync_single()
            return {'map': b.map, 'agent_location': b.agent_location, 'agent_facing_id': b.agent_facing_id,
                    'inventory_items_quantity': b.inventory_items_quantity}
        return {'map': h.map, 'agent_location': h.pose[:, 0:2], 'agent_facing_id': h.pose[:, 2],
                'inventory_items_quantity': {n: h.inventory[:, i] for i, n in enumerate(names) if n in self.base.items}}

    def agent_map(self, view):
        h = self.handle
        side = 2 * view + 1
        out = torch.empty((h.n, side, side), dtype=torch.int8, device=h.device)
        capi.check(h.lib, h.lib.ngw_agent_map(h._h, _ptr(out), int(view), h._stream()))
        return out[0].cpu().numpy().astype(np.int64) if self.single else out

    def lidar_observation(self):
        obs = self.handle.observe()
        if self.handle.obs_format == 'i32':
            obs = obs[:, :self.compiled.obs_dim]
        return obs[0].cpu().numpy().astype(np.int64) if self.single else obs

    def _sync_single(self):
        """num_envs == 1: refresh the attribute mirrors reference scripts read (env.map, env.agent_location, ...)."""
        b, h = self.base, self.handle
        pose = h.pose[0].cpu().numpy()
        inv = h.inventory[0].cpu().numpy()
        names = self.compiled.item_names
        # like the reference, `map` and `inventory_items_quantity` are LIVE objects updated in place (Dict observations and
        # SaveTrajectories states alias them, pogostick_v1_env.py:222-226, wrappers.py:29-45)
        grid = h.map[0].cpu().numpy().astype(np.int64)
        if isinstance(b.map, np.ndarray) and b.map.shape == grid.shape:
            b.map[...] = grid
        else:
            b.map = grid
        b.agent_location = (int(pose[0]), int(pose[1]))
        b.agent_facing_id = int(pose[2])
        b.agent_facing_str = [k for k, v in b.direction_id.items() if v == b.agent_facing_id][0]
        quantities = {n: int(inv[i]) for i, n in enumerate(names) if n in b.items}
        if isinstance(b.inventory_items_quantity, dict) and set(b.inventory_items_quantity) == set(quantities):
            b.inventory_items_quantity.update(quantities)
        else:
            b.inventory_items_quantity = quantities
        b.selected_item = names[int(pose[3])] if pose[3] else ''
        dr, dc = {0: (-1, 0), 1: (1, 0), 2: (0, -1), 3: (0, 1)}[b.agent_facing_id]
        fr, fc = b.agent_location[0] + dr, b.agent_location[1] + dc
        b.block_in_front_location = (fr, fc)
        b.block_in_front_id = int(b.map[fr][fc])
        b.block_in_front_str = names[b.block_in_front_id]

    def _restore_from(self, src_env):
        """The `env=` branch of reset (pogostick_v1_env.py:89-109, tests/test_multi_agent.py:55): tables and state are
        copied from another env (device-to-device through ngw_load_state); selected_item is NOT copied, as there."""
        import copy
        b, src = self.base, src_env.unwrapped
        src_rt = src._runtime
        if src_rt is None or src_rt.handle is None:
            raise RuntimeError("the env to restore from has not been reset yet")
        b.map_size = copy.deepcopy(src.map_size)
        b.items_id = copy.deepcopy(src.items_id)
        b.items_quantity = copy.deepcopy(src.items_quantity)
        h = self._ensure()
        sh = src_rt.handle
        if sh.n != h.n:
            raise ValueError("restore needs the same num_envs (%d vs %d)" % (sh.n, h.n))
        pose = sh.pose.clone()
        pose[:, 3] = h.pose[:, 3]
        n = min(sh.inv_stride, h.inv_stride)
        h.load_state(sh.map, pose, sh.inventory[:, :n].contiguous())
        obs = h.observe() if self.compiled.reset_returns == 'lidar' else None
        return h, obs

    def reset(self, **kwargs):
        if self.base.env is not None:
            print("RESTORING " + self.base.env_id + " ...")                # pogostick_v1_env.py:90
            h, obs = self._restore_from(self.base.env)
            cc = self.compiled
        else:
            h = self._ensure()
            cc = self.compiled
            if self.global_stream:
                obs = global_stream_reset(h, want_obs=(cc.reset_returns == 'lidar'))
            else:
                obs = h.reset(want_obs=(cc.reset_returns == 'lidar'))
        if self.single:
            torch.cuda.current_stream(h.device).synchronize()
            if int(h.error_flags[0].item()) & oc.ERR_PLACEMENT:
                raise AssertionError("Cannot place items, increase map size!")      # pogostick_v1_env.py:167
            b = self.base
            b.map, b.inventory_items_quantity = None, None         # an episode gets fresh live objects
            if b.env is None:                                       # pogostick_v1_env.py:119-127
                b.last_action, b.last_done, b.last_reward, b.last_step_cost, b.step_count = 'Forward', False, 0, 0, 0
            else:                                                   # restore: bookkeeping is copied, pogostick_v1_env.py:98-101
                src = b.env.unwrapped
                b.last_action, b.step_count, b.last_reward, b.last_done = src.last_action, src.step_count, src.last_reward, False
            self._sync_single()
        else:
            b = self.base
            b.map, b.agent_location, b.agent_facing_id = h.map, h.pose[:, 0:2], h.pose[:, 2]
            b.inventory_items_quantity = {n: h.inventory[:, i] for i, n in enumerate(cc.item_names) if n in b.items}
        if cc.reset_returns == 'lidar':
            o = obs if h.obs_format != 'i32' else obs[:, :cc.obs_dim]
            return o[0].cpu().numpy().astype(np.int64) if self.single else o
        return self.dict_observation()

    def step(self, action):
        if self.handle is None:
            self._ensure()
        h, cc = self.handle, self.compiled
        if self.single:
            a = torch.tensor([int(action)], dtype=torch.int32, device=h.device)
            obs, reward, done, cost, result = h.step(a)
            torch.cuda.current_stream(h.device).synchronize()
            flags = int(h.error_flags[0].item())
            if flags & oc.ERR_INVALID_ACTION:
                h.error_flags[0] = flags & ~oc.ERR_INVALID_ACTION
                why = cc.invalid_reasons.get(int(action), "Action ID " + str(action) + " is not valid")
                raise (ValueError if why.startswith('ValueError') else AssertionError)(why)
            self._sync_single()
            b = self.base
            b.step_count += 1
            b.last_reward, b.last_done = int(reward[0].item()), bool(done[0].item())
            # the float32 the kernel wrote, as the shortest decimal that round-trips it: 27.906975, 3600.0, ... — the very
            # doubles the reference reports
            b.last_step_cost = float(str(np.float32(cost[0].item())))
            # name of the action as the outermost wrapper sees it (pogostick_v1_env.py:236, wrappers.py:78)
            top = b._top
            ids = getattr(top, 'limited_actions_id', None) or top.actions_id
            for name, aid in ids.items():
                if aid == int(action):
                    b.last_action = name
                    break
            info = {'result': bool(result[0].item()), 'step_cost': b.last_step_cost,
                    'message': decode_message(h.msg[0].item(), cc)}
            o = (obs[0, :cc.obs_dim].cpu().numpy().astype(np.int64) if cc.obs_dim else self.dict_observation())
            return o, b.last_reward, b.last_done, info
        lidar_cols = slice(None) if h.obs_format != 'i32' else slice(0, cc.obs_dim)    # narrow rows: see BatchHandle.split_obs
        if isinstance(action, torch.Tensor) and action.is_cuda:
            obs, reward, done, cost, result = h.step(action, self.auto_reset, self.max_episode_steps)
            self._check_actions(action)
            o = obs[:, lidar_cols] if cc.obs_dim else self.dict_observation()
            end = None
            if self.episode_end_info:
                end = (h.truncated.view(torch.bool), h.final_obs[:, lidar_cols] if cc.obs_dim else None)
            return o, reward, done.view(torch.bool), LazyInfo(result.view(torch.bool), cost, getattr(h, 'msg', None), [cc],
                                                              flags=h.error_flags, episode_end=end)
        obs, reward, done, cost, result = h.step_host(action, self.auto_reset, self.max_episode_steps)
        self._check_actions(action)
        o = obs[:, lidar_cols] if cc.obs_dim else self.dict_observation()
        end = None
        if self.episode_end_info:
            def end():                          # the step's device buffers, fetched on access
                trunc = h.truncated.cpu().numpy().view(np.bool_)
                return trunc, (h.final_obs[:, lidar_cols].cpu().numpy() if cc.obs_dim else None)
        # the message codes sit in the handle's device buffer, complete once step_host returned; decoded on access
        return o, reward, done.view(np.bool_), LazyInfo(result.view(np.bool_), cost, getattr(h, 'msg', None), [cc],
                                                        flags=h.error_flags, episode_end=end)

    def _check_actions(self, action):
        """strict_actions: raise what the reference raises as soon as one env of the batch got a rejected id."""
        if not self.base.strict_actions:
            return
        h, cc = self.handle, self.compiled
        bad = torch.nonzero((h.error_flags & oc.ERR_INVALID_ACTION) != 0)
        if bad.numel() == 0:
            return
        i = int(bad[0].item())
        h.error_flags.bitwise_and_(~oc.ERR_INVALID_ACTION)
        a = int(action[i].item()) if hasattr(action[i], 'item') else int(action[i])
        why = cc.invalid_reasons.get(a, "Action ID " + str(a) + " is not valid")
        raise (ValueError if why.startswith('ValueError') else AssertionError)("env %d of %d: %s" % (i, int(bad.numel()), why))


class MixedBatch(object):
    """Several wrapper chains (configs) in one batch: env i runs config cfg_id[i] — one launch per step."""

    def __init__(self, tops, num_envs, cfg_id=None, device=None, seed=0, first_env_gid=0, assignment='interleaved',
                 reset_rng='philox'):
        self.compiled = [compile_chain(t) for t in tops]
        n_cfg = len(self.compiled)
        if cfg_id is None:
            idx = np.arange(num_envs, dtype=np.int64)
            gid = idx + int(first_env_gid)
            cfg_id = (gid % n_cfg) if assignment == 'interleaved' else np.minimum(idx * n_cfg // num_envs, n_cfg - 1)
        self.cfg_id_host = np.asarray(cfg_id, dtype=np.int32)
        self.handle = BatchHandle(self.compiled, num_envs, device, seed, first_env_gid, cfg_id=self.cfg_id_host,
                                  reset_rng=reset_rng)
        self.n_actions = np.array([cc.c.n_actions for cc in self.compiled], dtype=np.int32)

    def reset(self, mask=None):
        return self.handle.reset(mask)

    def step(self, actions, auto_reset=False, max_episode_steps=0):
        return self.handle.step(actions, auto_reset, max_episode_steps)

    def close(self):
        self.handle.close()
