"""Batched multi-agent env (mirrors gridworld/multiagent_env.py:20-230).

``MultiAgentEnv(**env_config)`` takes the reference's config dict unchanged
(``common_config`` / ``pf_config`` / ``agents`` with ``cls`` objects from this
package) plus ``num_envs``.  The constructor is the *spec compiler*: it walks the
agent tree, packs parameters, per-event exogenous tables and the compiled feeder
into the structure-of-arrays tables of ``include/pgw.h`` and creates the device
handle.  ``reset``/``step`` then run entirely on the GPU:

  * ``num_envs == 1``: the reference's dict API (obs / reward / done / meta dicts
    keyed by agent and component names);
  * any ``num_envs``: ``reset_batch`` / ``step_batch`` on device tensors laid out
    ``[rows, num_envs]`` (env index fastest), and ``step_host`` / ``reset_host`` on
    pinned host arrays (the end-to-end path).

``io_dtype="float32"`` makes the actions and observations of the batched and host-buffer
calls float32 (the dtype of a policy network's inputs and outputs).  The simulation itself
stays float64: actions are widened where the kernels read them, observations are computed
in float64 and rounded to nearest when stored.  Rewards, done flags, initial SOCs and all
state keep their types.  The dict API keeps the reference's float64 contract.

Deviations from the reference, all deliberate: ``history`` is only recorded when
``record_history=True``; overriding ``get_external_obs_vars`` is rejected (the grid
variables are assembled on the device with the reference's one-step lag).  The
``meta`` dicts of ``step`` are rebuilt from the device state (``_step_meta``; the
batched form is ``meta_batch``).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional

import numpy as np
import pandas as pd

from powergridworld_b200 import _native as N
from powergridworld_b200.base import ComponentEnv, MultiComponentEnv
from powergridworld_b200.distribution_system.opendss import ZBusSolver
from powergridworld_b200.distribution_system.powerflow import PowerFlowSolver


def _torch():
    import torch
    return torch


class SpecBuilder:
    """Collects component descriptors, parameter blocks and per-event table writers."""

    def __init__(self, nl: int):
        self.header = 2 + 2 * nl          # done, reserved, base kW[nl], base kvar[nl]
        self.comps: List[N.Component] = []
        self.objs: List[ComponentEnv] = []
        self.dpar: List[float] = []
        self.ipar: List[int] = []
        self.sd_rows = self.si_rows = self.act_dim = self.obs_dim = 0
        self.dwidth = self.header
        self.iwidth = 0
        self.dwriters, self.iwriters = [], []
        self.storages: List[ComponentEnv] = []
        self.needs_grid = False
        self.max_events = np.inf

    def next_storage_ordinal(self, obj) -> int:
        self.storages.append(obj)
        return len(self.storages) - 1

    def add_component(self, obj, ctype, agent_index, flags=0, dpar=(), ipar=(), sd_rows=0,
                      si_rows=0, dtab_width=0, dtab_fn=None, itab_width=0, itab_fn=None,
                      needs_grid=False, max_events=None):
        c = N.Component()
        c.type, c.agent, c.flags = ctype, agent_index, flags
        c.act_off, c.obs_off, c.obs_dim = self.act_dim, self.obs_dim, obj._obs_dim
        c.sd_off, c.si_off = self.sd_rows, self.si_rows
        c.dtab_off, c.itab_off = self.dwidth, self.iwidth
        c.dpar_off, c.ipar_off = len(self.dpar), len(self.ipar)
        self.dpar += [float(x) for x in dpar]
        self.ipar += [int(x) for x in ipar]
        self.act_dim += obj._act_dim
        self.obs_dim += obj._obs_dim
        self.sd_rows += sd_rows
        self.si_rows += si_rows
        if dtab_width:
            self.dwriters.append((self.dwidth, dtab_width, dtab_fn))
            self.dwidth += dtab_width
        if itab_width:
            self.iwriters.append((self.iwidth, itab_width, itab_fn))
            self.iwidth += itab_width
        self.needs_grid |= bool(needs_grid)
        if max_events is not None:
            self.max_events = min(self.max_events, max_events)
        obj._slot = {"act": (c.act_off, obj._act_dim), "obs": (c.obs_off, obj._obs_dim),
                     "sd": (c.sd_off, sd_rows), "si": (c.si_off, si_rows),
                     "dpar": (c.dpar_off, len(dpar)), "ipar": (c.ipar_off, len(ipar)),
                     "dtab": (c.dtab_off, dtab_width), "itab": (c.itab_off, itab_width)}
        self.comps.append(c)
        self.objs.append(obj)


class _MetaCtx:
    """What a component's ``_meta`` hook reads to rebuild the reference's step meta: rows of the
    double state and of the delivered observation (NumPy scalars for one env, ``[E]`` tensors
    for a batch), the host copy of the step's event row, and the lagged grid variables the
    step's observations were built from."""

    def __init__(self, env, agent_index, sd, obs, event, lag, batch):
        self.env, self.agent, self._sd, self._obs = env, agent_index, sd, obs
        self.event, self.lag, self.batch = event, lag, batch
        self._si = None

    def si(self, row):
        """Row of the uint32 state (fetched on first use: only the EV station's meta reads it)."""
        if self._si is None:
            si = self.env.get_field(N.FIELD_STATE_I)
            self._si = si if self.batch else si[:, 0].cpu().numpy()
        return self._si[row]

    def sd(self, row):
        return self._sd[row]

    def obs(self, row):
        return self._obs[row]

    def dtab(self, col):
        return float(self.env._dtab[self.event, col])

    def scalar(self, v):
        return v if self.batch else np.float64(v)

    def vector(self, items):
        return _torch().stack(list(items)) if self.batch else np.array(items, dtype=np.float64)

    def grid(self, key):
        if self.lag is None:
            return None
        if key == "bus_voltage":
            return self.lag["vbus"][self.agent]
        return self.lag["vmin" if key == "min_voltage" else "vmax"]


try:                                                   # multiagent_env.py:13-17: an RLlib env when ray is there
    from ray.rllib.env.multi_agent_env import MultiAgentEnv as _Env
except ImportError:
    _Env = object


class MultiAgentEnv(_Env):
    """gridworld/multiagent_env.py:20-230 over ``num_envs`` instances on one GPU."""

    # grid-level reward hook; subclasses set these (see CoordinatedMultiBuildingControlEnv)
    _penalty = None     # (vlo, vhi, unit_penalty) or None

    def __init__(self, common_config: dict = {}, pf_config: dict = None, agents: list = None,
                 max_episode_steps: int = None, rescale_spaces: bool = True,
                 num_envs: int = 1, device=None, record_history: bool = False,
                 pf_tol: float = None, pf_max_iter: int = None, pf_kernel: str = "fp64",
                 io_dtype: str = "float64", _dry_run: bool = False, **kwargs):
        if type(self).get_external_obs_vars is not MultiAgentEnv.get_external_obs_vars:
            raise NotImplementedError(
                "overriding get_external_obs_vars is not supported: grid variables are "
                "assembled on the device (no CPU fallback)")
        if _Env is not object:
            super().__init__()
        self.common_config = common_config
        self.rescale_spaces = rescale_spaces
        assert agents is not None and len(agents) > 0, "need at least one agent!"
        self.start_time = pd.Timestamp(common_config["start_time"])
        self.end_time = pd.Timestamp(common_config["end_time"])
        self.control_timedelta = common_config["control_timedelta"]
        self.pf_config = pf_config
        self.max_episode_steps = max_episode_steps if max_episode_steps is not None else np.inf
        self.num_envs = int(num_envs)
        if io_dtype not in self._IO_DTYPES:
            raise ValueError(f"io_dtype must be one of {list(self._IO_DTYPES)}, not {io_dtype!r}")
        self.io_dtype = io_dtype
        self.record_history = record_history
        self.episode_step = None
        self.history = None

        # ---- agents (same constructor call as multiagent_env.py:57-70)
        self.agents: List[ComponentEnv] = []
        for a in agents:
            cfg = {k: v for k, v in a["config"].items() if k != "name"}
            self.agents.append(a["cls"](name=a["name"], **cfg, **self.common_config))
        self.agent_name_bus_map = {a["name"]: a["bus"] for a in agents}
        self.agent_names = [a.name for a in self.agents]
        assert len(set(self.agent_names)) == len(agents), "all agents need unique names"
        for ag in self.agents:
            if not isinstance(ag, ComponentEnv):
                raise TypeError(f"agent class {type(ag).__name__} is not a powergridworld_b200 "
                                "component: arbitrary Python agents cannot run on the device")

        # ---- power-flow plugin
        self.pf_solver: Optional[ZBusSolver] = None
        if pf_config and (pf_config.get("cls") is not None or "instance" in pf_config):
            solver = pf_config["instance"] if "instance" in pf_config \
                else pf_config["cls"](**pf_config.get("config", {}))
            if not isinstance(solver, ZBusSolver):
                raise TypeError("pf_config['cls'] must be powergridworld_b200's OpenDSSSolver/"
                                "ZBusSolver: a Python PowerFlowSolver cannot run on the device")
            if pf_tol is not None:
                solver.tol = pf_tol
            if pf_max_iter is not None:
                solver.max_iter = pf_max_iter
            if not getattr(self, "_is_solver_host", False):
                solver._env = self
            self.pf_solver = solver

        self.observation_space = {a.name: a.observation_space for a in self.agents}
        self.action_space = {a.name: a.action_space for a in self.agents}

        self._compile()
        self._h = None
        if pf_kernel not in self._PF_KERNELS:
            raise ValueError(f"pf_kernel must be one of {sorted(self._PF_KERNELS)}")
        if not _dry_run:        # tests inspect the compiled tables without a GPU
            self._open(device)
            if self.pf_solver is not None and pf_kernel != "fp64":
                self._select_pf_kernel(pf_kernel)

    # power-flow kernels (PGW_OPT_PF_KERNEL): "fp64" = FP64 SIMT fixed point (default, agrees with
    # the oracle to ~1e-9 p.u.), "tc" / "tc2" = tcgen05 solvers (1e-6 p.u., what bench.py runs),
    # "auto" = tc2 when the feeder fits it (<= 88 load branches), else fp64
    _PF_KERNELS = {"fp64": 0, "tc": 1, "tc2": 2, "auto": 2}
    # element type of the actions / observations of the batched and host-buffer API
    _IO_DTYPES = ("float64", "float32")

    def _select_pf_kernel(self, name: str):
        try:
            self.set_option(N.OPT_PF_KERNEL, self._PF_KERNELS[name])
        except N.NativeError:
            if name != "auto":
                raise
            self.set_option(N.OPT_PF_KERNEL, 0)

    @property
    def time(self):
        """Simulation time of the current step (multiagent_env.py:129, :160), derived from the
        step counter so that the hot loop does no pandas arithmetic."""
        if self.episode_step is None:
            return None
        return self.start_time + self.episode_step * self.control_timedelta

    # ------------------------------------------------------------------ spec compiler
    def _compile(self):
        feeder = self.pf_solver.feeder if self.pf_solver else None
        nl = feeder.nl if feeder else 0
        b = SpecBuilder(nl)
        agent_recs = (N.Agent * len(self.agents))()
        for ai, ag in enumerate(self.agents):
            begin = len(b.comps)
            for comp in getattr(ag, "envs", [ag]):
                comp._num_envs = self.num_envs          # randomised stations: one roster per env instance
            ag._emit(b, ai, standalone=not isinstance(ag, MultiComponentEnv))
            rec = agent_recs[ai]
            rec.comp_begin, rec.comp_end = begin, len(b.comps)
            rec.load_slot, rec.bus_node = -1, -1
            if feeder is not None:
                bus = self.agent_name_bus_map[ag.name]
                try:
                    rec.load_slot = feeder.load_index(bus)
                except ValueError:
                    # the reference only walks the feeder's own load names (opendss.py:115-129):
                    # power reported under any other name silently never reaches the circuit
                    import warnings
                    warnings.warn(f"agent {ag.name!r}: the feeder has no load named {bus!r} "
                                  f"(loads: {', '.join(feeder.load_names)}); its power is ignored "
                                  "by the power flow, as in the reference")
                    rec.load_slot = -1
                if rec.load_slot >= 0 and feeder.load_model[rec.load_slot] != 1:
                    # the reference only manipulates Model=1 (PQ) loads (opendss.py:54-77,
                    # :115-129): power of an agent on any other load never reaches the feeder
                    import warnings
                    warnings.warn(f"agent {ag.name!r} sits on load {bus!r} whose model is not 1: "
                                  "its power is ignored by the power flow, as in the reference")
                    rec.load_slot = -1
                node = self.pf_solver.node_for_bus_name(str(bus))
                if "bus_voltage" in ag.obs_labels and node is None:
                    raise ValueError(f"agent {ag.name!r} observes bus_voltage but {bus!r} is a "
                                     "three-phase bus name (the reference yields a list there)")
                rec.bus_node = node if node is not None else -1
        if b.needs_grid and feeder is None:
            raise ValueError("a component observes grid voltages but pf_config is empty")

        # episode length: first step count at which anything reports done (:199-207)
        span = (self.end_time - self.start_time) / self.control_timedelta
        limits = [a._terminal_after() for a in self.agents] + \
                 [self.max_episode_steps - 1, int(np.ceil(span)), b.max_events]
        limits = [x for x in limits if x is not None and x >= 1]
        L = int(min(limits))
        self.episode_length = L
        n_events = L + 1

        dstride = b.dwidth + (b.dwidth % 2)
        istride = (b.iwidth + 3) // 4 * 4
        dtab = np.zeros((n_events, dstride), dtype=np.float64)
        itab = np.zeros((n_events, max(istride, 0)), dtype=np.int32)
        for r in range(n_events):
            dtab[r, 0] = 1.0 if r == L else 0.0
            if feeder is not None:
                kw, kvar = self.pf_solver.base_load_at(self.start_time + r * self.control_timedelta)
                dtab[r, 2:2 + nl] = kw
                dtab[r, 2 + nl:2 + 2 * nl] = kvar
            for off, width, fn in b.dwriters:
                dtab[r, off:off + width] = fn(r)
            for off, width, fn in b.iwriters:
                itab[r, off:off + width] = fn(r)

        self._b = b
        self._agent_recs = agent_recs
        self._dpar = np.asarray(b.dpar if b.dpar else [0.0], dtype=np.float64)
        self._dtab, self._itab = dtab, itab
        self._dstride, self._istride = dstride, istride
        self.act_dim, self.obs_dim = b.act_dim, b.obs_dim
        self.num_storage = len(b.storages)
        # name-keyed layout of the flat action / observation rows
        self.act_slices, self.obs_slices = {}, {}
        for ag in self.agents:
            if isinstance(ag, MultiComponentEnv):
                self.act_slices[ag.name] = {e.name: e._slot["act"] for e in ag.envs}
                self.obs_slices[ag.name] = {e.name: e._slot["obs"] for e in ag.envs}
            else:
                self.act_slices[ag.name] = ag._slot["act"]
                self.obs_slices[ag.name] = ag._slot["obs"]

    def _build_spec(self):
        """The pgw_spec of the compiled scenario + the objects that keep its pointers alive."""
        b = self._b
        spec = N.Spec()
        spec.abi_version = N.ABI_VERSION
        spec.num_envs, spec.num_agents, spec.num_components = self.num_envs, len(self.agents), len(b.comps)
        spec.act_dim, spec.obs_dim = b.act_dim, b.obs_dim
        spec.sd_rows, spec.si_rows = b.sd_rows, b.si_rows
        spec.num_storage = self.num_storage
        spec.num_events = self._dtab.shape[0]
        spec.dtab_stride, spec.itab_stride = self._dstride, self._istride
        comps = (N.Component * len(b.comps))(*b.comps)
        dpar = self._dpar
        ipar = np.asarray(b.ipar if b.ipar else [0], dtype=np.int32)
        spec.dpar_len, spec.ipar_len = len(b.dpar), len(b.ipar)
        dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
        ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
        spec.agents, spec.components = self._agent_recs, comps
        spec.dpar, spec.ipar = dp(dpar), ip(ipar)
        dtab = self._dtab = np.ascontiguousarray(self._dtab)
        itab = np.ascontiguousarray(self._itab if self._istride else np.zeros((1, 4), np.int32))
        if self._istride:
            self._itab = itab
        spec.dtab, spec.itab = dp(dtab), ip(itab)
        keep = [comps, dpar, ipar, dtab, itab]
        if self.pf_solver is not None:
            f = self.pf_solver.feeder
            fd = N.Feeder()
            fd.nb, fd.nn, fd.nl = f.nb, f.nn, f.nl
            fd.max_iter, fd.tol = self.pf_solver.max_iter, self.pf_solver.tol
            cplx = lambda a: np.ascontiguousarray(a, dtype=np.complex128).view(np.float64)
            arrs = dict(zbb=cplx(f.zbb), u0=cplx(f.u0), znb=cplx(f.znb), w=cplx(f.w),
                        share=np.ascontiguousarray(f.branch_share, dtype=np.float64),
                        vmin=np.ascontiguousarray(f.branch_vmin, dtype=np.float64),
                        vmax=np.ascontiguousarray(f.branch_vmax, dtype=np.float64),
                        bl=np.ascontiguousarray(f.branch_load, dtype=np.int32),
                        bm=np.ascontiguousarray(f.branch_model, dtype=np.int32))
            fd.zbb, fd.u0, fd.znb, fd.w = dp(arrs["zbb"]), dp(arrs["u0"]), dp(arrs["znb"]), dp(arrs["w"])
            fd.branch_share, fd.vminpu, fd.vmaxpu = dp(arrs["share"]), dp(arrs["vmin"]), dp(arrs["vmax"])
            fd.branch_load, fd.branch_model = ip(arrs["bl"]), ip(arrs["bm"])
            fd.penalty_node, fd.penalty_unit = -1, 0.0
            if self._penalty is not None:
                buses = set(self.agent_name_bus_map.values())
                assert len(buses) == 1, "In this example, all buildings should be on the same bus."
                node = self.pf_solver.node_for_bus_name(str(list(buses)[0]))
                if node is None:
                    raise ValueError("the shared-penalty bus must be a single-phase load name")
                fd.penalty_node = node
                fd.penalty_vlo, fd.penalty_vhi, fd.penalty_unit = self._penalty
            spec.feeder = C.pointer(fd)
            keep += [fd, arrs]
        return spec, keep

    def _open(self, device):
        torch = _torch()
        if not torch.cuda.is_available():
            raise N.NativeError("powergridworld_b200 needs a CUDA device (B200, sm_100a); "
                                "there is no CPU fallback")
        self.device = torch.device(device if device is not None else
                                   f"cuda:{torch.cuda.current_device()}")
        lib = N.lib()
        spec, keep = self._build_spec()
        handle = C.c_void_p()
        with torch.cuda.device(self.device):
            N.check(lib.pgw_create(C.byref(spec), C.byref(handle)))
        self._h = handle
        self._lib = lib
        E, A = self.num_envs, len(self.agents)
        f64 = dict(dtype=torch.float64, device=self.device)
        io32 = self.io_dtype == "float32"
        self._io_torch = torch.float32 if io32 else torch.float64
        self._pgw_reset = lib.pgw_reset_f32 if io32 else lib.pgw_reset
        self._pgw_step = lib.pgw_step_f32 if io32 else lib.pgw_step
        self._pgw_reset_host = lib.pgw_reset_host_f32 if io32 else lib.pgw_reset_host
        self._pgw_step_host = lib.pgw_step_host_f32 if io32 else lib.pgw_step_host
        io = dict(dtype=self._io_torch, device=self.device)
        self.obs = torch.zeros((self.obs_dim, E), **io)
        self.rew = torch.zeros((A, E), **f64)
        self.done = torch.zeros((E,), dtype=torch.uint8, device=self.device)
        self._act = torch.zeros((self.act_dim, E), **io)
        self._act_shape = self._act.shape
        self._obs_ptr, self._rew_ptr = self.obs.data_ptr(), self.rew.data_ptr()
        self._done_ptr = self.done.data_ptr()
        self._pin = None
        self._host_step = None
        self._needs_reset = True
        self._lag = None
        self._dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()

    def close(self):
        if getattr(self, "_h", None):
            self._lib.pgw_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ hooks (reference API)
    def get_external_obs_vars(self, agent) -> dict:
        """multiagent_env.py:90-115, evaluated from the device state (E == 1)."""
        kw = {}
        if "bus_voltage" in agent.obs_labels:
            kw["bus_voltage"] = self.pf_solver.get_bus_voltage_by_name(
                self.agent_name_bus_map[agent.name])
        if "max_voltage" in agent.obs_labels:
            kw["max_voltage"] = max(list(self.voltages.values()))
        if "min_voltage" in agent.obs_labels:
            kw["min_voltage"] = min(list(self.voltages.values()))
        return kw

    def reward_transform(self, rew_dict) -> dict:
        return rew_dict

    def meta_transform(self, meta) -> dict:
        return meta

    @property
    def agent_dict(self) -> Dict[str, ComponentEnv]:
        return {a.name: a for a in self.agents}

    # ------------------------------------------------------------------ batched API
    def _stream(self):
        return C.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    def _randomised(self):
        return [o for o in self._b.objs if getattr(o, "randomize", False) and hasattr(o, "_retable")]

    def _rebuild_roster_tables(self):
        """Rewrite (host side, in place) the parameter and event columns of every randomised
        charging station from its current roster draw; widths never change."""
        n_events = self._dtab.shape[0]
        for o in self._randomised():
            dpar, dtab_fn, itab_fn = o._retable()
            off, n = o._slot["dpar"]
            assert len(dpar) == n
            self._dpar[off:off + n] = dpar
            doff, dw = o._slot["dtab"]
            ioff, iw = o._slot["itab"]
            for r in range(n_events):
                self._dtab[r, doff:doff + dw] = dtab_fn(r)
                if iw:
                    self._itab[r, ioff:ioff + iw] = itab_fn(r)

    def _reset_draws(self, init_storage):
        """Host-side randomness of a reset in the reference's order -- agents in turn, their
        components in turn (multiagent_env.py:131-137): a storage draws its initial SOC
        (energy_storage_env.py:82-84), an EVChargingEnv(randomize=True) its roster
        (ev_charging_env.py:154-157; NumPy's global RNG, shared by all envs of the batch).  New
        rosters are pushed to the device with pgw_update_tables before the reset kernel runs.
        Returns the [num_storage, E] initial SOCs (or ``init_storage`` when given)."""
        rand = self._randomised()
        draw_soc = self.num_storage and init_storage is None
        # the reference clips an explicit init_storage to the storage range but not the value it
        # draws itself (energy_storage_env.py:82-89): tell the reset kernel which one this is
        if self.num_storage and self._h is not None:
            self.set_option(N.OPT_CLIP_INIT_SOC, 0 if draw_soc else 1)
        self._soc_drawn = bool(draw_soc)
        if not rand:
            return self.draw_initial_storage() if draw_soc else init_storage
        soc = []
        for o in self._b.objs:
            if any(o is r for r in rand):
                o._draw_roster()
            elif draw_soc and any(o is s for s in self._b.storages):
                x = o.draw_initial_storage() if self.num_envs == 1 \
                    else o.draw_initial_storage(size=self.num_envs)
                soc.append(np.broadcast_to(np.asarray(x, dtype=np.float64), (self.num_envs,)))
        self._push_roster_tables()
        return np.stack(soc) if draw_soc else init_storage

    def _per_env_roster_rows(self):
        """[(field, first row, array [rows, E])] of the per-env rosters just drawn: window words into
        the uint32 state behind each station's charging-set words, initial energies into its
        double state (PGW_F_EV_PER_ENV)."""
        out = []
        for o in self._randomised():
            if getattr(o, "_per_env", False) and o._rows is not None:
                words, energy = o._per_env_rows()
                out.append((N.FIELD_STATE_I, o._slot["si"][0] + (o.num_vehicles + 31) // 32, words))
                out.append((N.FIELD_STATE_D, o._slot["sd"][0], energy))
        return out

    def _push_roster_tables(self):
        self._rebuild_roster_tables()
        if self._h is not None:
            torch = _torch()
            for field, row0, arr in self._per_env_roster_rows():
                t = torch.from_numpy(arr.view(np.int32) if arr.dtype == np.uint32 else arr).to(self.device)
                with torch.cuda.device(self.device):
                    N.check(self._lib.pgw_set_rows(self._h, field, row0, arr.shape[0],
                                                   C.c_void_p(t.data_ptr()), t.numel() * t.element_size(),
                                                   self._stream()))
                self._keep_rows = getattr(self, "_keep_rows", [])[-8:] + [t]   # alive until the copy ran
        if self._h is not None:
            dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
            with _torch().cuda.device(self.device):
                N.check(self._lib.pgw_update_tables(
                    self._h, dp(self._dpar), len(self._b.dpar), dp(self._dtab),
                    self._itab.ctypes.data_as(C.POINTER(C.c_int32)) if self._istride else None,
                    self._stream()))

    def draw_initial_storage(self) -> np.ndarray:
        """[num_storage, E] initial SOC drawn like the reference does on reset
        (energy_storage_env.py:82-84): one scalar truncnorm draw per storage in agent /
        component order for E == 1, a vectorised draw otherwise."""
        if self.num_storage == 0:
            return np.zeros((0, self.num_envs))
        if self.num_envs == 1:
            return np.array([[float(s.draw_initial_storage())] for s in self._b.storages])
        return np.stack([s.draw_initial_storage(size=self.num_envs) for s in self._b.storages])

    def reset_batch(self, init_storage=None):
        """Reset all envs; returns the observation tensor ``[obs_dim, E]`` (reused buffer)."""
        torch = _torch()
        soc_ptr = None
        init_storage = self._reset_draws(init_storage)
        if self.num_storage:
            if not isinstance(init_storage, torch.Tensor):
                init_storage = torch.as_tensor(np.ascontiguousarray(init_storage, dtype=np.float64))
            soc = init_storage.to(self.device, dtype=torch.float64).contiguous()
            if tuple(soc.shape) != (self.num_storage, self.num_envs):
                raise ValueError(f"init_storage must be [{self.num_storage}, {self.num_envs}]")
            self._soc = soc
            soc_ptr = C.c_void_p(soc.data_ptr())
        with torch.cuda.device(self.device):
            N.check(self._pgw_reset(self._h, soc_ptr, C.c_void_p(self.obs.data_ptr()), self._stream()))
        self.episode_step = 0
        self._needs_reset = False
        self._lag = None
        if self.record_history:
            self.history = {"timestamp": [], "voltage": [], "agent_power_p": []}
        return self.obs

    def step_batch(self, actions):
        """actions ``[act_dim, E]`` device tensor of the env's ``io_dtype`` -> (obs, rew, done,
        all_done).  The returned tensors are the env's own buffers, overwritten by the next call."""
        torch = _torch()
        if self._needs_reset:
            raise RuntimeError("call reset before step")
        if actions.dtype != self._io_torch or actions.shape != self._act_shape \
                or not actions.is_contiguous() or actions.device != self.device:
            raise ValueError(f"actions must be a contiguous {self.io_dtype} [{self.act_dim}, "
                             f"{self.num_envs}] tensor on {self.device}")
        stream = torch.cuda.current_stream(self.device).cuda_stream
        if torch.cuda.current_device() == self._dev_index:
            rc = self._pgw_step(self._h, actions.data_ptr(), self._obs_ptr, self._rew_ptr,
                                self._done_ptr, stream)
        else:                                       # the caller's current device is another GPU
            with torch.cuda.device(self.device):
                rc = self._pgw_step(self._h, actions.data_ptr(), self._obs_ptr, self._rew_ptr,
                                    self._done_ptr, stream)
        if rc:
            N.check(rc)
        self.episode_step += 1
        all_done = self.episode_step >= self.episode_length
        if all_done:
            self._needs_reset = True
        return self.obs, self.rew, self.done, all_done

    # ---- host-buffer (end-to-end) path
    def _pinned(self):
        if self._pin is None:
            torch = _torch()
            E, A = self.num_envs, len(self.agents)
            mk = lambda *s, dt=torch.float64: torch.zeros(s, dtype=dt).pin_memory()
            io = self._io_torch
            self._pin = dict(act=mk(self.act_dim, E, dt=io), obs=mk(self.obs_dim, E, dt=io), rew=mk(A, E),
                             done=mk(E, dt=torch.uint8), soc=mk(max(self.num_storage, 1), E))
        return self._pin

    def reset_host(self, init_storage=None) -> np.ndarray:
        torch = _torch()
        pin = self._pinned()
        soc_ptr = None
        init_storage = self._reset_draws(init_storage)
        if self.num_storage:
            pin["soc"][:self.num_storage].copy_(torch.as_tensor(np.asarray(init_storage, dtype=np.float64)))
            soc_ptr = C.c_void_p(pin["soc"].data_ptr())
        with torch.cuda.device(self.device):
            N.check(self._pgw_reset_host(self._h, soc_ptr, C.c_void_p(pin["obs"].data_ptr()),
                                         self._stream()))
        self.episode_step = 0
        self._needs_reset = False
        return pin["obs"].numpy()

    def step_host(self, actions: np.ndarray):
        """``actions`` host array [act_dim, E] -> (obs, rew, done) host arrays (pinned buffers
        owned by the env; obs in the env's ``io_dtype``).  Copies to and from the device are part
        of the call; actions that are not a page-locked array of the env's dtype are copied into
        the env's pinned action buffer first."""
        torch = _torch()
        if self._needs_reset:
            raise RuntimeError("call reset before step")
        hs = self._host_step
        if hs is None:
            pin = self._pinned()
            hs = self._host_step = {
                "ptrs": (pin["obs"].data_ptr(), pin["rew"].data_ptr(), pin["done"].data_ptr()),
                "out": (pin["obs"].numpy(), pin["rew"].numpy(), pin["done"].numpy()),
                "act": pin["act"], "act_ptr": pin["act"].data_ptr(),
                "numel": self.act_dim * self.num_envs, "pinned": {},
                "dev": self.device.index if self.device.index is not None else 0}
        if isinstance(actions, torch.Tensor):
            src = actions
        else:
            src = torch.from_numpy(np.ascontiguousarray(actions, dtype=self.io_dtype))
        if src.numel() != hs["numel"]:
            raise ValueError(f"actions must be [{self.act_dim}, {self.num_envs}]")
        act_ptr = src.data_ptr()
        ok = src.dtype == self._io_torch and src.is_contiguous()
        if ok:                                      # page-locked as well: the DMA reads it in place
            ok = hs["pinned"].get(act_ptr)          # (is_pinned() is a driver query: remembered)
            if ok is None:
                ok = bool(src.is_pinned())
                if len(hs["pinned"]) < 64:
                    hs["pinned"][act_ptr] = ok
        if not ok:
            hs["act"].copy_(src.reshape(self.act_dim, self.num_envs))
            act_ptr = hs["act_ptr"]
        po, pr, pd = hs["ptrs"]
        stream = torch.cuda.current_stream(self.device).cuda_stream
        if torch.cuda.current_device() == hs["dev"]:
            rc = self._pgw_step_host(self._h, act_ptr, po, pr, pd, stream)
        else:
            with torch.cuda.device(self.device):
                rc = self._pgw_step_host(self._h, act_ptr, po, pr, pd, stream)
        if rc:
            N.check(rc)
        self.episode_step += 1
        if self.episode_step >= self.episode_length:
            self._needs_reset = True
        return hs["out"]

    # ---- device state access
    def get_field(self, field: int):
        torch = _torch()
        E, A = self.num_envs, len(self.agents)
        nn = self.pf_solver.feeder.nn if self.pf_solver else 0
        shapes = {N.FIELD_STATE_D: ((self._b.sd_rows, E), torch.float64),
                  N.FIELD_STATE_I: ((self._b.si_rows, E), torch.int32),
                  N.FIELD_AGENT_P: ((A, E), torch.float64),
                  N.FIELD_VOLTAGES: ((nn, E), torch.float64),
                  N.FIELD_VMIN: ((E,), torch.float64), N.FIELD_VMAX: ((E,), torch.float64),
                  N.FIELD_VBUS: ((A, E), torch.float64),
                  N.FIELD_PF_ITERS: ((E,), torch.int32),
                  N.FIELD_EP_RETURN: ((A, E), torch.float64),
                  N.FIELD_PF_STATE: ((self._nbp(), E, 2), torch.float64)}
        shape, dt = shapes[field]
        out = torch.empty(shape, dtype=dt, device=self.device)
        if out.numel():
            with torch.cuda.device(self.device):
                N.check(self._lib.pgw_get(self._h, field, C.c_void_p(out.data_ptr()),
                                          out.numel() * out.element_size(), self._stream()))
        return out

    def _nbp(self):
        if self.pf_solver is None:
            return 0
        nb = self.pf_solver.feeder.nb
        return 16 if nb <= 16 else (nb + 31) // 32 * 32

    # ---- checkpoint / resume (SURVEY.md section 5: the reference has none at the env level)
    _STATE_FIELDS = (N.FIELD_STATE_D, N.FIELD_STATE_I, N.FIELD_AGENT_P, N.FIELD_VOLTAGES,
                     N.FIELD_VMIN, N.FIELD_VMAX, N.FIELD_VBUS, N.FIELD_PF_ITERS,
                     N.FIELD_EP_RETURN, N.FIELD_PF_STATE)

    def state_dict(self) -> dict:
        """Everything needed to resume the batch bit for bit: device fields + episode clock (the
        last observations in the env's ``io_dtype``)."""
        fields = {}
        for f in self._STATE_FIELDS:
            if self.pf_solver is None and f in (N.FIELD_VOLTAGES, N.FIELD_VMIN, N.FIELD_VMAX,
                                                N.FIELD_VBUS, N.FIELD_PF_ITERS, N.FIELD_PF_STATE):
                continue
            fields[f] = self.get_field(f).clone()
        state = {"fields": fields, "episode_step": self.episode_step, "obs": self.obs.clone(),
                 "needs_reset": self._needs_reset,
                 # resets taken so far: the first reset of a handle gives the state that the
                 # reference keeps across episodes its constructor value (house meta state,
                 # storage cost), later ones must not
                 "resets": int(self._lib.pgw_reset_count(self._h))}
        rand = self._randomised()
        if rand:                                    # the rosters drawn at the last reset
            state["rosters"] = [None if o._rows is None else np.array(o._rows) for o in rand]
        return state

    def load_state_dict(self, state: dict):
        torch = _torch()
        if state["obs"].dtype != self.obs.dtype:
            raise ValueError(f"checkpoint observations are {state['obs'].dtype}, this env's io_dtype is "
                             f"{self.io_dtype}: load it into an env with the io_dtype it was taken with")
        rand = self._randomised()
        if rand:
            rosters = state.get("rosters")
            if rosters is None or len(rosters) != len(rand):
                raise ValueError("checkpoint holds no rosters for the randomised charging stations")
            for o, rows in zip(rand, rosters):
                o._rows = None if rows is None else np.array(rows)
            self._push_roster_tables()
        for f, t in state["fields"].items():
            t = t.to(self.device).contiguous()
            if t.numel():
                N.check(self._lib.pgw_set(self._h, int(f), C.c_void_p(t.data_ptr()),
                                          t.numel() * t.element_size(), self._stream()))
        N.check(self._lib.pgw_set_reset_count(self._h, int(state.get("resets", 1))))
        if state["episode_step"] is None:           # checkpoint taken before the first reset
            self.episode_step, self._needs_reset = None, True
        else:
            N.check(self._lib.pgw_set_clock(self._h, int(state["episode_step"]), self._stream()))
            self.episode_step = int(state["episode_step"])
            self._needs_reset = bool(state["needs_reset"])
        self.obs.copy_(state["obs"])
        self._lag = None

    def stats(self):
        """Episode statistics reduced on the device: tensor[8], see include/pgw.h."""
        torch = _torch()
        out = torch.empty((N.NUM_STATS,), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            N.check(self._lib.pgw_stats(self._h, C.c_void_p(out.data_ptr()), self._stream()))
        return out

    def all_reduce_stats(self, group=None):
        """The single collective of the multi-GPU path (envs are sharded over ranks with no
        data-path exchange): the 8-entry statistics vector reduced over ``torch.distributed``."""
        return reduce_stats(self.stats(), group)

    def set_option(self, option: int, value: int):
        """Runtime options of the device handle (N.OPT_PF_KERNEL / OPT_WARM_START / OPT_GRAPHS)."""
        N.check(self._lib.pgw_set_option(self._h, int(option), int(value)))

    def set_kernel_timing(self, enabled: bool):
        N.check(self._lib.pgw_set_timing(self._h, int(bool(enabled))))

    def kernel_timing(self):
        """(component-kernel ms, power-flow-kernel ms, steps) since the last call."""
        out = (C.c_double * 3)()
        N.check(self._lib.pgw_get_timing(self._h, C.cast(out, C.c_void_p), self._stream()))
        return float(out[0]), float(out[1]), int(out[2])

    @property
    def launch_count(self) -> int:
        return int(self._lib.pgw_launch_count(self._h))

    # ---- stand-alone power flow (used by ZBusSolver.calculate_power_flow)
    def _solve_loads(self, kw: np.ndarray, kvar: np.ndarray):
        torch = _torch()
        f = self.pf_solver.feeder
        mk = lambda a: torch.as_tensor(np.array(                          # (a writable copy)
            np.broadcast_to(np.asarray(a, dtype=np.float64).reshape(f.nl, -1),
                            (f.nl, self.num_envs)), order="C")).to(self.device)
        tkw, tkvar = mk(kw), mk(kvar)
        with torch.cuda.device(self.device):
            N.check(self._lib.pgw_pf_solve(self._h, C.c_void_p(tkw.data_ptr()),
                                           C.c_void_p(tkvar.data_ptr()), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()

    def _voltage_dict(self, env_index: int = 0) -> Dict[str, float]:
        v = self.get_field(N.FIELD_VOLTAGES)[:, env_index].cpu().numpy()
        return {n: float(x) for n, x in zip(self.pf_solver.feeder.node_names, v)}

    @property
    def voltages(self):
        """{node: p.u. magnitude} of env 0 (the reference's ``self.voltages``)."""
        if self.pf_solver is None:
            return None
        return self._voltage_dict(0)

    # ------------------------------------------------------------------ dict API (E == 1)
    def _require_single(self):
        if self.num_envs != 1:
            raise RuntimeError("the dict API serves num_envs == 1; use reset_batch/step_batch")

    def _require_dict_api(self):
        self._require_single()
        if self.io_dtype != "float64":
            raise RuntimeError(f"the dict API keeps the reference's float64 observations and actions; "
                               f"with io_dtype={self.io_dtype!r} use reset_batch/step_batch or "
                               "reset_host/step_host")

    def _obs_dict(self, flat: np.ndarray) -> dict:
        out = {}
        for ag in self.agents:
            sl = self.obs_slices[ag.name]
            if isinstance(sl, dict):
                out[ag.name] = {k: flat[o:o + n].copy() for k, (o, n) in sl.items()}
            else:
                out[ag.name] = flat[sl[0]:sl[0] + sl[1]].copy()
        return out

    def flatten_action(self, action: dict) -> np.ndarray:
        flat = np.zeros(self.act_dim, dtype=np.float64)
        for ag in self.agents:
            sl = self.act_slices[ag.name]
            if isinstance(sl, dict):
                for k, (o, n) in sl.items():
                    flat[o:o + n] = np.asarray(action[ag.name][k], dtype=np.float64).reshape(-1)
            else:
                flat[sl[0]:sl[0] + sl[1]] = np.asarray(action[ag.name], dtype=np.float64).reshape(-1)
        return flat

    def reset(self, init_storage=None) -> Dict[str, any]:
        """multiagent_env.py:125-140.  ``init_storage`` ([num_storage] or [num_storage, 1])
        overrides the host RNG draw of the storages' initial SOC."""
        self._require_dict_api()
        if init_storage is not None:
            init_storage = np.asarray(init_storage, dtype=np.float64).reshape(self.num_storage, 1)
        obs = self.reset_batch(init_storage)
        self._lag = self._grid_snapshot()
        return self._obs_dict(obs[:, 0].cpu().numpy())

    # ---- step meta (the 4th return value of gridworld's step, multiagent_env.py:168, :210)
    def _grid_snapshot(self, batch=False):
        """The grid variables of the last solve, i.e. what the NEXT step's observations (and
        the building's state dict) are built from (multiagent_env.py:90-115, :167)."""
        if self.pf_solver is None:
            return None
        vb, mn, mx = (self.get_field(f) for f in (N.FIELD_VBUS, N.FIELD_VMIN, N.FIELD_VMAX))
        if batch:
            return {"vbus": vb, "vmin": mn, "vmax": mx}
        vb, mn, mx = vb[:, 0].cpu().numpy(), mn.cpu().numpy(), mx.cpu().numpy()
        return {"vbus": [np.float64(x) for x in vb], "vmin": np.float64(mn[0]), "vmax": np.float64(mx[0])}

    def _step_meta(self, flat_obs: np.ndarray) -> dict:
        """{agent: meta} of the step just taken, one env: every stock component's meta as the
        reference returns it (storage ``state_of_charge``, PV ``real_power``, the EV station's
        and the building's state dicts), rebuilt from the device state."""
        sd = self.get_field(N.FIELD_STATE_D)[:, 0].cpu().numpy() if self._b.sd_rows else np.zeros(0)
        meta = {}
        for i, a in enumerate(self.agents):
            meta[a.name] = a._meta(_MetaCtx(self, i, sd, flat_obs, self.episode_step, self._lag, False))
        self._lag = self._grid_snapshot()
        return meta

    def meta_batch(self, lag=None) -> dict:
        """The same metas for the whole batch: {agent: {component: {key: tensor[E] or float}}}
        from the current device state.  The building's grid entries need the grid variables the
        step OBSERVED: pass ``lag=env._grid_snapshot(batch=True)`` taken before the step."""
        sd = self.get_field(N.FIELD_STATE_D)
        return {a.name: a._meta(_MetaCtx(self, i, sd, self.obs, self.episode_step, lag, True))
                for i, a in enumerate(self.agents)}

    def get_obs(self) -> Dict[str, any]:
        self._require_dict_api()
        return self._obs_dict(self.obs[:, 0].cpu().numpy())

    def step(self, action: Dict[str, any]):
        """multiagent_env.py:151-212 for the single-env case."""
        self._require_dict_api()
        torch = _torch()
        self._act.copy_(torch.from_numpy(self.flatten_action(action)).reshape(self.act_dim, 1))
        obs, rew, _, all_done = self.step_batch(self._act)
        host = torch.cat([obs[:, 0], rew[:, 0]]).cpu().numpy()
        obs_d = self._obs_dict(host[:self.obs_dim])
        rew_d = {a.name: float(host[self.obs_dim + i]) for i, a in enumerate(self.agents)}
        dones = {a.name: bool(all_done) for a in self.agents}
        dones["__all__"] = bool(all_done)
        meta = self._step_meta(host[:self.obs_dim])
        p = self.get_field(N.FIELD_AGENT_P)[:, 0].cpu().numpy()
        for i, a in enumerate(self.agents):
            a._real_power = float(p[i])             # agent.real_power (base.py:51-55)
        if self.record_history:
            self.history["timestamp"].append(self.time)
            self.history["voltage"].append(self.voltages)
            self.history["agent_power_p"].append([float(x) for x in p])
        return obs_d, self.reward_transform(rew_d), dones, self.meta_transform(meta)


def reduce_stats(s, group=None):
    """All-reduce of a ``pgw_stats`` vector in ONE collective: SUM on the additive entries 0-5
    (env-steps, reward sum, episode returns, violation sum, non-converged count, iterations),
    MIN on entry 6 (min voltage), MAX on entry 7.  The extrema travel in rank-owned slots of the
    summed vector (every other rank contributes 0 there) and are reduced locally afterwards;
    identity when no process group is initialised."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return s
    torch = _torch()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    packed = torch.zeros(6 + 2 * world, dtype=s.dtype, device=s.device)
    packed[:6] = s[:6]
    packed[6 + rank] = s[6]
    packed[6 + world + rank] = s[7]
    dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=group)
    return torch.cat([packed[:6], packed[6:6 + world].min().reshape(1),
                      packed[6 + world:].max().reshape(1)])


def shard_envs(total_envs: int, rank: int, world_size: int):
    """Contiguous block of env instances owned by ``rank`` (envs never interact, so the
    partition needs no halo and no collective): returns (first_env, num_envs)."""
    base, rem = divmod(int(total_envs), int(world_size))
    n = base + (1 if rank < rem else 0)
    first = rank * base + min(rank, rem)
    return first, n


class CoordinatedMultiBuildingControlEnv(MultiAgentEnv):
    """examples/marl/openai/train.py:37-88: the voltage-violation penalty at the common
    bus, computed from the fresh solve and split evenly over the agents -- applied on the
    device in the power-flow kernel's epilogue."""

    VOLTAGE_LIMITS = [0.95, 1.05]
    VV_UNIT_PENALTY = 1e4

    def __init__(self, *args, **kwargs):
        self._penalty = (self.VOLTAGE_LIMITS[0], self.VOLTAGE_LIMITS[1], self.VV_UNIT_PENALTY)
        super().__init__(*args, **kwargs)

    def get_voltage_violation(self):
        self._require_single()
        bus_id = list(set(self.agent_name_bus_map.values()))[0]
        v = self.pf_solver.get_bus_voltage_by_name(bus_id)
        return max([0.0, self.VOLTAGE_LIMITS[0] - v, v - self.VOLTAGE_LIMITS[1]])

    def meta_transform(self, meta) -> dict:
        meta.update({'voltage_violation': self.get_voltage_violation()})
        return meta


class _SolverHostEnv(MultiAgentEnv):
    """One-env handle that only hosts a feeder for stand-alone ``calculate_power_flow``."""
    _is_solver_host = True


def _standalone_solver_env(solver: ZBusSolver) -> MultiAgentEnv:
    from powergridworld_b200.agents.energy_storage import EnergyStorageEnv

    bus = solver.feeder.load_names[0]
    env = _SolverHostEnv(
        common_config={"start_time": "01-01-2021 00:00:00", "end_time": "01-02-2021 00:00:00",
                       "control_timedelta": pd.Timedelta(3600, "s")},
        pf_config={"instance": solver},
        agents=[{"name": "_", "bus": bus, "cls": EnergyStorageEnv, "config": {}}])
    return env
