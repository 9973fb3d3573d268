"""Drop-in surfaces of the reference for callers that step ONE game at a time.

The notebooks never touch ``DroneGame`` directly: they talk to ``DroneGameClient``
(/root/reference/delivery_drone/game/socket_client.py:31-224), which talks newline-delimited JSON
to ``GameSocketServer`` (game/socket_server.py:13-288), which calls the duck-typed game object
(``reset() step(action) get_state() _get_info() .done``).  This module provides all three layers on
top of one ``BatchedDroneEnv`` so existing code runs unchanged:

  * ``DroneGamePool`` / ``DroneGameView``  -- N per-index ``DroneGame`` look-alikes over one batched
    env (freeze-after-done, explicit ``reset()``, 16-key state dict, 7-key info dict, ``needs_reset``)
  * ``InProcessDroneGameClient``           -- the ``DroneGameClient`` API without a socket
  * ``DroneSocketServer`` / ``DroneGameClient`` -- the same wire protocol over TCP (compatibility shim)
  * ``install_aliases()``                  -- registers ``delivery_drone.game.*`` module names so that
    ``from delivery_drone.game.socket_client import DroneGameClient`` resolves here

Stepping one game is one kernel launch over the batch with every other env's action byte set to
DD_ACT_SKIP, then a small device->host read: this path exists for compatibility, not for speed --
batched callers use ``BatchedDroneEnv.step`` directly.
"""
from __future__ import annotations

import ctypes as C
import json
import socket
import sys
import threading
import types
from dataclasses import dataclass
from typing import Any, Dict, List, Optional, Sequence, Tuple

import torch

from . import _native as nv
from .env import BatchedDroneEnv

STATE_KEYS = ("drone_x", "drone_y", "drone_vx", "drone_vy", "drone_angle", "drone_angular_vel", "drone_fuel",
              "platform_x", "platform_y", "distance_to_platform", "dx_to_platform", "dy_to_platform", "speed",
              "landed", "crashed", "steps")                     # game_engine.py:160-177
INFO_KEYS = ("steps", "total_reward", "episode", "fuel_remaining", "distance_to_platform", "speed", "angle")


@dataclass
class DroneState:
    """The 16 fields of ``DroneGame.get_state()`` (socket_client.py:10-28); extra or missing keys
    raise ``TypeError`` exactly like the reference's ``DroneState(**state)``."""
    drone_x: float
    drone_y: float
    drone_vx: float
    drone_vy: float
    drone_angle: float
    drone_angular_vel: float
    drone_fuel: float
    platform_x: float
    platform_y: float
    distance_to_platform: float
    dx_to_platform: float
    dy_to_platform: float
    speed: float
    landed: bool
    crashed: bool
    steps: int


def action_bits(action: Optional[Dict[str, Any]]) -> int:
    """``bool(action.get(key, 0))`` per thruster (game_engine.py:114-118): missing keys are 0, any
    truthy value counts."""
    action = action or {}
    return ((nv.ACT_MAIN if action.get("main_thrust", 0) else 0)
            | (nv.ACT_LEFT if action.get("left_thrust", 0) else 0)
            | (nv.ACT_RIGHT if action.get("right_thrust", 0) else 0))


class _DroneFlags:
    """``game.drone.landed`` / ``game.drone.crashed`` (examples/random_agent.py:43, manual_play.py:80)."""

    def __init__(self, view: "DroneGameView"):
        self._v = view

    @property
    def landed(self) -> bool:
        return bool(self._v._flags() & nv.LANDED)

    @property
    def crashed(self) -> bool:
        return bool(self._v._flags() & nv.CRASHED)


class DroneGamePool:
    """``num_games`` reference-style games backed by ONE batched env on the GPU.

    float64 by default so that numbers match the reference's float64 engine to the last sin/cos ulp;
    ``auto_reset=False`` gives the reference's freeze-after-done."""

    def __init__(self, num_games: int, device="cuda", seed: int = 0, randomize_drone: bool = False,
                 randomize_platform: bool = True, dtype: torch.dtype = torch.float64):
        self.env = BatchedDroneEnv(num_games, device=device, seed=seed, randomize_drone=randomize_drone,
                                   randomize_platform=randomize_platform, auto_reset=False, dtype=dtype,
                                   obs_stride=16)
        n = num_games
        self.num_games = n
        # Pinned host buffers are device-mapped (unified addressing): the kernels read the per-call action / mask
        # bytes and write the per-game record straight through them, so one per-game step is two launches and one
        # stream synchronisation -- no separate copies, no index kernels.
        self._h_act = torch.full((n,), nv.ACT_SKIP, dtype=torch.uint8).pin_memory()
        self._h_mask = torch.zeros(n, dtype=torch.uint8).pin_memory()
        self._h_rec = torch.zeros(n, nv.ENV_RECORD_DOUBLES, dtype=torch.float64).pin_memory()
        self._rec_ok = [False] * n                     # record i is current (invalidated when game i changes)
        self._lock = threading.Lock()
        # DroneGame.__init__ (game_engine.py:40-53): fixed start positions, episode = 0, no reset() yet
        p, dev = self.env.params, self.env.device
        full = lambda v: torch.full((n,), float(v), dtype=dtype, device=dev)
        self.env.inject(full(p.start_x), full(p.start_y), full(p.plat_default_x), full(p.plat_default_y))
        self.env.episode.zero_()
        self.env.observe()                             # obs rows of the initial states
        self.games: List[DroneGameView] = [DroneGameView(self, i) for i in range(n)]

    def __len__(self) -> int:
        return self.num_games

    def __getitem__(self, i: int) -> "DroneGameView":
        return self.games[i]

    def invalidate(self) -> None:
        """Call after touching ``pool.env`` directly (set_state, inject, batched stepping)."""
        with self._lock:
            self.env.observe()
            self._rec_ok = [False] * self.num_games

    # -- device work --------------------------------------------------------------------------
    def _record(self, i: int) -> List[float]:
        """The DD_ENV_RECORD of game i (include/drone_b200.h dd_gather_env), fetched at most once per change."""
        if not self._rec_ok[i]:
            e = self.env
            nv.check(e._lib.dd_gather_env(C.byref(e._state), e.obs.data_ptr(), e.obs_stride, e.reward.data_ptr(),
                                          e.step_flags.data_ptr(), i, self.num_games, self._h_rec[i].data_ptr(),
                                          e._stream()), "dd_gather_env")
            torch.cuda.current_stream(e.device).synchronize()
            self._rec_ok[i] = True
        return self._h_rec[i].tolist()

    def _step_one(self, i: int, bits: int) -> Tuple[List[float], float, int]:
        with self._lock:
            self._h_act[i] = bits
            self.env.step_raw(self._h_act, stats=False)    # every other game carries DD_ACT_SKIP
            self._rec_ok[i] = False
            rec = self._record(i)                          # synchronises: the action byte may be rewritten now
            self._h_act[i] = nv.ACT_SKIP
        return rec[:16], rec[16], int(rec[17])

    def _reset_one(self, i: int) -> List[float]:
        with self._lock:
            e = self.env
            self._h_mask.zero_()
            self._h_mask[i] = 1
            nv.check(e._lib.dd_reset(C.byref(e._state), C.byref(e._params), C.byref(e._cfg), self._h_mask.data_ptr(),
                                     e.obs.data_ptr(), e.obs_stride, self.num_games, e._stream()), "dd_reset")
            e._needs_reset = False
            self._rec_ok[i] = False
            return self._record(i)[:16]

    def _observe_one(self, i: int) -> List[float]:
        with self._lock:
            return self._record(i)[:16]

    def _raw_one(self, i: int) -> Dict[str, float]:
        with self._lock:
            r = self._record(i)
            return {"x": r[21], "y": r[22], "vx": r[23], "vy": r[24], "angle": r[25], "angular_velocity": r[26],
                    "fuel": r[27], "total_reward": r[28], "platform_x": r[29], "platform_y": r[30],
                    "steps": int(r[19]), "episode": int(r[20]) & 0xffffffff, "flags": int(r[18])}


class DroneGameView:
    """One index of a ``DroneGamePool`` with the reference ``DroneGame`` surface
    (game_engine.py:14-298, headless): ``reset() -> dict16``, ``step(action) -> (dict16, float, bool,
    dict7 [+needs_reset])``, ``get_state()``, ``_get_info()``, ``render() -> None``, ``close()`` and the
    attributes callers read (``done steps episode total_reward drone.landed drone.crashed``)."""

    render_mode = None
    screen = None

    def __init__(self, pool: DroneGamePool, index: int):
        self._pool, self._i = pool, int(index)
        self.drone = _DroneFlags(self)

    # -- helpers ------------------------------------------------------------------------------
    def _flags(self) -> int:
        return self._pool._raw_one(self._i)["flags"]

    @staticmethod
    def _state_dict(row: Sequence[float], flags: int) -> Dict[str, Any]:
        d: Dict[str, Any] = {k: float(row[j]) for j, k in enumerate(STATE_KEYS[:13])}
        d["landed"] = bool(flags & nv.LANDED)
        d["crashed"] = bool(flags & nv.CRASHED)
        d["steps"] = int(row[15])
        return d

    # -- DroneGame API ------------------------------------------------------------------------
    def reset(self) -> Dict[str, Any]:
        return self._state_dict(self._pool._reset_one(self._i), 0)

    def step(self, action: Optional[Dict[str, Any]]):
        if self.done:                                   # game_engine.py:107-111, BUGFIX.md:40-52
            info = self._get_info()
            info["needs_reset"] = True
            return self.get_state(), 0, True, info
        row, reward, flags = self._pool._step_one(self._i, action_bits(action))
        return self._state_dict(row, flags), reward, bool(flags & nv.DONE), self._get_info()

    def get_state(self) -> Dict[str, Any]:
        raw = self._pool._raw_one(self._i)
        return self._state_dict(self._pool._observe_one(self._i), raw["flags"])

    def _get_info(self) -> Dict[str, Any]:
        """Raw-unit info dict (game_engine.py:281-298)."""
        r = self._pool._raw_one(self._i)
        dx, dy = r["platform_x"] - r["x"], r["platform_y"] - r["y"]
        return {"steps": r["steps"], "total_reward": r["total_reward"], "episode": r["episode"],
                "fuel_remaining": r["fuel"], "distance_to_platform": (dx * dx + dy * dy) ** 0.5,
                "speed": (r["vx"] * r["vx"] + r["vy"] * r["vy"]) ** 0.5, "angle": r["angle"]}

    def render(self):
        return None                                     # headless only (render_mode=None)

    def close(self) -> None:
        pass

    @property
    def done(self) -> bool:
        return bool(self._flags() & nv.DONE)

    @property
    def steps(self) -> int:
        return self._pool._raw_one(self._i)["steps"]

    @property
    def episode(self) -> int:
        return self._pool._raw_one(self._i)["episode"]

    @property
    def total_reward(self) -> float:
        return self._pool._raw_one(self._i)["total_reward"]


# =================================================================================================
# DroneGameClient without a socket
# =================================================================================================
class InProcessDroneGameClient:
    """``DroneGameClient`` (socket_client.py:31-224) served directly by a list of game objects
    (``DroneGamePool`` views or anything with the ``DroneGame`` surface).  Same return types, same
    exceptions: ``ValueError`` for a bad ``game_id``, ``RuntimeError`` when not connected."""

    def __init__(self, games, host: str = "in-process", port: int = 0, timeout: float = 30.0):
        self.games = list(games.games) if isinstance(games, DroneGamePool) else list(games)
        self.host, self.port, self.timeout = host, port, timeout
        self.connected = False
        self.num_games = len(self.games)

    def connect(self) -> None:
        self.connected = True

    def disconnect(self) -> None:
        self.connected = False

    close = disconnect

    def _check(self, game_id: int) -> None:
        if game_id < 0 or game_id >= self.num_games:
            raise ValueError(f"Invalid game_id: {game_id}. Must be in range [0, {self.num_games})")

    def reset(self, game_id: int = 0) -> DroneState:
        if not self.connected:
            self.connect()
        self._check(game_id)
        return DroneState(**self.games[game_id].reset())

    def step(self, action: Dict[str, int], game_id: int = 0) -> Tuple[DroneState, float, bool, Dict]:
        if not self.connected:
            raise RuntimeError("Not connected to server. Call connect() or reset() first.")
        self._check(game_id)
        state, reward, done, info = self.games[game_id].step(action)
        return DroneState(**state), float(reward), bool(done), info

    def get_state(self, game_id: int = 0) -> DroneState:
        if not self.connected:
            raise RuntimeError("Not connected to server")
        self._check(game_id)
        return DroneState(**self.games[game_id].get_state())

    def __enter__(self):
        self.connect()
        return self

    def __exit__(self, *exc):
        self.disconnect()


# =================================================================================================
# the wire protocol (newline-delimited UTF-8 JSON), both ends
# =================================================================================================
def _send_json(sock: socket.socket, message: Dict) -> None:
    sock.sendall((json.dumps(message) + "\n").encode("utf-8"))


class _LineReader:
    def __init__(self, sock: socket.socket):
        self.sock, self.buf = sock, b""

    def read(self) -> Optional[Dict]:
        """Next JSON message, or None at EOF."""
        while b"\n" not in self.buf:
            data = self.sock.recv(4096)
            if not data:
                return None
            self.buf += data
        line, self.buf = self.buf.split(b"\n", 1)
        return json.loads(line.decode("utf-8")) if line.strip() else self.read()


class DroneSocketServer:
    """Serves a list of game objects over the reference's protocol (game/socket_server.py:126-263):
    ``{"type":"HANDSHAKE","num_games":N}`` on accept, then per request one
    ``{"type":"STATE","game_id","state","reward","done","info"}`` or ``{"type":"ERROR","message"}``.
    RESET replies reward 0.0 / done False / info {}; GET_STATE replies reward 0.0, the game's done flag
    and its info dict; CLOSE ends the session.  One client at a time, like the reference.

    Unlike the reference there is no fps-paced main loop between the socket and the game: requests
    are executed as they arrive."""

    def __init__(self, games, host: str = "localhost", port: int = 5555):
        self.games = list(games.games) if isinstance(games, DroneGamePool) else list(games)
        self.num_games = len(self.games)
        self.host, self.port = host, port
        self.connected = False
        self.running = False
        self._srv: Optional[socket.socket] = None
        self._thread: Optional[threading.Thread] = None

    def start(self, background: bool = True) -> None:
        self._srv = socket.socket(socket.AF_INET, socket.SOCK_STREAM)
        self._srv.setsockopt(socket.SOL_SOCKET, socket.SO_REUSEADDR, 1)
        self._srv.bind((self.host, self.port))
        self.port = self._srv.getsockname()[1]          # port 0 -> the one the OS picked
        self._srv.listen(1)
        self.running = True
        if background:
            self._thread = threading.Thread(target=self.serve_forever, daemon=True)
            self._thread.start()
        else:
            self.serve_forever()

    def serve_forever(self) -> None:
        assert self._srv is not None
        self._srv.settimeout(0.2)
        while self.running:
            try:
                conn, _ = self._srv.accept()
            except socket.timeout:
                continue
            except OSError:
                break
            with conn:
                self.connected = True
                self._session(conn)
                self.connected = False

    def _session(self, conn: socket.socket) -> None:
        _send_json(conn, {"type": "HANDSHAKE", "num_games": self.num_games})
        reader = _LineReader(conn)
        while self.running:
            try:
                msg = reader.read()
            except json.JSONDecodeError as e:
                _send_json(conn, {"type": "ERROR", "message": f"Invalid JSON: {e}"})
                continue
            except OSError:
                return
            if msg is None:
                return                                  # client went away
            try:
                reply = self._execute(msg)
            except Exception as e:                      # never kill the session on a bad request
                reply = {"type": "ERROR", "message": f"Error handling message: {e}"}
            if reply is None:
                return
            try:
                _send_json(conn, reply)
            except OSError:
                return

    def _execute(self, msg: Dict) -> Optional[Dict]:
        kind = msg.get("type")
        gid = msg.get("game_id", 0)                     # default 0: single-game clients
        if not isinstance(gid, int) or gid < 0 or gid >= self.num_games:
            return {"type": "ERROR", "message": f"Invalid game_id: {gid}. Must be in range [0, {self.num_games})"}
        game = self.games[gid]
        if kind == "RESET":
            state, reward, done, info = game.reset(), 0.0, False, {}
        elif kind == "STEP":
            state, reward, done, info = game.step(msg.get("action", {}))
        elif kind == "GET_STATE":
            state, reward, done, info = game.get_state(), 0.0, game.done, game._get_info()
        elif kind == "CLOSE":
            return None
        else:
            return {"type": "ERROR", "message": f"Unknown message type: {kind}"}
        return {"type": "STATE", "game_id": gid, "state": state, "reward": float(reward), "done": bool(done),
                "info": info}

    def stop(self) -> None:
        self.running = False
        if self._srv is not None:
            try:
                self._srv.close()
            except OSError:
                pass
        if self._thread is not None:
            self._thread.join(timeout=2.0)


class DroneGameClient(InProcessDroneGameClient):
    """TCP client with the reference's constructor and behaviour (socket_client.py:31-224):
    lazy connect on ``reset()``, ``ConnectionError`` on EOF, ``RuntimeError`` on a server ERROR."""

    def __init__(self, host: str = "localhost", port: int = 5555, timeout: float = 30.0):
        self.games = []
        self.host, self.port, self.timeout = host, port, timeout
        self.connected = False
        self.num_games = 1                              # until the handshake says otherwise
        self.socket: Optional[socket.socket] = None
        self._reader: Optional[_LineReader] = None

    def connect(self) -> None:
        if self.connected:
            return
        self.socket = socket.create_connection((self.host, self.port), timeout=self.timeout)
        self._reader = _LineReader(self.socket)
        self.connected = True
        hello = self._recv()
        if hello.get("type") == "HANDSHAKE":
            self.num_games = hello["num_games"]

    def disconnect(self) -> None:
        if self.socket is not None:
            try:
                _send_json(self.socket, {"type": "CLOSE"})
                self.socket.close()
            except OSError:
                pass
        self.connected, self.socket, self._reader = False, None, None

    close = disconnect

    def _recv(self) -> Dict:
        assert self._reader is not None
        msg = self._reader.read()
        if msg is None:
            raise ConnectionError("Server closed connection")
        return msg

    def _request(self, message: Dict) -> Dict:
        assert self.socket is not None
        _send_json(self.socket, message)
        reply = self._recv()
        if reply.get("type") == "ERROR":
            raise RuntimeError(f"Server error: {reply['message']}")
        return reply

    def reset(self, game_id: int = 0) -> DroneState:
        if not self.connected:
            self.connect()
        self._check(game_id)
        return DroneState(**self._request({"type": "RESET", "game_id": game_id})["state"])

    def step(self, action: Dict[str, int], game_id: int = 0):
        if not self.connected:
            raise RuntimeError("Not connected to server. Call connect() or reset() first.")
        self._check(game_id)
        r = self._request({"type": "STEP", "action": action, "game_id": game_id})
        return DroneState(**r["state"]), r["reward"], r["done"], r["info"]

    def get_state(self, game_id: int = 0) -> DroneState:
        if not self.connected:
            raise RuntimeError("Not connected to server")
        self._check(game_id)
        return DroneState(**self._request({"type": "GET_STATE", "game_id": game_id})["state"])


def install_aliases() -> None:
    """Make ``from delivery_drone.game.socket_client import DroneGameClient, DroneState`` (what every
    notebook does, Actor_Critic_PPO.ipynb c1:L9) resolve to this module's classes."""
    pkg = sys.modules.setdefault("delivery_drone", types.ModuleType("delivery_drone"))
    game = sys.modules.setdefault("delivery_drone.game", types.ModuleType("delivery_drone.game"))
    sc = types.ModuleType("delivery_drone.game.socket_client")
    sc.DroneGameClient, sc.DroneState = DroneGameClient, DroneState
    ss = types.ModuleType("delivery_drone.game.socket_server")
    ss.GameSocketServer = DroneSocketServer
    sys.modules["delivery_drone.game.socket_client"] = sc
    sys.modules["delivery_drone.game.socket_server"] = ss
    pkg.game, game.socket_client, game.socket_server = game, sc, ss
