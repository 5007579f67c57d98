"""Host-side driver of the self-play engine (Python plumbing over the C ABI).

Mirrors the call shapes of the reference's driver layer so that tests and
benchmarks read like the reference's own code:

    run_iteration(...)  ~ SPRL::runIteration   (cpp/src/selfplay/SelfPlay.hpp:203-248)
    run_worker(...)     ~ SPRL::runWorker      (cpp/src/selfplay/GridWorker.hpp:84-198)
    wait_model_path     ~ SPRL::waitModelPath  (cpp/src/selfplay/GridWorker.hpp:35-55)

All compute happens in libsprl_b200.so on the GPU; torch is used only to own
device buffers / streams and to run the reference's traced network.
"""
import ctypes as C
import os
import time

import numpy as np

from . import capi


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


# ---------------------------------------------------------------- environment only
def env_perft(game, depth, device=0):
    """Leaf-count perft from the start position; returns (count, device milliseconds)."""
    count, ms = C.c_uint64(), C.c_float()
    capi.check(capi.load().sprl_env_perft(device, game, depth, C.byref(count), C.byref(ms)))
    return count.value, ms.value


def env_rollout(game, seed, first_game, ngames, record=False, device=0):
    """Random playouts, one GPU thread per game.  With record=True returns the same
    per-position trace the oracle's rollout produces."""
    gi = capi.game_info(game)
    steps = np.zeros(ngames, np.int32)
    final_winner = np.zeros(ngames, np.int8)
    total, ms = C.c_int64(), C.c_float()
    out = dict(game_steps=steps, final_winner=final_winner)
    if record:
        cap = ngames * (gi.max_plies + 1)
        tr = dict(cells=np.zeros((cap, gi.cells), np.int8), player=np.zeros(cap, np.int8),
                  terminal=np.zeros(cap, np.int8), winner=np.zeros(cap, np.int8),
                  mask=np.zeros((cap, gi.actions), np.int8), action=np.zeros(cap, np.int32))
        capi.check(capi.load().sprl_env_rollout(device, game, seed, first_game, ngames, _ptr(steps), _ptr(final_winner),
                                                cap, _ptr(tr["cells"]), _ptr(tr["player"]), _ptr(tr["terminal"]),
                                                _ptr(tr["winner"]), _ptr(tr["mask"]), _ptr(tr["action"]),
                                                C.byref(total), C.byref(ms)))
        for k, v in tr.items():
            out[k] = v[:total.value]
    else:
        capi.check(capi.load().sprl_env_rollout(device, game, seed, first_game, ngames, _ptr(steps), _ptr(final_winner),
                                                0, None, None, None, None, None, None, C.byref(total), C.byref(ms)))
    out["total_positions"] = total.value
    out["elapsed_ms"] = ms.value
    return out


def env_step(game, cells, player, action, device=0):
    gi = capi.game_info(game)
    cells = np.ascontiguousarray(cells, np.int8).reshape(-1, gi.cells)
    n = cells.shape[0]
    player = np.ascontiguousarray(player, np.int8)
    action = np.ascontiguousarray(action, np.int32)
    out = dict(cells=np.zeros((n, gi.cells), np.int8), player=np.zeros(n, np.int8), terminal=np.zeros(n, np.int8),
               winner=np.zeros(n, np.int8), mask=np.zeros((n, gi.actions), np.int8))
    capi.check(capi.load().sprl_env_step(device, game, n, _ptr(cells), _ptr(player), _ptr(action), _ptr(out["cells"]),
                                         _ptr(out["player"]), _ptr(out["terminal"]), _ptr(out["winner"]), _ptr(out["mask"])))
    return out


def env_line(game, actions, device=0):
    """The positions along one line of play from the start position (a chain of GameNode::getAddChild calls,
    games/GameNode.hpp:96-110): dict of cells [n+1, cells], player / terminal / winner [n+1], mask [n+1, A].  Every game
    incl. Go; an illegal action raises SprlError."""
    gi = capi.game_info(game)
    actions = np.ascontiguousarray(actions, np.int32).reshape(-1)
    n = actions.shape[0] + 1
    out = dict(cells=np.zeros((n, gi.cells), np.int8), player=np.zeros(n, np.int8), terminal=np.zeros(n, np.int8),
               winner=np.zeros(n, np.int8), mask=np.zeros((n, gi.actions), np.int8))
    capi.check(capi.load().sprl_env_line(device, game, n - 1, _ptr(actions), _ptr(out["cells"]), _ptr(out["player"]),
                                         _ptr(out["terminal"]), _ptr(out["winner"]), _ptr(out["mask"])))
    return out


# ---------------------------------------------------------------------- the engine
class Engine:
    """One self-play engine = `num_slots` concurrent trees on one GPU."""

    def __init__(self, game, evaluator=capi.EVAL_UNIFORM, device=0, **overrides):
        self.lib = capi.load()
        self.cfg = capi.default_config(game)
        self.cfg.device = device
        self.cfg.evaluator = evaluator
        for k, v in overrides.items():
            if not hasattr(self.cfg, k):
                raise TypeError(f"unknown engine option {k}")
            setattr(self.cfg, k, v)
        self.gi = capi.game_info(game)
        self.handle = C.c_void_p()
        capi.check(self.lib.sprl_create(C.byref(self.cfg), C.byref(self.handle)))
        self.samples_per_move = self.gi.nsym if self.cfg.use_sym else 1
        self._nn = None
        self._match_running = False
        self._stream = None

    def close(self):
        if self.handle:
            self.lib.sprl_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- low level ------------------------------------------------------------------
    def set_stream(self, cuda_stream):
        capi.check(self.lib.sprl_set_stream(self.handle, C.c_void_p(cuda_stream)))

    def set_game_stride(self, stride):
        capi.check(self.lib.sprl_set_game_stride(self.handle, stride))

    def set_openings(self, lines):
        """Opening lines (sequences of actions from the start position) for the games and trees that the next
        run_iteration / run_match / begin_trees starts: stream id t starts from line t % len(lines), a match game from
        line (t // 2) % len(lines) with both colour assignments.  Samples and move records cover the searched moves only.
        An empty sequence turns openings off (sprl_set_openings)."""
        lines = [np.asarray(line, np.int64).reshape(-1) for line in lines]
        offsets = np.zeros(len(lines) + 1, np.int64)
        offsets[1:] = np.cumsum([len(line) for line in lines])
        actions = np.ascontiguousarray(np.concatenate(lines) if lines else np.zeros(0), np.int32)
        capi.check(self.lib.sprl_set_openings(self.handle, len(lines), _ptr(offsets), _ptr(actions)))

    @property
    def eval_batch(self):
        return self.lib.sprl_eval_batch(self.handle)

    def begin_iteration(self, first_game, num_games):
        capi.check(self.lib.sprl_begin_iteration(self.handle, first_game, num_games))

    def round(self):
        capi.check(self.lib.sprl_round(self.handle))

    def poll(self):
        playing, failed = C.c_int64(), C.c_int64()
        capi.check(self.lib.sprl_poll(self.handle, C.byref(playing), C.byref(failed)))
        return playing.value, failed.value

    def stats(self):
        s = capi.Stats()
        capi.check(self.lib.sprl_get_stats(self.handle, C.byref(s)))
        return s.as_dict()

    def check_guards(self):
        """(pools checked, pools whose guard bands were overwritten): out-of-bounds writes of the kernels."""
        n, bad = C.c_int64(), C.c_int64()
        capi.check(self.lib.sprl_debug_check_guards(self.handle, C.byref(n), C.byref(bad)))
        return n.value, bad.value

    def reset_stats(self):
        capi.check(self.lib.sprl_reset_stats(self.handle))

    # -- evaluator plumbing -----------------------------------------------------------
    def attach_network(self, module, use_cuda_graph=True):
        """Attach the reference's traced network (a torch.jit module on this GPU).  Leaf
        planes are written by the search kernel straight into the tensor the module reads,
        and its outputs are read in place by the next search launch: no host round trip."""
        import torch
        dev = torch.device("cuda", self.cfg.device)
        B, gi = self.eval_batch, self.gi
        nn = dict(module=module, graph=None, torch=torch, dev=dev)
        nn["inp"] = torch.zeros((B, 2 * gi.history + 1, gi.rows, gi.cols), dtype=torch.float32, device=dev)
        nn["logits"] = torch.zeros((B, gi.actions), dtype=torch.float32, device=dev)
        nn["value"] = torch.zeros((B,), dtype=torch.float32, device=dev)
        capi.check(self.lib.sprl_bind_eval_buffers(self.handle, C.c_void_p(nn["inp"].data_ptr()),
                                                    C.c_void_p(nn["logits"].data_ptr()), C.c_void_p(nn["value"].data_ptr())))
        nn["use_graph"] = use_cuda_graph
        rows = C.c_void_p()
        capi.check(self.lib.sprl_eval_rows(self.handle, C.byref(rows)))
        nn["rows"] = rows.value            # uint32[2] on the device: rows in use per launch (per agent in a match)
        self._nn = nn

    def attach_evalnet(self, evalnet, use_cuda_graph=True):
        """Attach the library's own evaluator (sprl_b200.evalnet.EvalNet, csrc/evalnet.cu): the search
        kernel writes leaf planes, the tcgen05 tower reads them and writes logits / value in place."""
        self.attach_network(None, use_cuda_graph)
        self._nn["evalnet"] = evalnet

    def attach_match_evaluators(self, evaluators, use_cuda_graph=True):
        """Match play with networks: evaluators[k] serves agent k's trees = rows [k*half, (k+1)*half) of the
        evaluator batch, half = (num_slots // 2) * max_queue.  An entry is an EvalNet, a traced module, or None
        (that agent uses a device evaluator)."""
        self.attach_network(None, use_cuda_graph)
        self._nn["match_evaluators"] = list(evaluators)

    def _forward_rows(self, ev, lo, n):
        nn = self._nn
        torch = nn["torch"]
        if hasattr(ev, "forward_ptr"):
            ev.forward_ptr(nn["inp"][lo:].data_ptr(), n, nn["logits"][lo:].data_ptr(), nn["value"][lo:].data_ptr(),
                           torch.cuda.current_stream(nn["dev"]).cuda_stream, d_rows=nn["rows"] + (4 if lo else 0))
        else:
            with torch.no_grad():
                logits, value = ev(nn["inp"][lo:lo + n])
                nn["logits"][lo:lo + n].copy_(logits)
                nn["value"][lo:lo + n].copy_(value.reshape(-1))

    def _forward(self):
        nn = self._nn
        torch = nn["torch"]
        if self._match_running and nn.get("match_evaluators") is not None:
            half = (self.cfg.num_slots // 2) * self.cfg.max_queue
            for k, ev in enumerate(nn["match_evaluators"]):
                if ev is not None:
                    self._forward_rows(ev, k * half, half)
            return
        if nn.get("evalnet") is not None:
            nn["evalnet"].forward_ptr(nn["inp"].data_ptr(), nn["inp"].shape[0], nn["logits"].data_ptr(),
                                      nn["value"].data_ptr(), torch.cuda.current_stream(nn["dev"]).cuda_stream,
                                      d_rows=nn["rows"] if nn.get("counted", True) else None)
            return
        with torch.no_grad():
            logits, value = nn["module"](nn["inp"])
            nn["logits"].copy_(logits)
            nn["value"].copy_(value.reshape(-1))

    def _round_with_network(self):
        self.round()
        self._forward()

    def _capture(self, key="graph"):
        """Captures [search launch -> network forward -> output copy] as one CUDA graph."""
        nn = self._nn
        torch = nn["torch"]
        side = torch.cuda.Stream(device=nn["dev"])
        side.wait_stream(torch.cuda.current_stream(nn["dev"]))
        with torch.cuda.stream(side):
            for _ in range(3):                      # warm up cuDNN autotune / lazy init outside capture
                self._forward()
        torch.cuda.current_stream(nn["dev"]).wait_stream(side)
        torch.cuda.synchronize(nn["dev"])
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self.set_stream(torch.cuda.current_stream(nn["dev"]).cuda_stream)
            self._round_with_network()
        self.set_stream(torch.cuda.current_stream(nn["dev"]).cuda_stream)
        nn[key] = graph

    # -- runIteration -------------------------------------------------------------------
    def run_iteration(self, num_games, first_game=0, collect=True, poll_every=None):
        """Plays games first_game .. first_game+num_games-1 to the end.  Returns
        (states [n,2H+1,R,C], distributions [n,A], outcomes [n]) as numpy arrays in the
        reference's order when collect=True."""
        if self.cfg.evaluator == capi.EVAL_EXTERNAL:
            if self._nn is None:
                raise capi.SprlError(capi.SPRL_E_STATE, "attach_network() first")
            nn = self._nn
            torch = nn["torch"]
            with torch.cuda.device(nn["dev"]):
                self.set_stream(torch.cuda.current_stream(nn["dev"]).cuda_stream)
                self.begin_iteration(first_game, num_games)
                if nn["use_graph"] and nn["graph"] is None:
                    self._capture()
                every = poll_every or 64
                while True:
                    for _ in range(every):
                        if nn["graph"] is not None:
                            nn["graph"].replay()
                        else:
                            self._round_with_network()
                    playing, failed = self.poll()
                    if failed:
                        self._raise_slot_failure()
                    if playing == 0:
                        break
        else:
            capi.check(self.lib.sprl_run_iteration(self.handle, first_game, num_games, None, None))
        self._check_evaluators()
        return self.collect_samples() if collect else None

    # -- step-wise trees: UCTTree's own surface (uct/UCTTree.hpp:62-210) ------------------------------
    def begin_trees(self, num_trees, first_game=0):
        """UCTTree(start position, ...) for trees 0..num_trees-1; tree i draws from stream first_game + i * stride."""
        if self._nn is not None:
            torch = self._nn["torch"]
            self.set_stream(torch.cuda.current_stream(self._nn["dev"]).cuda_stream)
        capi.check(self.lib.sprl_begin_trees(self.handle, first_game, num_trees))
        self._num_trees = num_trees

    def search(self, sims):
        """while (traversals < sims) { searchAndGetLeaves; evaluateAndBackpropLeaves } for every live tree."""
        if self.cfg.evaluator == capi.EVAL_EXTERNAL:
            if self._nn is None:
                raise capi.SprlError(capi.SPRL_E_STATE, "attach_network() first")
            torch = self._nn["torch"]

            def forward(user, d_in, batch, d_logits, d_value, stream):
                try:
                    self._forward()
                    return 0
                except Exception:           # must not propagate through the C frame
                    import traceback
                    traceback.print_exc()
                    return 1
            cb = capi.FORWARD_FN(forward)
            with torch.cuda.device(self._nn["dev"]):
                capi.check(self.lib.sprl_search(self.handle, sims, cb, None))
        else:
            capi.check(self.lib.sprl_search(self.handle, sims, None, None))

    def root_stats(self):
        """getDecisionNode()->getEdgeStatistics() of every tree: dict of N, W, P [trees, A], root_N, root_W, player,
        terminal, winner, traversals, queued [trees], mask [trees, A]."""
        n, A = self._num_trees, self.gi.actions
        r = dict(N=np.zeros((n, A), np.float32), W=np.zeros((n, A), np.float32), P=np.zeros((n, A), np.float32),
                 root_N=np.zeros(n, np.float32), root_W=np.zeros(n, np.float32), player=np.zeros(n, np.int8),
                 terminal=np.zeros(n, np.int8), winner=np.zeros(n, np.int8), traversals=np.zeros(n, np.int32),
                 mask=np.zeros((n, A), np.int8), queued=np.zeros(n, np.int32))
        capi.check(self.lib.sprl_root_stats(self.handle, n, _ptr(r["N"]), _ptr(r["W"]), _ptr(r["P"]), _ptr(r["root_N"]),
                                            _ptr(r["root_W"]), _ptr(r["player"]), _ptr(r["terminal"]), _ptr(r["winner"]),
                                            _ptr(r["traversals"]), _ptr(r["mask"]), _ptr(r["queued"])))
        return r

    def advance(self, actions):
        """advanceDecision(actions[i]) for tree i; -1 leaves a tree where it is."""
        a = np.ascontiguousarray(actions, np.int32)
        capi.check(self.lib.sprl_advance(self.handle, _ptr(a), a.shape[0]))

    # -- match play (Evaluate.cpp) ----------------------------------------------------------
    def run_match(self, agents, num_games, first_game=0, poll_every=None):
        """Plays a match of `num_games` games between two agents on num_slots // 2 concurrent pairs of trees.
        agents: two dicts with evaluator (capi.EVAL_*), use_sym, init_q and, for HashNet, hash_salt; agents with
        EVAL_EXTERNAL take their network from attach_match_evaluators().  Returns winner / moves / rng draws per
        game and the tally (wins of agent 0, wins of agent 1, draws) as Evaluate.cpp counts it."""
        cfgs = (capi.AgentConfig * 2)()
        for k, ag in enumerate(agents):
            cfgs[k] = capi.AgentConfig(evaluator=ag["evaluator"], use_sym=int(ag.get("use_sym", 1)),
                                       init_q=ag.get("init_q", capi.INITQ_PARENT), hash_salt=ag.get("hash_salt", 0))
        external = any(ag["evaluator"] == capi.EVAL_EXTERNAL for ag in agents)
        self._match_running = True
        try:
            if external:
                nn = self._nn
                if nn is None or nn.get("match_evaluators") is None:
                    raise capi.SprlError(capi.SPRL_E_STATE, "attach_match_evaluators() first")
                torch = nn["torch"]
                with torch.cuda.device(nn["dev"]):
                    self.set_stream(torch.cuda.current_stream(nn["dev"]).cuda_stream)
                    capi.check(self.lib.sprl_match_begin(self.handle, cfgs, first_game, num_games))
                    if nn["use_graph"] and nn.get("graph_match") is None:
                        self._capture("graph_match")
                    self._poll_loop(nn.get("graph_match"), poll_every or 64, True)
            else:
                capi.check(self.lib.sprl_run_match(self.handle, cfgs, first_game, num_games, None, None))
        finally:
            self._match_running = False
        self._check_evaluators()
        winner = np.zeros(num_games, np.int8)
        moves = np.zeros(num_games, np.int32)
        draws = np.zeros(num_games, np.uint64)
        wins = (C.c_int64 * 2)()
        ties = C.c_int64()
        capi.check(self.lib.sprl_match_results(self.handle, num_games, _ptr(winner), _ptr(moves), _ptr(draws), wins, C.byref(ties)))
        return dict(game_winner=winner, game_moves=moves, game_rng_draws=draws, wins=(wins[0], wins[1]), draws=ties.value)

    def _poll_loop(self, graph, every, forward):
        while True:
            for _ in range(every):
                if graph is not None:
                    graph.replay()
                elif forward:
                    self._round_with_network()
                else:
                    self.round()
            playing, failed = self.poll()
            if failed:
                self._raise_slot_failure()
            if playing == 0:
                return

    def _check_evaluators(self):
        """Raises when a library evaluator reported a failure during the run (pipeline time-out, or an activation
        outside the range of its fp16 split): outputs are never silently clamped."""
        nn = self._nn or {}
        for ev in [nn.get("evalnet")] + list(nn.get("match_evaluators") or []):
            if ev is not None and hasattr(ev, "status"):
                ev.status()

    def _raise_slot_failure(self):
        # run_iteration's C path formats the message; reuse it through a zero-round call
        raise capi.SprlError(capi.SPRL_E_CAPACITY, "a tree slot ran out of node units or moves; raise units_per_tree")

    def iteration_counts(self):
        m, s = C.c_int64(), C.c_int64()
        capi.check(self.lib.sprl_iteration_counts(self.handle, C.byref(m), C.byref(s)))
        return m.value, s.value

    def stream_samples(self, cap_samples):
        """Streamed sample output (sprl_stream_samples): allocates page-locked host arrays for up to cap_samples rows; from
        now on finished games are embedded and copied while the others still play, and collect_samples() / run_iteration()
        return views of these arrays (valid until the next iteration).  cap_samples = 0 turns it off."""
        gi = self.gi
        if not cap_samples:
            capi.check(self.lib.sprl_stream_samples(self.handle, 0, None, None, None, 0))
            self._stream = None
            return
        bufs = (np.empty((cap_samples, 2 * gi.history + 1, gi.rows, gi.cols), np.float32), np.empty((cap_samples, gi.actions), np.float32),
                np.empty((cap_samples,), np.float32))
        capi.check(self.lib.sprl_stream_samples(self.handle, cap_samples, _ptr(bufs[0]), _ptr(bufs[1]), _ptr(bufs[2]), 1))
        self._stream = bufs

    def stream_info(self):
        g, n, c = C.c_int64(), C.c_int64(), C.c_uint64()
        capi.check(self.lib.sprl_stream_info(self.handle, C.byref(g), C.byref(n), C.byref(c)))
        return dict(games_done=g.value, samples_done=n.value, chunks_while_playing=c.value)

    def collect_samples(self):
        gi = self.gi
        if getattr(self, "_stream", None) is not None:
            st, di, ou = self._stream
            got = C.c_int64()
            capi.check(self.lib.sprl_collect_samples(self.handle, st.shape[0], _ptr(st), _ptr(di), _ptr(ou), C.byref(got)))
            return st[:got.value], di[:got.value], ou[:got.value]
        _, n = self.iteration_counts()
        states = np.empty((n, 2 * gi.history + 1, gi.rows, gi.cols), np.float32)
        dists = np.empty((n, gi.actions), np.float32)
        outcomes = np.empty((n,), np.float32)
        got = C.c_int64()
        capi.check(self.lib.sprl_collect_samples(self.handle, n, _ptr(states), _ptr(dists), _ptr(outcomes), C.byref(got)))
        assert got.value == n
        return states, dists, outcomes

    def collect_samples_device(self):
        """The iteration's samples left on the GPU (SURVEY.md 8f N1: hand-off to an in-process trainer
        without the filesystem): torch tensors that alias engine-owned device memory, valid until the
        next begin_iteration / collect call.  Same order and layout as collect_samples()."""
        import torch
        gi = self.gi
        ds, dd, do, n = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_int64()
        capi.check(self.lib.sprl_collect_samples_device(self.handle, C.byref(ds), C.byref(dd), C.byref(do), C.byref(n)))
        dev = torch.device("cuda", self.cfg.device)

        class _View:            # __cuda_array_interface__ v3 over a raw device pointer
            def __init__(self, ptr, shape):
                self.__cuda_array_interface__ = dict(shape=shape, typestr="<f4", data=(ptr, False), version=3, strides=None,
                                                     stream=None)

        def view(ptr, shape):
            if n.value == 0:
                return torch.empty(shape, dtype=torch.float32, device=dev)
            return torch.as_tensor(_View(ptr.value, shape), device=dev)

        torch.cuda.synchronize(dev)
        return (view(ds, (n.value, 2 * gi.history + 1, gi.rows, gi.cols)), view(dd, (n.value, gi.actions)),
                view(do, (n.value,)))

    def move_stats(self, num_games):
        """Per-move root statistics of the last iteration (engine created with record_stats=1)."""
        gi = self.gi
        m, _ = self.iteration_counts()
        A = gi.actions
        r = dict(move_N=np.zeros((m, A), np.float32), move_W=np.zeros((m, A), np.float32),
                 move_P=np.zeros((m, A), np.float32), move_root_N=np.zeros(m, np.float32),
                 move_root_W=np.zeros(m, np.float32), move_action=np.zeros(m, np.int32),
                 move_traversals=np.zeros(m, np.int32), move_player=np.zeros(m, np.int8),
                 game_moves=np.zeros(num_games, np.int32), game_rng_draws=np.zeros(num_games, np.uint64))
        got = C.c_int64()
        capi.check(self.lib.sprl_move_stats(self.handle, m, _ptr(r["move_N"]), _ptr(r["move_W"]), _ptr(r["move_P"]),
                                            _ptr(r["move_root_N"]), _ptr(r["move_root_W"]), _ptr(r["move_action"]),
                                            _ptr(r["move_traversals"]), _ptr(r["move_player"]), _ptr(r["game_moves"]),
                                            _ptr(r["game_rng_draws"]), C.byref(got)))
        return r


def write_npy(path, array):
    """npy::write_npy of the reference (float32, C order), through the library's writer."""
    a = np.ascontiguousarray(array, np.float32)
    shape = (C.c_uint64 * max(a.ndim, 1))(*a.shape)
    capi.check(capi.load().sprl_write_npy_f32(path.encode(), _ptr(a), shape, a.ndim))


def wait_model_path(iteration, run_name, interval=30.0, settle=5.0, root="."):
    """SPRL::waitModelPath: "random" for iteration -1, else block until the controller's
    traced model file exists (data/models/<run>/traced_<run>_iteration_<i>.pt)."""
    if iteration == -1:
        return "random"
    path = os.path.join(root, "data", "models", run_name, f"traced_{run_name}_iteration_{iteration}.pt")
    while not os.path.exists(path):
        print(f"Spinning on traced model from iteration {iteration}...", flush=True)
        time.sleep(interval)
    time.sleep(settle)
    return path


def run_worker(run_name, save_dir, game, num_iters, init_games, init_sims, init_batch, init_queue,
               games, sims, batch, queue, dir_eps, dir_alpha, num_slots=None, device=0, seed=0,
               load_model=None, root=".", wait_interval=30.0, settle=5.0, first_game_of_iter=None):
    """SPRL::runWorker: per iteration wait for the controller's model, play the games, write
    <save_dir>/<run>_iteration_<i>_{states,distributions,outcomes}.npy.  Iteration 0 uses the
    uniform evaluator (the reference passes RandomNetwork as initialNetwork, OTHWorker.cpp:51)
    and the init* search parameters; later iterations load the traced module with `load_model` (default: torch.jit.load onto
    the engine's GPU).  (The reference self-initialises maxBatchSize/maxQueueSize
    for iter > 0, GridWorker.hpp:120-121, which is undefined behaviour; the intended values are used.)"""
    os.makedirs(save_dir, exist_ok=True)
    if load_model is None:
        def load_model(path):
            import torch
            return torch.jit.load(path, map_location=torch.device("cuda", device)).eval()
    for it in range(num_iters):
        print(f"Starting iteration {it}...", flush=True)
        model_path = wait_model_path(it - 1, run_name, wait_interval, settle, root)
        n_games = init_games if it == 0 else games
        opts = dict(sims=init_sims if it == 0 else sims, max_batch=init_batch if it == 0 else batch,
                    max_queue=init_queue if it == 0 else queue, dir_eps=dir_eps, dir_alpha=dir_alpha,
                    num_slots=min(num_slots or n_games, n_games), max_games=n_games, seed=seed, device=device)
        first = first_game_of_iter(it) if first_game_of_iter else it * max(init_games, games)
        if model_path == "random":
            print("Using initial network...", flush=True)
            eng = Engine(game, capi.EVAL_UNIFORM, **opts)
        else:
            print("Using traced PyTorch network...", flush=True)
            eng = Engine(game, capi.EVAL_EXTERNAL, **opts)
            module = load_model(model_path)
            try:        # the library's tcgen05 evaluator fed with the module's parameters; other shapes run the module itself
                from .evalnet import EvalNet
                eng.attach_evalnet(EvalNet(module, device=device, rows=eng.gi.rows, cols=eng.gi.cols))
            except (capi.SprlError, KeyError):
                eng.attach_network(module)
        with eng:
            states, dists, outcomes = eng.run_iteration(n_games, first_game=first)
        base = os.path.join(save_dir, f"{run_name}_iteration_{it}")
        write_npy(base + "_states.npy", states)
        write_npy(base + "_distributions.npy", dists)
        write_npy(base + "_outcomes.npy", outcomes)
