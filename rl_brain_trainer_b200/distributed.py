"""Multi-GPU plumbing: envs / episodes shard by index, collectives only where the path has a real exchange.

* evaluation: no data-path collective; one all-reduce (sum) of a small statistics vector at the end.
* training: one all-reduce (sum) of the flat gradient (+ the statistics) per minibatch; every rank then applies the
  identical Adam step.  Curriculum promotion replays the reference's per-episode windowed rule on the rollout's ordered outcome
  stream, gathered over ranks in env order, so all ranks switch stage together (``CurriculumTracker``).

All helpers take plain tensors and an optional process group, so they run under NCCL (one rank per GPU) and under gloo on
CPU tensors (tests/test_distributed_gloo.py, world_size 2).

``PeerGradExchange`` is the NVLink peer-memory form of the training all-reduce (``csrc/kin_peer.cu``): the reduction kernel pushes
the rank's gradient straight into every peer's receive buffer and a gather kernel sums the slots in rank order -- two small
kernels per minibatch instead of a latency-bound NCCL call; ``torch.distributed`` only carries the one-off IPC handle exchange.
"""

from __future__ import annotations

from typing import Any

import numpy as np
import torch
import torch.distributed as dist


def world(group: Any = None) -> tuple[int, int]:
    """(rank, world_size); (0, 1) when torch.distributed is not initialised."""
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def shard_slice(n_total: int, rank: int, world_size: int) -> slice:
    """Contiguous shard of ``n_total`` independent units (episodes, envs, route replicas) owned by ``rank``.

    The first ``n_total % world_size`` ranks get one extra unit, so every unit is owned exactly once.
    """
    base, extra = divmod(int(n_total), int(world_size))
    start = rank * base + min(rank, extra)
    return slice(start, start + base + (1 if rank < extra else 0))


def allreduce_sum_(t: torch.Tensor, group: Any = None) -> torch.Tensor:
    """In-place sum over ranks (no-op for a single process)."""
    if world(group)[1] > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


def allreduce_max_(t: torch.Tensor, group: Any = None) -> torch.Tensor:
    if world(group)[1] > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return t


def check_same_on_all_ranks(value: Any, what: str, group: Any = None) -> None:
    """Raise on every rank unless every rank of ``group`` holds an equal ``value`` (a small picklable, e.g. a table checksum)."""
    n = world(group)[1]
    if n > 1:
        values: list[Any] = [None] * n
        dist.all_gather_object(values, value, group=group)
        if any(v != values[0] for v in values):
            raise RuntimeError(f"{what} differs between ranks: {values}")


def reduce_eval_stats(success: torch.Tensor, final_pos: torch.Tensor, final_ori: torch.Tensor, env_steps: torch.Tensor | int,
                      group: Any = None) -> dict[str, float]:
    """Success rate / mean errors / env-steps over all ranks from per-rank episode rows (one small all-reduce)."""
    v = torch.stack([success.double().sum(), torch.as_tensor(float(success.numel()), dtype=torch.float64, device=success.device),
                     final_pos.double().sum(), final_ori.double().sum(),
                     torch.as_tensor(env_steps, dtype=torch.float64, device=success.device).reshape(())])
    allreduce_sum_(v, group)
    n = max(float(v[1]), 1.0)
    return {"episodes": float(v[1]), "success_rate": float(v[0]) / n, "mean_final_position_error": float(v[2]) / n,
            "mean_final_orientation_error": float(v[3]) / n, "env_steps": float(v[4])}


class PeerGradExchange:
    """Per-minibatch gradient all-reduce (sum) over CUDA-IPC peer buffers of the GPUs of one node (``kin_peer_*`` in the C ABI).

    Two forms.  Fused (the tensor-core update): ``kin_ppo_grad_tc_exchange`` does the whole exchange in the gradient kernel's tail --
    ``next_epoch()`` hands it the exchange counter, ``buffers`` / ``timed_out`` the rest.  Two-kernel (the strict-fp32 update):
    ``push(partials, n_cta, global_batch)`` reduces this rank's per-CTA rows and stores them into every rank's buffer;
    ``gather(grad, stats)`` waits on the device for all ranks and writes the rank-ordered sum (bitwise identical everywhere).
    Everything only enqueues kernels on the current stream.  ``check()`` raises if a peer never arrived (device-side timeout).
    """

    def __init__(self, n_params: int, device: torch.device, group: Any = None) -> None:
        import ctypes

        from . import _lib

        self._L, self._check = _lib.lib(), _lib.check
        self.rank, self.world = world(group)
        if self.world > 8:
            raise _lib.KinError("PeerGradExchange: at most 8 ranks (the GPUs of one NVSwitch node)")
        self.P, self.device = int(n_params), torch.device(device)
        self.epoch = 0
        with torch.cuda.device(self.device):
            own = ctypes.c_void_p()
            handle = ctypes.create_string_buffer(_lib.define("KIN_PEER_HANDLE_BYTES"))
            self._check(self._L.kin_peer_buffer_create(self.P, self.world, ctypes.byref(own), handle))
            self._own = own.value
            handles: list[Any] = [None] * self.world
            if self.world > 1:
                dist.all_gather_object(handles, bytes(handle.raw), group=group)
            self._bufs = self.buffers = (ctypes.c_void_p * self.world)()
            self._opened: list[int] = []
            for r in range(self.world):
                if r == self.rank:
                    self._bufs[r] = self._own
                else:
                    ptr = ctypes.c_void_p()
                    self._check(self._L.kin_peer_buffer_open(handles[r], ctypes.byref(ptr)))
                    self._bufs[r] = ptr.value
                    self._opened.append(ptr.value)
            self.timed_out = torch.zeros(1, dtype=torch.int32, device=self.device)
            torch.cuda.synchronize(self.device)
        if self.world > 1:
            dist.barrier(group=group)        # every buffer exists and is zeroed before the first push can reach it

    def push(self, partials: torch.Tensor, n_cta: int, global_batch: int) -> None:
        self.epoch += 1
        self._check(self._L.kin_peer_grad_push(partials.data_ptr(), int(n_cta), self.P, int(global_batch), self._bufs, self.rank, self.world,
                                               self.epoch, torch.cuda.current_stream(self.device).cuda_stream))

    def next_epoch(self) -> int:
        """Exchange counter for the fused form (``kin_ppo_grad_tc_exchange``: push + gather inside the gradient kernel's tail)."""
        self.epoch += 1
        return self.epoch

    def gather(self, grad: torch.Tensor, stats: torch.Tensor | None) -> None:
        self._check(self._L.kin_peer_grad_gather(self._own, self.P, self.world, self.epoch, grad.data_ptr(),
                                                 None if stats is None else stats.data_ptr(), self.timed_out.data_ptr(),
                                                 torch.cuda.current_stream(self.device).cuda_stream))

    def poll(self) -> None:
        """Non-blocking form of ``check``: enqueue a copy of the device flag into pinned host memory and look at the PREVIOUS poll's copy
        (no stream synchronisation; a dead peer is noticed one poll late at worst, the blocking ``check`` at the end of the update still runs)."""
        if not hasattr(self, "_host_flag"):
            self._host_flag = torch.zeros(1, dtype=torch.int32).pin_memory()
        if int(self._host_flag[0]):
            self.check()
        self._host_flag.copy_(self.timed_out, non_blocking=True)

    def check(self) -> None:
        if int(self.timed_out.item()):
            from . import _lib

            raise _lib.KinError("PeerGradExchange: a peer rank never delivered its gradient (device-side wait timed out)")

    def close(self) -> None:
        """Unmap the peers' buffers and free this rank's (after the stream drained).  Every rank must have finished its last
        gather before any rank closes: call it at the same point of the program on all ranks (``PPOTrainer.close`` does)."""
        if getattr(self, "_own", None) is None:
            return
        torch.cuda.synchronize(self.device)
        for ptr in self._opened:
            self._L.kin_peer_buffer_close(ptr)
        self._L.kin_peer_buffer_destroy(self._own)
        self._own, self._opened = None, []

    def __del__(self) -> None:  # pragma: no cover - interpreter shutdown order is not ours
        try:
            self.close()
        except Exception:
            pass


class CurriculumTracker:
    """``PointCurriculumTracker`` / ``PointCurriculumCallback`` (envs/curriculum.py:104-154, training/callbacks.py:54-92), exact:
    a deque of the last ``window_episodes`` episode outcomes, checked after EVERY finished episode in the order SB3's callback sees
    them (time step, then env index); promotion needs ``min_episodes_per_stage`` episodes since the last promotion, a full window and
    a windowed rate >= the threshold, and clears the window.

    The batched trainer finishes thousands of episodes per rollout, so the tracker takes the rollout's ordered outcome stream
    (``record_stream``) and replays the per-episode rule on it with prefix sums -- the decisions (which episode triggers, the trigger
    rate, the history) are the reference's; several promotions inside one rollout are possible, as in the reference.  With several
    ranks the per-rank streams are gathered and merged in (time step, rank, env) order = the single-process env order, so every rank
    takes the same decisions.  The env's stage is switched by the caller after the rollout (the fused collection runs a whole rollout
    in one launch), i.e. up to ``n_steps`` later than the reference's callback switches it.
    """

    def __init__(self, n_stages: int, success_rate_threshold: float, window_episodes: int, min_episodes_per_stage: int, stage_index: int = 0) -> None:
        self.n_stages, self.threshold = int(n_stages), float(success_rate_threshold)
        self.window, self.min_episodes = max(int(window_episodes), 1), max(int(min_episodes_per_stage), 1)
        self.stage_index = int(stage_index)
        self.stage_episode_count = 0
        self.recent = np.zeros(0, dtype=np.int64)      # the deque: at most `window` latest outcomes, oldest first
        self.history: list[dict[str, float | int]] = []

    @property
    def max_stage_index(self) -> int:
        return max(self.n_stages - 1, 0)

    def record_episode(self, success: bool) -> bool:
        """One finished episode (the reference's ``record_episode``)."""
        return self.record_stream(np.array([1 if success else 0], dtype=np.int64)) > 0

    def record_stream(self, outcomes: np.ndarray | torch.Tensor, total_timesteps: int | None = None) -> int:
        """Feed finished episodes in callback order (1 = success).  Returns the number of promotions it caused."""
        x = outcomes.detach().cpu().numpy() if isinstance(outcomes, torch.Tensor) else np.asarray(outcomes)
        x = (x != 0).astype(np.int64).reshape(-1)
        promotions = 0
        W = self.window
        while x.size:
            if self.stage_index >= self.max_stage_index:      # the last stage only keeps the window current
                self.stage_episode_count += int(x.size)
                self.recent = np.concatenate([self.recent, x])[-W:]
                return promotions
            seq = np.concatenate([self.recent, x])
            c = np.concatenate([[0], np.cumsum(seq)])
            k = np.arange(x.size)
            end = self.recent.size + k + 1                    # window [end - W, end) after episode k
            full = end >= W
            wsum = c[end] - c[np.maximum(end - W, 0)]
            ok = full & (self.stage_episode_count + k + 1 >= self.min_episodes) & (wsum.astype(np.float64) / float(W) >= self.threshold)
            hit = np.nonzero(ok)[0]
            if hit.size == 0:
                self.stage_episode_count += int(x.size)
                self.recent = seq[-W:]
                return promotions
            j = int(hit[0])
            rec: dict[str, float | int] = {"from_stage_index": self.stage_index, "to_stage_index": self.stage_index + 1,
                                            "trigger_success_rate": float(wsum[j]) / float(W)}
            if total_timesteps is not None:
                rec["total_timesteps"] = int(total_timesteps)
            self.history.append(rec)
            self.stage_index += 1
            self.stage_episode_count = 0
            self.recent = np.zeros(0, dtype=np.int64)
            promotions += 1
            x = x[j + 1:]
        return promotions

    def record_rollout(self, finished: torch.Tensor, success: torch.Tensor, group: Any = None, total_timesteps: int | None = None) -> int:
        """``finished`` / ``success``: bool ``[T, N_local]`` of one rollout.  Builds the ordered outcome stream -- over all ranks of
        ``group`` in (time step, rank, env) order -- and replays it.  Identical result on every rank."""
        t_idx, _ = torch.nonzero(finished, as_tuple=True)     # row-major: time step, then env
        outcome = success[finished].to(torch.int32)
        rank, n_ranks = world(group)
        if n_ranks > 1:
            dev = finished.device if dist.get_backend(group) == "nccl" else torch.device("cpu")
            count = torch.tensor([int(t_idx.numel())], dtype=torch.int64, device=dev)
            counts = [torch.zeros_like(count) for _ in range(n_ranks)]
            dist.all_gather(counts, count, group=group)
            m = int(max(int(c.item()) for c in counts))
            pad = torch.full((2, max(m, 1)), -1, dtype=torch.int32, device=dev)
            pad[0, : t_idx.numel()] = t_idx.to(device=dev, dtype=torch.int32)
            pad[1, : t_idx.numel()] = outcome.to(dev)
            parts = [torch.zeros_like(pad) for _ in range(n_ranks)]
            dist.all_gather(parts, pad, group=group)
            ts = torch.cat([p_[0, : int(c.item())] for p_, c in zip(parts, counts)]).cpu().numpy()
            oc = torch.cat([p_[1, : int(c.item())] for p_, c in zip(parts, counts)]).cpu().numpy()
            order = np.argsort(ts, kind="stable")             # per-rank lists are time-ordered: stable sort = (t, rank, env)
            stream = oc[order]
        else:
            stream = outcome.cpu().numpy()
        return self.record_stream(stream, total_timesteps)

    def snapshot(self) -> dict[str, object]:
        rate = float(self.recent.sum()) / float(self.recent.size) if self.recent.size else 0.0
        return {"stage_index": self.stage_index, "stage_episode_count": self.stage_episode_count, "recent_success_rate": rate,
                "history": list(self.history)}

    def state_dict(self) -> dict[str, Any]:
        return {"stage_index": self.stage_index, "stage_episode_count": self.stage_episode_count, "recent": self.recent.tolist(),
                "history": list(self.history)}

    def load_state_dict(self, d: dict[str, Any]) -> None:
        self.stage_index, self.stage_episode_count = int(d["stage_index"]), int(d["stage_episode_count"])
        self.recent = np.asarray(d.get("recent", []), dtype=np.int64)
        self.history = list(d.get("history", []))
