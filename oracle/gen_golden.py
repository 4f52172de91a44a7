"""Generate tests/golden/*.npz from the UNMODIFIED reference (build container only).

    python -m oracle.gen_golden            # needs /root/reference (or $R2D2_REF)

What is pinned (all inputs are regenerated from seeds by ``oracle.synth``; the
fixtures hold only small side arrays and the reference's OUTPUTS):

  tree_small.npz      ``PriorityTree`` (priority_tree.py:4-45): a scripted
                      sequence of update()/sample() calls incl. duplicate
                      indices, zero priorities, an empty update and a
                      non-power-of-two capacity; the full tree after every op,
                      sampled indices and IS weights.
  tree_large.npz      the same class at 50,000 and 2^16 leaves: two rounds of
                      sample() + update() of the sampled leaves per capacity.
  replay_ragged.npz   ``LocalBuffer.finish`` -> ``ReplayBuffer.add`` ->
                      ``sample_batch`` / ``update_priorities`` (worker.py:141-261,
                      437-497) on the ragged episode script: per-block metadata,
                      checksums of the frame arrays, the sampled batch (minus
                      frames) and the tree after stale-masked priority updates.
  learner_ragged.npz  ``Learner.run`` (worker.py:318-369) for K consecutive
                      updates on batches sampled from that replay: per update the
                      raw TD vector, mixed priorities, loss, the three Q tensors,
                      per-parameter gradient norms and post-step parameter
                      checksums.
  learner_cfg0.npz    same for BASELINE config #1's shape (batch 4, b/l/f 8/8/4,
                      block_length 40).
"""
from __future__ import annotations

import os
import queue
import sys
import zlib

import numpy as np
import torch

from . import ref_harness, synth
from .learner import init_params

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
A = 9


def crc(a: np.ndarray) -> int:
    return zlib.crc32(np.ascontiguousarray(a).tobytes())


# ------------------------------------------------------------------------------ tree
def tree_script(capacity: int, seed: int):
    """Deterministic op list shared by the generator and the tests."""
    rng = np.random.default_rng([seed, 0x7EE])
    ops = []
    ops.append(("update", np.arange(capacity, dtype=np.int64),
                rng.uniform(1e-3, 1.0, capacity).astype(np.float32)))
    ops.append(("sample", 64, 101))
    dup = rng.integers(0, capacity, 200).astype(np.int64)           # duplicates: last write wins
    ops.append(("update", dup, rng.uniform(0.0, 2.0, 200).astype(np.float32)))
    ops.append(("sample", 17, 102))
    nz = max(1, min(50, capacity // 3))
    z = rng.choice(capacity, nz, replace=False).astype(np.int64)    # zero priorities
    ops.append(("update", z, np.zeros(nz, dtype=np.float32)))
    ops.append(("update", np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.float32)))  # empty
    ops.append(("sample", 256, 103))
    ops.append(("update", dup[:10], rng.uniform(5.0, 9.0, 10).astype(np.float32)))
    ops.append(("sample", 1, 104))
    return ops


def gen_tree(ref):
    out = {}
    for tag, cap in (("p2", 1024), ("np2", 1000), ("tiny", 3)):
        tree = ref.priority_tree.PriorityTree(cap, 0.9, 0.6)
        out[f"{tag}_num_layers"] = np.int64(tree.num_layers)
        for k, op in enumerate(tree_script(cap, 5)):
            if op[0] == "update":
                tree.update(op[1], op[2])
                out[f"{tag}_op{k}_tree"] = tree.ptree.copy()
            else:
                np.random.seed(op[2])
                idx, w = tree.sample(op[1])
                out[f"{tag}_op{k}_idx"] = idx.copy()
                out[f"{tag}_op{k}_isw"] = w.copy()
    np.savez_compressed(os.path.join(OUT, "tree_small.npz"), **out)
    print("tree_small.npz", len(out), "arrays")


def tree_large_script():
    """Per capacity: every leaf's TD error, then two rounds of (n, TD errors written to the n leaves sampled with
    np.random.seed(n))."""
    rng = np.random.default_rng(0)
    cases = []
    for cap in (50_000, 1 << 16):
        td = rng.uniform(1e-3, 1, cap).astype(np.float32)
        cases.append((cap, td, [(n, rng.uniform(0, 2, n).astype(np.float32)) for n in (64, 4096)]))
    return cases


def gen_tree_large(ref):
    """Sampled indices and IS weights of every round, and the tree after its update: a CRC of the whole node array
    plus 2048 nodes at seeded positions (the full trees would be 2 MB)."""
    out = {}
    for cap, td, rounds in tree_large_script():
        tree = ref.priority_tree.PriorityTree(cap, 0.9, 0.6)
        tree.update(np.arange(cap), td)
        pos = np.sort(np.random.default_rng(cap).choice(tree.ptree.size, 2048, replace=False))
        for n, t2 in rounds:
            np.random.seed(n)
            idx, w = tree.sample(n)
            tree.update(idx, t2)
            tag = f"c{cap}_n{n}"
            out[f"{tag}_idx"], out[f"{tag}_isw"] = idx.copy(), w.copy()
            out[f"{tag}_tree_crc"] = np.int64(crc(tree.ptree))
            out[f"{tag}_tree_pos"], out[f"{tag}_tree_sample"] = pos, tree.ptree[pos].copy()
    np.savez_compressed(os.path.join(OUT, "tree_large.npz"), **out)
    print("tree_large.npz", len(out), "arrays")


# ------------------------------------------------------------------------------ replay + learner
def build_reference_replay(ref, script, num_blocks, batch_size, bl=400, ls=40, bi=40, fs=5):
    w = ref.worker
    rb = w.ReplayBuffer([], None, None, buffer_capacity=num_blocks * bl, batch_size=batch_size)
    assert rb.seq_pre_block == bl // ls
    blocks = []
    for seed, steps, done in script:
        lb = w.LocalBuffer(A, forward_steps=fs, burn_in_steps=bi, learning_steps=ls, block_length=bl)
        for blk, prio, ep in synth.drive_actor(lb, seed, steps, done, A, block_length=bl):
            rb.add(blk, prio, ep)
            blocks.append((blk, prio, ep))
    return rb, blocks


def block_meta(prefix, blocks, out):
    for i, (blk, prio, ep) in enumerate(blocks):
        out[f"{prefix}blk{i}_obs_crc"] = np.int64(crc(blk.obs))
        out[f"{prefix}blk{i}_last_action_crc"] = np.int64(crc(blk.last_action))
        out[f"{prefix}blk{i}_last_reward"] = blk.last_reward
        out[f"{prefix}blk{i}_action"] = blk.action
        out[f"{prefix}blk{i}_n_step_reward"] = blk.n_step_reward
        out[f"{prefix}blk{i}_gamma"] = blk.gamma
        out[f"{prefix}blk{i}_hidden_crc"] = np.int64(crc(blk.hidden))
        out[f"{prefix}blk{i}_steps"] = np.stack([blk.burn_in_steps, blk.learning_steps, blk.forward_steps])
        out[f"{prefix}blk{i}_prio"] = prio
        out[f"{prefix}blk{i}_ep"] = np.float64(-1.0 if ep is None else ep)


def batch_to_out(prefix, data, out):
    names = ["obs", "last_action", "last_reward", "hidden", "action", "n_step_reward", "gamma",
             "burn_in", "learning", "forward", "idxes", "is_weights", "old_ptr", "env_steps"]
    for name, val in zip(names, data):
        v = val.numpy() if isinstance(val, torch.Tensor) else np.asarray(val)
        if name in ("obs", "last_action", "hidden"):
            out[f"{prefix}{name}_crc"] = np.int64(crc(np.ascontiguousarray(v)))
            out[f"{prefix}{name}_shape"] = np.array(v.shape, dtype=np.int64)
        else:
            out[f"{prefix}{name}"] = v


def gen_replay(ref):
    out = {}
    rb, blocks = build_reference_replay(ref, synth.RAGGED_SCRIPT, num_blocks=8, batch_size=8)
    block_meta("", blocks, out)
    out["tree_after_add"] = rb.priority_tree.ptree.copy()
    np.random.seed(7)
    data = rb.sample_batch()
    batch_to_out("s0_", data, out)
    # stale masks, worker.py:247-256: equal / ptr>old / ptr<old
    idx = np.array([0, 5, 12, 23, 31, 44, 52, 61], dtype=np.int64)
    td = np.linspace(0.2, 1.7, len(idx)).astype(np.float32)
    out["upd_idx"], out["upd_td"] = idx, td
    for tag, old_ptr in (("eq", rb.block_ptr), ("gt", 2), ("lt", 7)):
        rb2, _ = build_reference_replay(ref, synth.RAGGED_SCRIPT, num_blocks=8, batch_size=8)
        rb2.update_priorities(idx, td, old_ptr, 0.0)
        out[f"upd_{tag}_tree"] = rb2.priority_tree.ptree.copy()
        out[f"upd_{tag}_old_ptr"] = np.int64(old_ptr)
    out["block_ptr"] = np.int64(rb.block_ptr)
    np.savez_compressed(os.path.join(OUT, "replay_ragged.npz"), **out)
    print("replay_ragged.npz", len(out), "arrays")


def run_reference_learner(ref, batches, params, K):
    w, m = ref.worker, ref.model
    net = m.Network(A)
    net.load_state_dict(params)
    rec = dict(qn=[], q=[], grads=[], params=[])
    orig_q_, orig_q = m.Network.calculate_q_, m.Network.calculate_q
    orig_clip = torch.nn.utils.clip_grad_norm_

    def q__(self, *a, **k):
        r = orig_q_(self, *a, **k)
        rec["qn"].append(r.detach().clone())
        return r

    def q_(self, *a, **k):
        r = orig_q(self, *a, **k)
        rec["q"].append(r.detach().clone())
        return r

    m.Network.calculate_q_, m.Network.calculate_q = q__, q_
    learner_box = {}

    def clip(parameters, max_norm, *a, **k):
        plist = list(parameters)
        names = [n for n, _ in learner_box["l"].online_net.named_parameters()]
        rec["grads"].append({n: p.grad.detach().clone() for n, p in zip(names, plist)})
        return orig_clip(plist, max_norm, *a, **k)

    w.nn.utils.clip_grad_norm_ = clip
    try:
        ref.config.training_steps = K
        pq = queue.Queue()
        learner = w.Learner(queue.Queue(), pq, net)
        learner_box["l"] = learner
        learner.batched_data = list(batches)
        ref.captured_td.clear()
        # snapshot params after every update through the priority queue hook
        orig_put = pq.put

        def put(item):
            rec["params"].append({k: v.detach().clone() for k, v in learner.online_net.state_dict().items()})
            orig_put(item)
        pq.put = put
        learner.run()
    finally:
        m.Network.calculate_q_, m.Network.calculate_q = orig_q_, orig_q
        w.nn.utils.clip_grad_norm_ = orig_clip
    results = [pq.get() for _ in range(K)]
    return results, rec, [t.copy() for t in ref.captured_td]


def gen_learner(ref, name, script, num_blocks, batch_size, K, bl, ls, bi, fs, seed0):
    cfg = ref.config
    saved = (cfg.block_length, cfg.learning_steps, cfg.burn_in_steps, cfg.forward_steps)
    cfg.block_length, cfg.learning_steps, cfg.burn_in_steps, cfg.forward_steps = bl, ls, bi, fs
    try:
        rb, blocks = build_reference_replay(ref, script, num_blocks, batch_size, bl, ls, bi, fs)
        batches = []
        out = {}
        for k in range(K):
            np.random.seed(seed0 + k)
            data = rb.sample_batch()
            batches.append(data)
            batch_to_out(f"k{k}_", data, out)
        params = init_params(A, seed=3)
        # Network captures config.forward_steps at construction (model.py:37)
        results, rec, tds = run_reference_learner(ref, batches, params, K)
        for k, (idxes, prio, old_ptr, loss) in enumerate(results):
            out[f"k{k}_out_idxes"] = np.asarray(idxes)
            out[f"k{k}_out_priorities"] = np.asarray(prio)
            out[f"k{k}_out_loss"] = np.float64(loss)
            out[f"k{k}_out_td"] = tds[k]
            out[f"k{k}_out_qn_online"] = rec["qn"][2 * k].numpy()
            out[f"k{k}_out_qn_target"] = rec["qn"][2 * k + 1].numpy()
            out[f"k{k}_out_q"] = rec["q"][k].numpy()
            for n, g in rec["grads"][k].items():
                out[f"k{k}_gradnorm_{n}"] = np.float64(g.double().norm().item())
                out[f"k{k}_gradhead_{n}"] = g.flatten()[:16].numpy().copy()
            for n, p in rec["params"][k].items():
                out[f"k{k}_psum_{n}"] = np.float64(p.double().sum().item())
                out[f"k{k}_pabs_{n}"] = np.float64(p.double().abs().sum().item())
                out[f"k{k}_phead_{n}"] = p.flatten()[:16].numpy().copy()
        out["meta"] = np.array([batch_size, K, bl, ls, bi, fs, seed0, num_blocks], dtype=np.int64)
        np.savez_compressed(os.path.join(OUT, name), **out)
        print(name, len(out), "arrays")
    finally:
        cfg.block_length, cfg.learning_steps, cfg.burn_in_steps, cfg.forward_steps = saved


CFG0_SCRIPT = [(21, 95, True), (22, 40, False), (23, 13, True)]


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.manual_seed(0)
    torch.set_num_threads(8)
    ref = ref_harness.load()
    gen_tree(ref)
    gen_tree_large(ref)
    gen_replay(ref)
    gen_learner(ref, "learner_ragged.npz", synth.RAGGED_SCRIPT, 8, 8, 3, 400, 40, 40, 5, seed0=40)
    gen_learner(ref, "learner_cfg0.npz", CFG0_SCRIPT, 8, 4, 2, 40, 8, 8, 4, seed0=60)


if __name__ == "__main__":
    sys.exit(main())
