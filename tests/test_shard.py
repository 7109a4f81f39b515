"""Clip-wise sharding (SURVEY.md section 8e): partition properties, and the N>1 plumbing (barrier, max / sum over ranks,
per-rank host tracking of its own clips) on 2 CPU processes with the gloo backend."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_clip_range_partitions():
    from classifier_pipeline_b200.shard import clip_range, shard

    for n in (0, 1, 7, 8, 1024, 8192, 8193):
        for world in (1, 2, 3, 8):
            spans = [clip_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1
    assert shard(list(range(10)), 1, 3) == [4, 5, 6]
    with pytest.raises(ValueError):
        clip_range(4, 2, 2)


WORKER = r"""
import json, os, sys
sys.path.insert(0, {root!r})
import numpy as np
from classifier_pipeline_b200 import shard
from tests import helpers
from tests.tracking_helpers import track_clip_from_golden

dist = shard.init_distributed("gloo")
rank, _, world = shard.env_rank()
names = ["possum_raw", "hedgehog_raw", "synth0_raw", "synth1_raw", "synth2_raw", "synth3_raw"]
mine = shard.shard(names, rank, world)
tracks = 0
for n in mine:
    clip = track_clip_from_golden(n)
    tracks += len(clip.tracks)
dist.barrier()
total = shard.sum_over_ranks(tracks, dist)
slowest = shard.max_over_ranks(1.0 + rank, dist)
print(json.dumps(dict(rank=rank, world=world, mine=mine, tracks=tracks, total=total, slowest=slowest)))
dist.destroy_process_group()
"""


def free_port():
    """A port no other process on the host listens on (a fixed one can be taken on a shared machine)."""
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_two_ranks_gloo(tmp_path):
    from tests.tracking_helpers import track_clip_from_golden

    script = tmp_path / "worker.py"
    script.write_text(WORKER.format(root=ROOT))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(free_port()), WORLD_SIZE="2", PYTHONPATH=ROOT)
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r), LOCAL_RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.PIPE, text=True) for r in range(2)]
    outs = []
    for p in procs:
        out, err = p.communicate(timeout=300)
        assert p.returncode == 0, err[-2000:]
        outs.append(json.loads(out.strip().splitlines()[-1]))
    outs.sort(key=lambda o: o["rank"])
    assert outs[0]["mine"] + outs[1]["mine"] == ["possum_raw", "hedgehog_raw", "synth0_raw", "synth1_raw", "synth2_raw", "synth3_raw"]
    expected = sum(len(track_clip_from_golden(n).tracks) for n in outs[0]["mine"] + outs[1]["mine"])
    assert outs[0]["total"] == outs[1]["total"] == expected == outs[0]["tracks"] + outs[1]["tracks"]
    assert outs[0]["slowest"] == outs[1]["slowest"] == 2.0
