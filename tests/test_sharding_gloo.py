"""N>1 host logic on CPU: two `gloo` ranks shard a read batch, align their shards through the C-ABI
(host-emulation build) and gather the results on rank 0; the gathered lines must equal the oracle's
output for the unsharded batch."""
import os
import socket
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import os, sys
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch, torch.distributed as dist
import oracle_lib as O
from metagraph_b200.aligner import B200Aligner, BOSSTable, DBGSuccinctIndex, format_alignment
from metagraph_b200.config import cli_defaults
from metagraph_b200.sharding import align_sharded, shard_range
EMU = os.path.join(ROOT, "tests", "emu", "build", "libmgb_emu.so")
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
rng = np.random.default_rng(5)
genome = "".join(np.array(list("ACGT"))[rng.integers(0, 4, 20000)])
comp = str.maketrans("ACGT", "TGCA")
reads = []
for i in range(37):
    p = int(rng.integers(0, len(genome) - 100)); r = genome[p:p + 100]
    reads.append((("r%d" % i), r.translate(comp)[::-1] if i % 3 == 0 else r))
k = 21
boss = BOSSTable.from_sequences(k, [genome], lib=EMU)
idx = DBGSuccinctIndex(boss, lib=EMU)
cfg = cli_defaults(k)
lines = align_sharded(B200Aligner(idx, cfg), reads, lambda h, r: format_alignment(h, r, 0, with_nodes=True))
# entries need not be single lines (ADVICE r1: JSON output has one line per alternative alignment)
multi = align_sharded(B200Aligner(idx, cfg), reads, lambda h, r: h + "\n" + format_alignment(h, r, 0))
assert shard_range(37, 0, 2) == (0, 18) and shard_range(37, 1, 2) == (18, 37)
if rank == 0:
    g = O.OracleGraph(k, [genome])
    exp = g.align_tsv(cfg, [s for _, s in reads], headers=[h for h, _ in reads], with_nodes=True)
    assert lines == exp, (len(lines), len(exp))
    assert len(multi) == len(reads) and all(m.split("\n")[0] == h for m, (h, _) in zip(multi, reads))
    print("SHARDING_OK", len(lines))
else:
    assert lines is None
dist.destroy_process_group()
'''


def test_two_rank_sharding_gloo(tmp_path):
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "emu")], stdout=subprocess.DEVNULL)
    script = tmp_path / "worker.py"
    script.write_text("ROOT = %r\n" % ROOT + WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", OMP_NUM_THREADS="1")
    with socket.socket() as s:   # a free port: other jobs on the host may hold any fixed one
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)],
                         capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    assert "SHARDING_OK 37" in out.stdout
