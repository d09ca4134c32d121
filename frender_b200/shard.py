"""Host-side sharding of the scan across ranks (one process per GPU, SURVEY.md 8e).

Units (files, or record-aligned chunks of one file) are independent; a unit's key list carries
`first = (unit ordinal << 40) | read ordinal inside the unit`, so that the merged table -- counts
add, `first` takes the minimum -- is the same for every rank count and equals the reference's
first-appearance order over the whole input (F:199-205).  On the device the merge is
frb_allmerge (NCCL all-gather of the per-rank lists + a merge kernel); `merge_lists` is the same
monoid on the host, used by the CPU tests and by callers that gather lists themselves.
frb_shardmerge sends every key to one owner rank instead (`key_owner`, the host twin of the device
function of the same name); `shard_lists` / `fold_share` are that exchange on the host.

`Ranks` runs the per-rank processes of a multi-GPU scan or demux.
"""
import multiprocessing as mp
from multiprocessing.connection import wait

from ._lib import FrbError

_M64 = (1 << 64) - 1


def assign(units, rank, world):
    """Round-robin ownership: unit i belongs to rank i % world."""
    return [u for i, u in enumerate(units) if i % world == rank]


class WorkerFailed(SystemExit):
    """A rank of a multi-GPU run failed (text: what it raised) or exited without a result (text None).  frb_code is
    the FrbError code it raised, None for any other error.  A SystemExit: the command line ends with the message."""

    def __init__(self, rank, text=None, frb_code=None):
        super().__init__(f"GPU worker {rank} exited without a result" if text is None
                         else f"GPU worker {rank} failed: {text}")
        self.rank, self.frb_code = rank, frb_code


def _rank_main(target, args, conn):
    """A rank's process: target(*args, conn) sends (kind, payload) messages; what it raises goes to the parent as
    ("error", (FrbError code or None, text))."""
    try:
        target(*args, conn)
    except BaseException as exc:
        code = exc.code if isinstance(exc, FrbError) else None
        try:
            conn.send(("error", (code, str(exc) if isinstance(exc, SystemExit) else repr(exc))))
        except OSError:
            pass
    finally:
        conn.close()


class Ranks:
    """One `spawn` process per entry of `rank_args`, running target(*rank_args[rank], conn) with a duplex pipe to
    the parent.  collect() listens to all pipes and to the processes' exit at once, and raises WorkerFailed on the
    first error a rank reports or on a rank that exits without a message.  Leaving the `with` block by an exception
    stops every rank first, so that none is left waiting in a collective that can never complete; leaving it in
    any way joins every process."""

    def __init__(self, target, rank_args):
        self.target, self.rank_args = target, list(rank_args)
        self.procs, self.pipes = [], []

    def __enter__(self):
        mpc = mp.get_context("spawn")
        for args in self.rank_args:
            parent, child = mpc.Pipe(duplex=True)
            p = mpc.Process(target=_rank_main, args=(self.target, args, child))
            p.start()
            child.close()
            self.procs.append(p)
            self.pipes.append(parent)
        return self

    def __exit__(self, *exc):
        if exc[0] is not None:
            self.stop()
        for p in self.procs:
            p.join()

    def send_all(self, value):
        for conn in self.pipes:
            conn.send(value)

    def stop(self):
        """No-go to every rank, a short grace period, then terminate what is still alive."""
        for conn in self.pipes:
            try:
                conn.send(False)
            except OSError:
                pass
        for p in self.procs:
            p.join(timeout=5)
            if p.is_alive():
                p.terminate()

    def collect(self, kind):
        """One message of `kind` from every rank: their payloads, in rank order."""
        got = {}
        while len(got) < len(self.procs):
            pending = [r for r in range(len(self.procs)) if r not in got]
            ready = wait([self.pipes[r] for r in pending] + [self.procs[r].sentinel for r in pending])
            for r in pending:
                if self.pipes[r] in ready:
                    try:
                        status, payload = self.pipes[r].recv()
                    except EOFError:
                        raise WorkerFailed(r) from None
                    if status == "error":
                        code, text = payload
                        raise WorkerFailed(r, text, code)
                    assert status == kind, (r, status, kind)
                    got[r] = payload
                elif self.procs[r].sentinel in ready and not self.pipes[r].poll():
                    raise WorkerFailed(r)
        return [got[r] for r in range(len(self.procs))]


def merge_lists(lists):
    """[(key, count, first), ...] per unit -> {key: count} ordered by the smallest `first`."""
    count, first = {}, {}
    for lst in lists:
        for key, n, pos in lst:
            count[key] = count.get(key, 0) + n
            first[key] = min(first.get(key, pos), pos)
    return {k: count[k] for k in sorted(count, key=first.__getitem__)}


def _hash64(k):
    """murmur3 finaliser, as hash64() in csrc/common.cuh."""
    k ^= k >> 33
    k = (k * 0xFF51AFD7ED558CCD) & _M64
    k ^= k >> 33
    k = (k * 0xC4CEB9FE1A85EC53) & _M64
    return k ^ (k >> 33)


def key_owner(packed_key, world):
    """Owner rank of a packed key in the sharded merge (csrc/table_kernels.cuh key_owner)."""
    return (_hash64(int(packed_key)) >> 40) % world


def shard_lists(entries, world, pack):
    """[(key, count, first), ...] of one rank -> per-owner parts (what the rank sends to every peer).
    `pack` maps a key string to its packed 64-bit form."""
    parts = [[] for _ in range(world)]
    for key, n, pos in entries:
        parts[key_owner(pack(key), world)].append((key, n, pos))
    return parts


def fold_share(received):
    """What an owner does with the parts it receives: one entry per key (count: +, first: min), ordered by
    first appearance.  Returns [(key, count, first), ...]."""
    count, first = {}, {}
    for part in received:
        for key, n, pos in part:
            count[key] = count.get(key, 0) + n
            first[key] = min(first.get(key, pos), pos)
    return [(k, count[k], first[k]) for k in sorted(count, key=first.__getitem__)]
