"""Multi-GPU sharding of the AES-GCM path (SURVEY 8(e)); one process per GPU.

Two regimes, matching the structure of the algorithm rather than inventing
communication:

* independent messages: `batch_split` hands each rank a contiguous message range;
  there is NO data-path collective.
* one large message: `shard_plan` splits the CT block range into contiguous
  counter ranges.  Rank r runs the fused kernel on its range with counter start
  2 + first_block (src/aes_icb.vhd:100) and gets a 16-byte GHASH partial already
  scaled by H^(blocks after the shard) (agcm_stream_part).  One all_gather of 16
  bytes per rank (NCCL over NVLink; NCCL has no XOR reduction, so gather + XOR
  inside agcm_stream_finish) and any rank can finish the tag.  The combine rests
  on the linearity the reference itself uses at src/gcm_ghash.vhd:317-344.
"""
from dataclasses import dataclass


@dataclass(frozen=True)
class Shard:
    rank: int
    first_block: int    # index of the shard's first 16-byte block in the message
    byte_offset: int
    n_bytes: int        # bytes in this shard (only the last non-empty shard may be ragged)
    blocks_after: int   # CT blocks of the message that follow this shard


def shard_plan(n_bytes, world_size):
    """Contiguous, block-aligned counter ranges; empty shards allowed when the
    message has fewer blocks than ranks."""
    if n_bytes < 0 or world_size < 1:
        raise ValueError("bad shard request")
    blocks = (n_bytes + 15) // 16
    if blocks > 0xFFFFFFFE:
        raise OverflowError("more than 2^32-2 blocks under one IV (src/aes_icb.vhd:114)")
    per = (blocks + world_size - 1) // world_size
    plan = []
    for r in range(world_size):
        fb = min(r * per, blocks)
        nb = min(per, blocks - fb)
        off = fb * 16
        nbytes = max(0, min(n_bytes - off, nb * 16))
        plan.append(Shard(r, fb, off, nbytes, blocks - fb - nb))
    return plan


def batch_split(n_msgs, world_size, rank):
    """[lo, hi) message range of `rank` (balanced to within one message)."""
    base, rem = divmod(n_msgs, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def gather_partials(partial16, group=None):
    """all_gather of one 16-byte uint8 tensor per rank -> [world, 16] tensor on the
    same device (NCCL for CUDA tensors, gloo for CPU tensors in the host tests)."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    out = torch.empty((world, 16), dtype=torch.uint8, device=partial16.device)
    dist.all_gather_into_tensor(out.view(-1), partial16.contiguous().view(-1), group=group)
    return out


def stream_crypt_sharded(engine, decrypt, iv, aad, shard, data_in, data_out, total_bytes, tag, ok=None, group=None,
                         stream=None):
    """Rank-local part + gather + finish.  `data_in`/`data_out` hold THIS rank's
    shard (CUDA uint8, shard.n_bytes long); `aad` is the full AAD (CUDA uint8 or
    None) on every rank; every rank ends up with the tag / ok flag."""
    import torch
    part = torch.empty(16, dtype=torch.uint8, device=data_in.device)
    engine.stream_part_device(decrypt, iv, shard.first_block, data_in, data_out, shard.blocks_after, part,
                              n_bytes=shard.n_bytes, stream=stream)
    parts = gather_partials(part, group)
    engine.stream_finish_device(decrypt, iv, parts, parts.shape[0], aad, total_bytes, tag, ok, stream=stream)
    return parts


class PeerExchange:
    """Peer-memory (NVLink) exchange buffers for `GcmEngine.stream_crypt_peer_device`.

    Each rank's engine exports its own small exchange buffer as a CUDA IPC handle (`peer_export`); the
    handles go round the group once (`all_gather_object`), every engine maps the others' buffers
    (`peer_import`), and the ranks barrier once.  After that a sharded message costs one bulk kernel per
    rank plus a one-warp finish on the engine's side stream, and no collective call: the 16-byte partials
    cross NVLink as plain stores from the bulk kernel's tail (src/gcm_ghash.vhd:317-344 linearity).
    `close()` unmaps the peers' buffers on every rank before any engine is closed.
    """

    def __init__(self, engine, group=None):
        import torch
        import torch.distributed as dist
        self.group = group if group is not None else dist.group.WORLD
        self.rank, self.world = dist.get_rank(self.group), dist.get_world_size(self.group)
        handles = [None] * self.world
        dist.all_gather_object(handles, engine.peer_export(), group=self.group)
        engine.peer_import(self.rank, self.world, handles)
        dist.barrier(self.group)   # every buffer is zeroed before anyone stores into it
        torch.cuda.synchronize(torch.device("cuda", engine.device))
        self.engine = engine

    def close(self):
        """Leave the exchange: unmap the peers' buffers, then barrier, so that no rank frees its buffer (by closing its
        engine) while another still maps it."""
        import torch.distributed as dist
        self.engine.peer_close()
        dist.barrier(self.group)

    def crypt(self, decrypt, iv, aad, shard, data_in, data_out, total_bytes, tag, ok=None, stream=None, defer=False):
        """This rank's shard of one message.  defer=True keeps the ranks free-running (the finish of
        message k overlaps the bulk kernel of message k+1); `join()` before `tag` / `ok` are read.
        A rank that never posts makes the others fail closed (zero tag, ok = 0) after the timeout;
        every later call then raises AgcmError(E_PEER_TIMEOUT), and `check()` raises at once."""
        self.engine.stream_crypt_peer_device(decrypt, iv, shard.first_block, data_in if shard.n_bytes else None,
                                             data_out if shard.n_bytes else None, shard.blocks_after, aad, total_bytes, tag,
                                             ok, n_bytes=shard.n_bytes, stream=stream, defer=defer)

    def crypt_host(self, decrypt, iv, aad, shard, h_in, h_out, total_bytes, tag=None):
        """The same for a shard held in (pinned) HOST memory: chunked H2D / kernel / D2H, the rank's
        partial posted to the peers, tag (encrypt) or ok flag (decrypt) returned on every rank."""
        return self.engine.stream_crypt_peer_host(decrypt, iv, shard.first_block, h_in[:shard.n_bytes], h_out[:shard.n_bytes],
                                                  shard.blocks_after, aad, total_bytes, tag)

    def decrypt_verified(self, iv, aad, shard, ct, pt, total_bytes, tag, ok, stream=None):
        """Verify-then-release decrypt of this rank's shard: ok[0] = 1 on every rank if and only if the whole message's
        tag matches, and no rank writes any plaintext otherwise.  `ok` and `pt` are valid in stream order (no join)."""
        self.engine.stream_decrypt_verified_peer_device(iv, shard.first_block, ct if shard.n_bytes else None,
                                                        pt if shard.n_bytes else None, shard.blocks_after, aad, total_bytes,
                                                        tag, ok, n_bytes=shard.n_bytes, stream=stream)

    def decrypt_verified_host(self, iv, aad, shard, h_ct, h_pt, total_bytes, tag):
        """The same for a shard in (pinned) HOST memory.  -> ok; on False h_pt is untouched."""
        return self.engine.stream_decrypt_verified_peer_host(iv, shard.first_block, h_ct[:shard.n_bytes], h_pt[:shard.n_bytes],
                                                             shard.blocks_after, aad, total_bytes, tag)

    def join(self, stream=None):
        self.engine.peer_join(stream)

    def check(self):
        """Synchronise the finishes issued so far and raise if any of them timed out."""
        if self.engine.peer_timed_out():
            from . import _lib
            raise _lib.AgcmError(_lib.E_PEER_TIMEOUT)
