"""How the encode path is spread over the GPUs of one box (SURVEY.md section 8e).

* Batches shard by image: rank r owns images [lo, hi) -- no data-path collective at all.
* One very large image shards by strips of whole MCU rows whose boundaries are restart boundaries
  of every scan. Each rank encodes its strip; the only exchange is the gather of the strips'
  per-scan byte pieces to rank 0 (sizes first, then one grouped batch of variable-length sends over
  NCCL/NVLink), where they are concatenated scan-major. With optimized Huffman tables the strips
  first all-reduce their symbol histograms (the tables describe the whole image).
* Without restart intervals a scan is one bit string. Strips of whole MCU rows still code on their own ranks: they
  all-gather the DC values at their edges, code their pieces against the strip in front, and store the pieces at
  their bit positions in rank 0's buffer (PeerGather.gather_bits); rank 0 adds leads, pad bits and EOI and stuffs 0xFF
  once over the joined stream (PeerGather.finish_bits).

The exchange functions work on whatever device the tensors live on: NCCL with CUDA tensors on the
B200 box, gloo with CPU tensors in the world_size-2 CPU tests.
"""
import torch
import torch.distributed as dist


def shard_batch(n_images, world, rank):
    """Contiguous, balanced image range of `rank`: sizes differ by at most one."""
    base, extra = divmod(n_images, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def assemble_pieces(pieces_by_strip):
    """pieces_by_strip[s][k] = bytes of scan k produced by strip s. The file is scan-major:
    for each scan, strips in order (strip 0's piece carries the header / SOS, the last strip's last
    piece the EOI)."""
    n_scans = len(pieces_by_strip[0])
    out = bytearray()
    for k in range(n_scans):
        for strip in pieces_by_strip:
            out += strip[k]
    return bytes(out)


def split_pieces(buf, offsets):
    return [bytes(buf[offsets[k]:offsets[k + 1]]) for k in range(len(offsets) - 1)]


def exchange_strip_histograms(hist, edge_dc, device, group=None):
    """Optimized Huffman tables with strips (include/jpegenc_b200.h, steps 2): the strips' symbol histograms
    are summed with one all-reduce (2 x 2 x 257 u32; NCCL over NVLink on the GPU box) and the DC values at
    the strip edges are all-gathered in rank order. Returns (hist_sum list, edge_dc list of world * 8)."""
    h = torch.tensor(hist, dtype=torch.int64, device=device)  # NCCL has no u32 sum; counts fit easily
    dist.all_reduce(h, op=dist.ReduceOp.SUM, group=group)
    return h.cpu().tolist(), exchange_edge_dc(edge_dc, device, group)


def exchange_edge_dc(edge_dc, device, group=None):
    """Strips without restart intervals: all-gather the strips' edge_dc arrays (8 values each) in rank order."""
    e = torch.tensor(edge_dc, dtype=torch.int32, device=device)
    world = dist.get_world_size(group)
    table = torch.empty(world * 8, dtype=torch.int32, device=device)
    dist.all_gather_into_tensor(table, e, group=group)
    return table.cpu().tolist()


def join_destinations(table, leads):
    """Strips without restart intervals. table[r][k] = bits of rank r's piece of scan k, leads[k] = bytes in front of scan
    k's data (the header for scan 0, its SOS otherwise). Returns (dest, src, total): dest[r][k] = bit position of the
    piece in the joined stream, src[r][k] = byte offset of the piece in rank r's own buffer (each piece rounded up to 16
    bytes), total = bytes of the joined stream with pad bits and EOI. The arithmetic of csrc/gather.cu, restated."""
    world, n = len(table), len(table[0])
    dest = [[0] * n for _ in range(world)]
    src = [[0] * n for _ in range(world)]
    at = 0
    for k in range(n):
        at += leads[k]
        bit = at * 8
        for r in range(world):
            dest[r][k] = bit
            bit += table[r][k]
            if k + 1 < n:
                src[r][k + 1] = src[r][k] + (table[r][k] + 127) // 128 * 16
        at = (bit + 7) // 8
    return dest, src, at + 2


def join_words(dest_bit, bits):
    """The 32-bit words of the joined stream a piece at [dest_bit, dest_bit + bits) touches: (owned, shared), owned the
    range of words wholly inside the piece (stored by the rank), shared the words it shares with a neighbour (sent
    through the side table and ORed in by rank 0)."""
    end = dest_bit + bits
    owned = range((dest_bit + 31) // 32, end // 32)
    shared = []
    if bits and dest_bit % 32:
        shared.append(dest_bit // 32)
    if bits and end % 32 and (end - 1) // 32 not in shared:
        shared.append((end - 1) // 32)
    return owned, shared


def piece_destinations(table):
    """table[r][k] = offset of rank r's piece k inside its own output (n_scans + 1 entries per rank). Returns
    (dest, total): dest[r][k] = byte offset of that piece in the assembled file -- behind every piece of the scans
    before k and behind the pieces of scan k of the ranks before r. The arithmetic of csrc/gather.cu, restated."""
    world, n = len(table), len(table[0]) - 1
    dest = [[0] * n for _ in range(world)]
    at = 0
    for k in range(n):
        for r in range(world):
            dest[r][k] = at
            at += table[r][k + 1] - table[r][k]
    return dest, at


class PeerGather:
    """Device-placed gather of the strips' pieces on rank 0 (BASELINE config 5: "peer copy, with NCCL only for that
    gather"). Set up once: rank 0 owns the target buffer, the other ranks map it through CUDA IPC (NVLink peer
    access). Every step: one NCCL all-gather of the (n_scans + 1) piece offsets -- device tensors, no host copy -- then
    each rank's kernel stores its pieces at their final scan-major offsets inside rank 0's buffer, then one barrier.
    The file is complete in rank 0's device memory; its size is read together with whatever the caller syncs on next."""

    def __init__(self, dev, capacity, rank, world, torch_device, group=None):
        import ctypes as C
        self.dev, self.rank, self.world, self.group, self.tdev = dev, rank, world, group, torch_device
        self.capacity = int(capacity)
        handle = torch.zeros(64, dtype=torch.uint8)
        ptr = C.c_void_p()
        if rank == 0:
            h = (C.c_uint8 * 64)()
            rc = dev.lib.jpgb_gather_target_create(dev.handle, self.capacity, C.byref(ptr), h)
            if rc != 0:
                raise RuntimeError("jpgb_gather_target_create: %s" % dev.last_error())
            handle = torch.tensor(list(h), dtype=torch.uint8)
        if world > 1:
            hd = handle.to(torch_device)
            dist.broadcast(hd, 0, group=group)
            handle = hd.cpu()
            if rank != 0:
                h = (C.c_uint8 * 64)(*handle.tolist())
                rc = dev.lib.jpgb_gather_target_open(dev.handle, h, C.byref(ptr))
                if rc != 0:
                    raise RuntimeError("jpgb_gather_target_open: %s" % dev.last_error())
        self.target = ptr.value
        self.n_table = None
        self.table = None
        self.total = torch.zeros(1, dtype=torch.int64, device=torch_device)

    def gather(self):
        """Call right after encode_strip_device on this rank. Asynchronous; returns nothing. After `barrier()` the file
        lies in rank 0's target buffer (self.target) and self.total[0] holds its size on every rank."""
        import ctypes as C
        d_offs = C.c_void_p()
        n_scans = C.c_uint32()
        rc = self.dev.lib.jpgb_last_piece_offsets_device(self.dev.handle, C.byref(d_offs), C.byref(n_scans))
        if rc != 0:
            raise RuntimeError("jpgb_last_piece_offsets_device: %s" % self.dev.last_error())
        self._all_gather_table(d_offs.value, n_scans.value + 1)
        rc = self.dev.lib.jpgb_gather_place_pieces(self.dev.handle, C.c_void_p(self.target), self.capacity, C.c_void_p(self.table.data_ptr()),
                                                   self.world, self.rank, C.c_void_p(self.total.data_ptr()))
        if rc != 0:
            raise RuntimeError("jpgb_gather_place_pieces: %s" % self.dev.last_error())

    def barrier(self):
        """Every rank's stores have landed in rank 0's buffer once this returns on the stream (NCCL orders it behind each
        rank's placement kernel)."""
        if self.world > 1:
            dist.all_reduce(self.total.new_zeros(1), group=self.group)

    def result(self):
        """Rank 0: the assembled file as a uint8 device tensor (a view of the target buffer). Synchronises."""
        total = int(self.total.item())
        if total > self.capacity:
            raise RuntimeError("gather target too small: %d > %d" % (total, self.capacity))
        return _device_view(self.target, total, self.tdev, "|u1") if self.rank == 0 else None

    def _all_gather_table(self, d_ptr, n):
        if self.n_table != n:
            self.table = torch.empty(self.world * n, dtype=torch.int64, device=self.tdev)
            self.n_table = n
        mine = _device_view(d_ptr, n, self.tdev)
        if self.world > 1:
            dist.all_gather_into_tensor(self.table, mine, group=self.group)
        else:
            self.table.copy_(mine)

    def gather_bits(self, encoder):
        """Bit-join mode (strips without restart intervals): call right after encoder.encode_contiguous_strip_device on
        this rank. One all-gather of the pieces' bit lengths (device tensors), then this rank's kernel stores its pieces
        at their bit positions in rank 0's buffer. Asynchronous; follow with barrier(), then finish_bits() on rank 0."""
        d_bits, n_scans = encoder.piece_bits_device()
        self._all_gather_table(d_bits, n_scans)
        encoder.join_place_bits(self.target, self.capacity, self.table.data_ptr(), self.world, self.rank)

    def finish_bits(self, encoder, width, height, color_type, hist_total=None):
        """Rank 0, after barrier(): leads, pad bits, EOI, the shared words, 0xFF stuffing. Returns the file as a uint8
        device tensor (a view of the encoder context's output, valid until its next call)."""
        d_file, n = encoder.join_finish_device(self.target, self.capacity, self.table.data_ptr(), self.world, width, height, color_type,
                                               hist_total=hist_total)
        return _device_view(d_file, n, self.tdev, "|u1")

    def close(self):
        if self.target:
            self.dev.lib.jpgb_gather_target_close(self.dev.handle, self.target, 0 if self.rank == 0 else 1)
            self.target = None


def _device_view(ptr, count, torch_device, typestr="<i8"):
    """Zero-copy torch view of device memory owned by the library."""
    class _Holder:
        pass

    h = _Holder()
    h.__cuda_array_interface__ = {"shape": (int(count),), "typestr": typestr, "data": (int(ptr), False), "version": 3}
    return torch.as_tensor(h, device=torch_device)


def gather_strip_pieces(local_bytes, piece_offsets, rank, world, device, group=None):
    """Host-orchestrated gather (works on any backend: the gloo CPU tests use it; on the B200 box PeerGather replaces it).
    local_bytes: uint8 tensor on `device` holding this rank's pieces back to back.
    Returns on rank 0 the assembled uint8 tensor of the whole file (scan-major), on other ranks None.
    Communication: one all_gather of the (n_scans + 1) offsets, then one batch of point-to-point
    transfers into rank 0 (a single grouped NCCL send/recv over NVLink; exact sizes, no padding)."""
    n = len(piece_offsets)
    mine = torch.tensor(piece_offsets, dtype=torch.int64, device=device)
    table = torch.empty(world * n, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(table, mine, group=group)
    table = table.cpu().view(world, n).tolist()
    if rank == 0:
        bufs = [local_bytes] + [torch.empty(table[r][-1], dtype=torch.uint8, device=device) for r in range(1, world)]
        ops = [dist.P2POp(dist.irecv, bufs[r], r, group) for r in range(1, world) if table[r][-1] > 0]
        if ops:
            for q in dist.batch_isend_irecv(ops):
                q.wait()
        parts = [bufs[r][table[r][k]:table[r][k + 1]] for k in range(n - 1) for r in range(world)]
        return torch.cat(parts)
    if piece_offsets[-1] > 0:
        for q in dist.batch_isend_irecv([dist.P2POp(dist.isend, local_bytes[:piece_offsets[-1]], 0, group)]):
            q.wait()
    return None
