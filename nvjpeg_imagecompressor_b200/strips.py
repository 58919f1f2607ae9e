"""Multi-GPU encode of ONE image as MCU-row strips, one process (rank) per GPU, torch.distributed for the plumbing.

Not in the reference (single GPU, no communication: SURVEY.md 2a); this is BASELINE.json's multi-GPU design
(SURVEY.md 8e). Per image every rank runs the staged C-ABI on its strip and the ranks exchange three small things:

  1. all_gather  last DC of each strip (3 x int16)        -> DC predictors at the next strip's start
  2. all_reduce  4 x 257 symbol counts (optimized Huffman) -> identical tables on every rank
  3. all_gather  (strip bit count, first 32 bits)          -> global bit phase of each strip and the bits that
                                                              complete the previous strip's last byte

Strip k then byte-stuffs its own bits shifted to phase G_k mod 8; it owns every output byte whose FIRST bit it holds,
so the concatenation [headers | strip 0 | ... | strip N-1 | EOI] is the single-GPU stream, byte for byte.

On GPUs (EngineBackend) the three exchanges are folded into ONE all_gather of a 4 KB record per strip (its own symbol
counts, first/last DCs, first tokens: include/b2jpeg.h b2j_strip_record): with every strip's counts and the final code
lengths each rank computes every strip's bit count itself, so nothing waits for another rank's entropy coder
(`phase1x` -> all_gather -> `phase2x`). When the GPUs can map each other's memory (CUDA IPC, one node) even that
collective goes: `phase1x` stores the record into every rank's arena over NVLink and raises a flag, `phase2x` waits for
the world's flags (B2J_STRIP_EXCHANGE=nccl keeps the all_gather). The three-step schedule above is what the host-visible phases implement and
what the CPU tests drive.

`backend` abstracts the device: EngineBackend drives libb2jpeg.so on a GPU; the CPU tests plug a checker-backed
backend into the same host logic over gloo.
"""
import os

import numpy as np
import torch
import torch.distributed as dist

from . import _native as N
from .engine import B2JError

_HS = {0: 1, 1: 2, 2: 1, 3: 2, 4: 4}
_VS = {0: 1, 1: 1, 2: 2, 3: 2, 4: 1}


def strip_rows(H, css, world):
    """Pixel-row range [y0, y1) of every rank: contiguous MCU rows, as even as possible."""
    mcu_h = 8 * _VS[css]
    mcuy = (H + mcu_h - 1) // mcu_h
    base, rem = divmod(mcuy, world)
    out, m0 = [], 0
    for r in range(world):
        n = base + (1 if r < rem else 0)
        out.append((min(H, m0 * mcu_h), min(H, (m0 + n) * mcu_h)))
        m0 += n
    return out


def seam_params(strip_bits, first_words):
    """strip_bits[k], first_words[k] (top-aligned first 32 bits) -> per strip (skip_bits, ext_byte)."""
    n = len(strip_bits)
    out, G = [], 0
    for k in range(n):
        skip = (8 - G % 8) % 8
        ext = 0xFF if k == n - 1 else (int(first_words[k + 1]) >> 24) & 0xFF
        out.append((skip, ext))
        G += int(strip_bits[k])
    return out


class _CudaView:
    """Zero-copy torch view of device memory owned by the C library (CUDA array interface)."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (int(ptr), False), "version": 3}


def _view(ptr, shape, typestr, device):
    return torch.as_tensor(_CudaView(ptr, shape, typestr), device=device)


class EngineBackend:
    """Strip phases on one GPU through the C-ABI (b2j_strip_*)."""

    def __init__(self, W, rows_max, quality, optimize, css, device):
        from .engine import Engine
        self.device = torch.device("cuda", device)
        self.eng = Engine(W, rows_max, quality, optimize, css, device=device)
        st = self.eng.strip_state()
        self.hist = _view(st.d_hist, (4 * 257,), "<i4", self.device)
        self.last_dc = _view(st.d_last_dc, (4,), "<i2", self.device)
        self.pred_in = _view(st.d_pred_in, (4,), "<i2", self.device)
        self.strip_bits = _view(st.d_strip_bits, (2,), "<i8", self.device)
        self.out_len = _view(st.d_out_len, (1,), "<i8", self.device)
        self._d_out = st.d_out
        self.record = _view(st.d_record, (N.STRIP_RECORD_BYTES,), "|u1", self.device)

    def set_stream(self, s):
        self.eng.set_stream(s)

    def phase1(self, d_ptr, step, W, rows):
        self.eng.strip_phase1(d_ptr, step, W, rows)

    def phase1b(self):
        self.eng.strip_phase1b()

    def phase2(self, W, H):
        self.eng.strip_phase2(W, H)

    def phase3(self, skip, ext, flags):
        self.eng.strip_phase3(skip, ext, flags)

    def phase3_dev(self, bits_all, rank, world, flags):
        """bits_all: device int64 [world][2] (all-gathered strip_bits); the seam is derived on the device."""
        self.eng.strip_phase3_dev(bits_all.data_ptr(), rank, world, flags)

    def phase1x(self, d_ptr, step, W, rows):
        self.eng.strip_phase1x(d_ptr, step, W, rows)

    def phase2x(self, records_all, rank, world, W, H, flags):
        """records_all: device uint8 [world][STRIP_RECORD_BYTES], the all-gathered `record`s in strip order."""
        self.eng.strip_phase2x(None if records_all is None else records_all.data_ptr(), rank, world, W, H, flags)

    def out_view(self, n):
        return _view(self._d_out, (int(n),), "|u1", self.device)


class StripEncoder:
    def __init__(self, W, H, quality=95, optimize=True, css="422", rank=None, world=None, backend=None, device=None,
                 group=None, peer=None):
        self.W, self.H = W, H
        self.css = N.CSS[css] if isinstance(css, str) else int(css)
        if self.css == N.CSS_GRAY:
            raise B2JError(-1, "StripEncoder: gray images are not supported (the strips' records and seams assume three components)")
        self.optimize = bool(optimize)
        self.group = group
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world = dist.get_world_size(group) if world is None else world
        self.rows = strip_rows(H, self.css, self.world)
        self.y0, self.y1 = self.rows[self.rank]
        if backend is None:
            dev = torch.cuda.current_device() if device is None else device
            backend = EngineBackend(W, max(y1 - y0 for y0, y1 in self.rows), quality, optimize, self.css, dev)
        self.b = backend
        dev = self.b.last_dc.device
        self._dc_all = torch.zeros((self.world, 4), dtype=torch.int16, device=dev)
        self._bits_all = torch.zeros((self.world, 2), dtype=torch.int64, device=dev)
        self._len_all = torch.zeros((self.world, 1), dtype=torch.int64, device=dev)
        self.one_collective = hasattr(self.b, "phase2x") and self.world > 1
        self.exchange = "three collectives"
        if self.one_collective:
            self._rec_all = torch.zeros((self.world, N.STRIP_RECORD_BYTES), dtype=torch.uint8, device=dev)
            self.exchange = "one all_gather"
            if peer is None:
                peer = os.environ.get("B2J_STRIP_EXCHANGE", "peer") == "peer"
            if peer and self._connect_peers():
                self.exchange = "peer memory"

    def _connect_peers(self):
        """Map every rank's exchange arena (CUDA IPC) so that records travel as plain NVLink stores. All ranks decide
        together: one rank that cannot map a peer sends everybody back to the all_gather schedule."""
        b, w, r = self.b, self.world, self.rank
        ok, arenas = 1, [None] * w
        try:
            handle, _ = b.eng.peer_export()
            handles = [None] * w
            dist.all_gather_object(handles, handle, group=self.group)
            for k in range(w):
                if k != r:
                    arenas[k] = b.eng.peer_open(handles[k])
        except Exception:
            ok = 0
        t = torch.tensor([ok], dtype=torch.int32, device=b.last_dc.device)
        dist.all_reduce(t, op=dist.ReduceOp.MIN, group=self.group)
        if int(t.item()) == 0:
            return False
        b.eng.peer_connect(r, w, arenas)
        dist.barrier(group=self.group)   # nobody pushes before every arena is mapped and zeroed
        return True

    def encode_strip(self, d_ptr, step):
        """d_ptr: this rank's strip (rows [y0, y1) of the image). Returns (stuffed byte count, all ranks' counts)."""
        b, w, r = self.b, self.world, self.rank
        flags = (1 if r == 0 else 0) | (2 if r == w - 1 else 0)
        if self.one_collective:
            b.phase1x(d_ptr, step, self.W, self.y1 - self.y0)
            if self.exchange == "peer memory":   # phase1x already stored the record into every rank's arena
                b.phase2x(None, r, w, self.W, self.H, flags)
                return b.out_len
            dist.all_gather_into_tensor(self._rec_all.view(-1), b.record, group=self.group)
            b.phase2x(self._rec_all, r, w, self.W, self.H, flags)
            return b.out_len
        b.phase1(d_ptr, step, self.W, self.y1 - self.y0)
        if w > 1:
            dist.all_gather_into_tensor(self._dc_all.view(torch.uint8).view(-1), b.last_dc.view(torch.uint8), group=self.group)
            if r > 0:
                b.pred_in.copy_(self._dc_all[r - 1])
            else:
                b.pred_in.zero_()
        else:
            b.pred_in.zero_()
        b.phase1b()
        if w > 1 and self.optimize:
            dist.all_reduce(b.hist, op=dist.ReduceOp.SUM, group=self.group)
        b.phase2(self.W, self.H)
        if w > 1:
            dist.all_gather_into_tensor(self._bits_all.view(-1), b.strip_bits, group=self.group)
            if hasattr(b, "phase3_dev"):   # GPU backend: seam parameters derived on the device, no host sync
                b.phase3_dev(self._bits_all, r, w, flags)
                return b.out_len
            bits = self._bits_all.cpu().numpy()
            skip, ext = seam_params(bits[:, 0], bits[:, 1].astype(np.uint64) & 0xFFFFFFFF)[r]
        else:
            skip, ext = 0, 0xFF
        b.phase3(skip, ext, flags)
        return b.out_len

    def gather_lengths(self):
        if self.world > 1:
            dist.all_gather_into_tensor(self._len_all.view(-1), self.b.out_len, group=self.group)
            return self._len_all.cpu().numpy()[:, 0]
        return self.b.out_len.cpu().numpy()

    def gather_jpeg(self, dst=0):
        """Concatenate the strips' bytes on rank `dst` (device tensor there, None elsewhere)."""
        lens = self.gather_lengths()
        mine = self.b.out_view(int(lens[self.rank]))
        if self.world == 1:
            return mine.clone()
        if self.rank == dst:
            total = torch.empty(int(lens.sum()), dtype=torch.uint8, device=mine.device)
            off = 0
            reqs = []
            for k in range(self.world):
                part = total[off:off + int(lens[k])]
                if k == dst:
                    part.copy_(mine)
                else:
                    reqs.append(dist.irecv(part, src=k, group=self.group))
                off += int(lens[k])
            for q in reqs:
                q.wait()
            return total
        dist.send(mine.contiguous(), dst=dst, group=self.group)
        return None


class StripSecondary:
    """Secondary compression of ONE image on N GPUs (BASELINE.json config 4): encode -> reconstruct -> difference map ->
    encode(difference) + PSNR, every step on the rank's own MCU-row strip; both JPEG streams are stitched single-image
    streams (two StripEncoders), the PSNR comes from an all_reduce of the strips' exact integer SSDs.

    The strip is reconstructed from the quantised coefficients its own encoder produced (b2j_reconstruct_planes /
    _color). Without vertical subsampling (444 / 422 / 411) that needs no exchange: quantisation, IDCT and the
    horizontal triangle upsampling never look across an MCU row, so the strip gives exactly the rows the whole image's
    decode would give (tests/test_gpu_strips.py). 420 / 440 upsample vertically with a filter that looks one chroma row
    across the strip border: neighbouring ranks swap that one Cb and one Cr row (a point-to-point exchange of
    2 * ceil(W / hs) bytes per border, dist.batch_isend_irecv) between the IDCT and the colour step.
    """

    def __init__(self, W, H, quality=95, optimize=True, css="422", diff_mode=1, rank=None, world=None, device=None,
                 group=None):
        from .engine import Engine
        self.W, self.H, self.mode, self.group = W, H, int(diff_mode), group
        css_id = N.CSS[css] if isinstance(css, str) else int(css)
        if css_id == N.CSS_GRAY:
            raise B2JError(-1, "StripSecondary: gray images are not supported")
        self.enc1 = StripEncoder(W, H, quality, optimize, css_id, rank, world, None, device, group)
        self.enc2 = StripEncoder(W, H, quality, optimize, css_id, rank, world, None, device, group)
        self.rank, self.world = self.enc1.rank, self.enc1.world
        self.y0, self.y1 = self.enc1.y0, self.enc1.y1
        # halo exchange partners: only for a vertical chroma filter; ranks without rows (world > MCU rows) sit at the tail
        rows = self.enc1.rows
        vert = _VS[css_id] != 1 and self.y1 > self.y0
        self.halo_top = vert and self.rank > 0
        self.halo_bottom = vert and self.rank + 1 < self.world and rows[self.rank + 1][1] > rows[self.rank + 1][0]
        rows_max = max(b - a for a, b in self.enc1.rows)
        dev = self.enc1.b.device
        self.recon = torch.empty((rows_max, W, 3), dtype=torch.uint8, device=dev)
        self.diff = torch.empty((rows_max, W, 3), dtype=torch.uint8, device=dev)
        self._ssd = torch.zeros(1, dtype=torch.int64, device=dev)
        # the primary encoder keeps its quantised coefficients: the strip is reconstructed from them (no entropy decode)
        self.enc1.b.eng.set_debug(1)
        # one stream for the two encoder states and torch's copies / collectives
        self.stream = torch.cuda.Stream(device=dev)
        for e in (self.enc1.b.eng, self.enc2.b.eng):
            e.set_stream(self.stream.cuda_stream)

    def run(self, d_ptr, step):
        """d_ptr: this rank's strip (rows [y0, y1)), pitch W*3. -> (primary strip bytes, secondary strip bytes, PSNR);
        the byte counts are device tensors, the strips' bytes are in enc1.b / enc2.b (gather_jpeg stitches them)."""
        assert step == self.W * 3, "the difference map runs over contiguous rows"
        self.stream.wait_stream(torch.cuda.current_stream(self.recon.device))
        with torch.cuda.stream(self.stream):
            return self._run(d_ptr, step)

    def _run(self, d_ptr, step):
        rows, W = self.y1 - self.y0, self.W
        n1 = self.enc1.encode_strip(d_ptr, step)
        # the strip's pixels as every decoder will reconstruct them: de-quantise + IDCT + upsample of the coefficients
        # the encoder just produced (b2j_reconstruct_device) -- nothing is encoded twice, decoded or sent to the host
        eng = self.enc1.b.eng
        rp = eng.reconstruct_planes()
        if self.halo_top or self.halo_bottom:
            self._swap_halos(rp)
        eng.reconstruct_color(self.recon.data_ptr(), W * 3, self.halo_top, self.halo_bottom)
        ssd_ptr = self.enc2.b.eng.diff_psnr_device(d_ptr, self.recon.data_ptr(), rows * W * 3, self.mode, self.diff.data_ptr())
        self._ssd.copy_(_view(ssd_ptr, (1,), "<i8", self.recon.device))
        if self.world > 1:
            dist.all_reduce(self._ssd, op=dist.ReduceOp.SUM, group=self.group)
        n2 = self.enc2.encode_strip(self.diff.data_ptr(), W * 3)
        ssd = int(self._ssd.item())
        psnr = 20.0 * np.log10(255.0 / (np.sqrt(ssd / (self.W * self.H * 3)) + 2.220446049250313e-16))   # cv::PSNR
        return n1, n2, float(psnr)


    def _swap_halos(self, rp):
        """One chroma row each way across every strip border this rank has (Cb then Cr, the same order on both sides)."""
        dev, n = self.recon.device, int(rp.row_bytes)
        v = lambda p: _view(p, (n,), "|u1", dev)
        peer = lambda r: dist.get_global_rank(self.group, r) if self.group is not None else r
        ops = []
        if self.halo_top:
            up = peer(self.rank - 1)
            ops += [dist.P2POp(dist.isend, v(rp.cb_first), up, self.group), dist.P2POp(dist.isend, v(rp.cr_first), up, self.group),
                    dist.P2POp(dist.irecv, v(rp.cb_halo_top), up, self.group), dist.P2POp(dist.irecv, v(rp.cr_halo_top), up, self.group)]
        if self.halo_bottom:
            dn = peer(self.rank + 1)
            ops += [dist.P2POp(dist.isend, v(rp.cb_last), dn, self.group), dist.P2POp(dist.isend, v(rp.cr_last), dn, self.group),
                    dist.P2POp(dist.irecv, v(rp.cb_halo_bottom), dn, self.group), dist.P2POp(dist.irecv, v(rp.cr_halo_bottom), dn, self.group)]
        for r in dist.batch_isend_irecv(ops):
            r.wait()


# ---------------------------------------------------------------------------------------------------------------
# One image decoded by N GPUs (SURVEY.md 8f N3). A stream whose restart intervals are whole MCU rows shards without
# any data-path collective: every interval starts byte aligned at a known state with zero DC predictors, so a run of
# intervals is a baseline scan of its own. Rank k takes the k-th N-th of the scan's BYTES, finds the RSTn markers in
# it on the GPU, learns from one all_gather of the marker counts which MCU row its first interval is, and decodes
# its intervals (plus one interval above and below: the vertical chroma filter of 4:2:0 / 4:4:0 looks one chroma row
# across) through b2j_decode_scan_device with the frame height replaced by its rows. Streams without restart markers
# do not shard (the synchronisation chain spans the scan): replicas only, as DESIGN.md says.
def parse_baseline_header(jpg):
    """-> dict(W, H, css, dri, scan_off, scan_end, hs, vs) of a baseline JPEG (host bytes)."""
    b = np.asarray(jpg, np.uint8)
    p, n = 2, b.size
    out = {"dri": 0}
    while p + 4 <= n:
        if b[p] != 0xFF:
            raise ValueError("not a marker")
        m = int(b[p + 1])
        if m == 0xFF:
            p += 1
            continue
        p += 2
        if m == 0x01 or 0xD0 <= m <= 0xD8:
            continue
        L = (int(b[p]) << 8) | int(b[p + 1])
        if m in (0xC0, 0xC1):
            out["H"], out["W"] = (int(b[p + 3]) << 8) | int(b[p + 4]), (int(b[p + 5]) << 8) | int(b[p + 6])
            out["hs"], out["vs"] = int(b[p + 9]) >> 4, int(b[p + 9]) & 15
            out["sof_height_pos"] = p + 3
        elif m == 0xDD:
            out["dri"] = (int(b[p + 2]) << 8) | int(b[p + 3])
        elif m == 0xDA:
            out["scan_off"] = p + L
            end = n - 2 if (b[n - 2] == 0xFF and b[n - 1] == 0xD9) else n
            out["scan_end"] = end
            return out
        p += L
    raise ValueError("no SOS")


class StripDecoder:
    """One rank of an N-rank decode of ONE image: count_markers() -> int (all-gather it over the ranks), then
    decode(counts_of_all_ranks) -> (first row, device tensor with this rank's rows)."""

    def __init__(self, jpg, rank, world, device=None):
        from .engine import Engine
        # a (pinned) torch tensor keeps its memory kind for the uploads; numpy input is wrapped
        self.jt = jpg if torch.is_tensor(jpg) else torch.from_numpy(np.ascontiguousarray(jpg, np.uint8))
        self.jpg = self.jt.numpy()
        self.rank, self.world = int(rank), int(world)
        h = parse_baseline_header(self.jpg)
        self.h = h
        W, H, hs, vs = h["W"], h["H"], h["hs"], h["vs"]
        self.mcu_h = 8 * vs
        mcux = -(-W // (8 * hs))
        self.mcuy = -(-H // self.mcu_h)
        if h["dri"] == 0 or h["dri"] % mcux:
            raise ValueError("single-image decode over several GPUs needs restart intervals of whole MCU rows (replicas otherwise)")
        self.rpi = h["dri"] // mcux                      # MCU rows per interval
        self.nint = -(-self.mcuy // self.rpi)
        self.dev = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        css = {(1, 1): 0, (2, 1): 1, (1, 2): 2, (2, 2): 3, (4, 1): 4}[(hs, vs)]
        # the split is by bytes, so a rank's share of the rows depends on the content: twice the fair share, plus the halo
        rows_cap = min(H, (2 * -(-self.nint // self.world) + 8) * self.rpi * self.mcu_h)
        self.eng = Engine(W, rows_cap, 95, True, css, device=self.dev.index)
        self.margin = 1 << 20                            # bytes read beyond the own range on both sides (halo intervals)

    def count_markers(self):
        h, jpg = self.h, self.jpg
        s0, s1 = h["scan_off"], h["scan_end"]
        n = s1 - s0
        self.lo_own, self.hi_own = s0 + n * self.rank // self.world, s0 + n * (self.rank + 1) // self.world
        self.lo, self.hi = max(s0, self.lo_own - self.margin), min(s1, self.hi_own + self.margin)
        self.d = self.jt[self.lo:self.hi].to(self.dev, non_blocking=True)
        d = self.d
        mk = ((d[:-1] == 0xFF) & ((d[1:] & 0xF8) == 0xD0)).nonzero().flatten()
        self.mk = mk.cpu().numpy().astype(np.int64) + self.lo          # file offsets of the FF of every RSTn in the window
        self.base = int(np.searchsorted(self.mk, self.lo_own))         # markers in the lower margin come first
        self.nown = int(np.searchsorted(self.mk, self.hi_own)) - self.base
        return self.nown

    def decode(self, counts):
        h, jpg = self.h, self.jpg
        s0, s1 = h["scan_off"], h["scan_end"]
        before = int(sum(counts[: self.rank]))            # markers before my byte range = ordinal of my first marker
        # interval 0 belongs to rank 0, interval j >= 1 to the rank whose byte range holds marker j - 1
        i0 = 0 if self.rank == 0 else before + 1
        i1 = min(self.nint, before + self.nown + 1)       # exclusive
        if i1 <= i0:
            return 0, torch.empty((0, h["W"], 3), dtype=torch.uint8, device=self.dev)
        j0, j1 = max(0, i0 - 1), min(self.nint, i1 + 1)   # with one interval of halo on either side

        def start_of(j):                                  # first byte of interval j: after marker j - 1
            if j == 0:
                return s0
            idx = self.base + (j - 1 - before)
            if idx < 0 or idx >= self.mk.size:
                raise RuntimeError("a restart interval is larger than the margin read around the rank's byte range")
            return int(self.mk[idx]) + 2

        b0 = start_of(j0)
        b1 = s1 if j1 >= self.nint else start_of(j1) - 2
        rows0, rows1 = j0 * self.rpi * self.mcu_h, min(h["H"], j1 * self.rpi * self.mcu_h)
        sub = torch.empty((rows1 - rows0, h["W"], 3), dtype=torch.uint8, device=self.dev)
        self.eng.decode_scan_device(jpg[: s0], self.d.data_ptr() + (b0 - self.lo), b1 - b0, sub.data_ptr(), h["W"] * 3, rows1 - rows0)
        y0, y1 = i0 * self.rpi * self.mcu_h, min(h["H"], i1 * self.rpi * self.mcu_h)
        return y0, sub[y0 - rows0: y1 - rows0]

    def close(self):
        self.eng.close()
