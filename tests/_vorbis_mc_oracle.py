"""The Vorbis front-end oracle (oracle/vorbis_frontend_oracle.py) for streams of any channel count.  TEST INFRASTRUCTURE ONLY.

The oracle's `decode` returns two planes, which is what the two-plane front-end writes; everything else in it (bit reader,
codebooks, floors, the residue reader and its partition-class vector) already loops over the stream's channels and coupling list.
This subclass only changes the layout of `decode`'s result: one plane per channel (at least two), lib.rs:146-250 otherwise
unchanged."""
import numpy as np

from oracle import packetizer_oracle as po
from oracle.vorbis_frontend_oracle import End, PacketBits
from oracle.vorbis_frontend_oracle import VorbisFrontend as _TwoPlane


class VorbisFrontend(_TwoPlane):
    def decode(self, packet, slot):
        """lib.rs:146-250.  Returns dict(block_flag, prev_block_flag, do_not_decode[P], floor[P] (index or None), floor_y [P][65],
        residue [P][slot] f32) with P = max(2, channels), or raises ReaderError for what the reference returns as an error."""
        pb = PacketBits(packet)
        try:
            if pb.read_bool():
                raise po.ReaderError(po.DECODE, "not an audio packet")
            modes = self.setup["modes"]
            mode_number = pb.read(po.ilog(len(modes) - 1))
            if mode_number >= len(modes):
                raise po.ReaderError(po.DECODE, "mode number")
            long_block, mapping_idx = modes[mode_number]
            if long_block:
                pb.read_bool(), pb.read_bool()
        except End:
            raise po.ReaderError(po.DECODE, "packet header cut")
        mapping = self.setup["mappings"][mapping_idx]
        bs_exp = self.ident["bs1_exp"] if long_block else self.ident["bs0_exp"]
        n_ch = self.ident["n_channels"]
        planes = max(2, n_ch)
        floor_y = np.zeros((planes, 65), dtype=np.uint16)
        residue = [np.zeros(slot, dtype=np.float32) for _ in range(planes)]
        dnd, floor_idx = [True] * planes, [None] * planes
        for ch in range(n_ch):
            fi = mapping["submaps"][mapping["multiplex"][ch]][0]
            y = self._floor(self.setup["floors"][fi], pb)
            dnd[ch] = y is None
            if y is not None:
                floor_idx[ch] = fi
                floor_y[ch, :len(y)] = y
        for mag, ang in mapping["couplings"]:
            if dnd[mag] != dnd[ang]:
                dnd[mag] = dnd[ang] = False
        for sm, (_, res_idx) in enumerate(mapping["submaps"]):
            chans = [c for c in range(n_ch) if mapping["multiplex"][c] == sm]
            if not chans:
                continue
            self._residue(self.setup["residues"][res_idx], pb, bs_exp, chans, dnd, residue)
        prev = long_block if self.prev_block_flag is None else self.prev_block_flag
        self.prev_block_flag = long_block
        return dict(block_flag=long_block, prev_block_flag=prev, do_not_decode=dnd, floor=floor_idx, floor_y=floor_y, residue=np.stack(residue))
