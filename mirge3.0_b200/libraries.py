"""Annotation libraries: FASTA -> 2-bit packed device text + sorted 16-mer index.

Replaces what bowtie-build / the ``index.Libs/*.ebwt`` files provide to the reference's rounds
(mirge/libs/manifoldAlign.py:97-99,133).  Library load is set-up work, not the per-read hot path:
torch does the byte->code mapping and the sort; the k-mer extraction is a kernel (mirge_lib_kmers)."""
from __future__ import annotations

import ctypes as C
import gzip
import math
import os
from typing import Dict, List, Sequence, Tuple

import numpy as np
import torch

from . import abi
from .device import Device, MirgeError, _ptr

MIN_INDEX_K = 4  # shortest seed piece the search ever looks up (csrc/annotate.cu MIN_SEED)

# library key of each round (manifoldAlign.py:84) and the DataFrame column it fills (digest.py:253)
ROUND_LIBS = ["mirna", "hairpin", "mature_trna", "pre_trna", "snorna", "rrna", "ncrna_others", "mrna", "mirna", "spike-in"]
ROUND_COLUMNS = ["exact miRNA", "hairpin miRNA", "mature tRNA", "primary tRNA", "snoRNA", "rRNA", "ncrna others", "mRNA",
                 "isomiR miRNA", "spike-in"]
INDEX_SUFFIX = ["_mirna_", "_hairpin_", "_mature_trna", "_pre_trna", "_snorna", "_rrna", "_ncrna_others", "_mrna", "_mirna_",
                "_spike-in"]


def round_policies() -> List[abi.RoundPolicy]:
    """bowtie parameters of the ten rounds (manifoldAlign.py:85) as effective policies
    (SURVEY.md section 8a): (round, select, seed_len, seed_mm, total_mm, trim5, trim3, strip_polyT)."""
    S = abi
    n = lambda r, sel, mm: abi.RoundPolicy(r, sel, 28, mm, 2, 0, 0, 0)  # -n mm -l 28 -e 70, all-'I' qualities
    return [
        n(0, S.SELECT_LEN_LT26, 0),  # -n 0
        n(1, S.SELECT_LEN_GT25, 1),  # -n 1
        abi.RoundPolicy(2, S.SELECT_UNANNOTATED, 0, 1, 1, 0, 0, 0),  # -v 1 -a --best --strata
        abi.RoundPolicy(3, S.SELECT_UNANNOTATED, 0, 0, 0, 0, 0, 1),  # -v 0 -a --best --strata, T{3,}$ stripped
        n(4, S.SELECT_UNANNOTATED, 1),
        n(5, S.SELECT_UNANNOTATED, 1),
        n(6, S.SELECT_UNANNOTATED, 1),
        n(7, S.SELECT_UNANNOTATED, 0),
        abi.RoundPolicy(8, S.SELECT_UNANNOTATED, 0, 2, 2, 1, 2, 0),  # -5 1 -3 2 -v 2 --best
        n(9, S.SELECT_UNANNOTATED, 0),
    ]


def read_fasta(path: str) -> Tuple[List[str], List[bytes]]:
    """(names, sequences); name = header up to the first whitespace, as bowtie reports RNAME."""
    op = gzip.open if path.endswith(".gz") else open
    names: List[str] = []
    seqs: List[bytes] = []
    cur: List[bytes] = []
    with op(path, "rb") as f:
        for line in f:
            if line.startswith(b">"):
                if names:
                    seqs.append(b"".join(cur))
                hdr = line[1:].split()
                names.append(hdr[0].decode("latin-1") if hdr else "")
                cur = []
            elif names:
                cur.append(line.strip())
    if names:
        seqs.append(b"".join(cur))
    return names, seqs


def _code_luts(device):
    code = torch.zeros(256, dtype=torch.int32, device=device)
    isn = torch.ones(256, dtype=torch.int32, device=device)
    for i, ch in enumerate("ACGT"):
        for c in (ord(ch), ord(ch.lower())):
            code[c] = i
            isn[c] = 0
    return code, isn


def pack_text(text: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """uint8 ASCII bases -> (2-bit words int32[ceil(n/16)], N-mask words int32[ceil(n/32) + 1])."""
    n = text.numel()
    dev = text.device
    code_lut, n_lut = _code_luts(dev)
    npad = (n + 31) // 32 * 32
    t = torch.zeros(npad, dtype=torch.int64, device=dev)
    t[:n] = text.to(torch.int64)
    code = code_lut[t].to(torch.int64)
    isn = n_lut[t].to(torch.int64)
    isn[n:] = 0
    sh2 = (2 * torch.arange(16, device=dev, dtype=torch.int64)).unsqueeze(0)
    words = (code.view(-1, 16) << sh2).sum(dim=1)
    sh1 = torch.arange(32, device=dev, dtype=torch.int64).unsqueeze(0)
    nm = (isn.view(-1, 32) << sh1).sum(dim=1)
    to_i32 = lambda x: torch.where(x >= (1 << 31), x - (1 << 32), x).to(torch.int32)
    nm = torch.cat([to_i32(nm), torch.zeros(1, dtype=torch.int32, device=dev)])
    return to_i32(words), nm


class DeviceLibrary:
    """One library on the device: packed text, N mask, reference offsets, names, sorted k-mer index."""

    def __init__(self, dev: Device, names: Sequence[str], seqs: Sequence[bytes], key: str = ""):
        self.dev = dev
        self.key = key
        self.names = list(names)
        lens = np.fromiter((len(s) for s in seqs), dtype=np.int64, count=len(seqs))
        off = np.zeros(len(seqs) + 1, dtype=np.int64)
        np.cumsum(lens, out=off[1:])
        self.n_refs = len(seqs)
        self.n_bases = int(off[-1])
        if self.n_bases >= (1 << 32) - 64:
            raise MirgeError("library %s too large for 32-bit positions" % key)
        if len(lens) and int(lens.max()) >= (1 << 28):
            raise MirgeError("library %s has a reference longer than 2^28 bases" % key)
        self.max_ref_len = int(lens.max()) if len(lens) else 0
        self.ref_off = torch.from_numpy(off.astype(np.uint32).view(np.int32)).to(dev.tdev)
        text = torch.frombuffer(bytearray(b"".join(seqs)), dtype=torch.uint8).to(dev.tdev) if self.n_bases else \
            torch.zeros(0, dtype=torch.uint8, device=dev.tdev)
        self.packed, self.nmask = pack_text(text)
        # MIRGE_LIB_PAD_WORDS zero words after the text: the verifier may read past the last reference
        self.packed = torch.cat([self.packed, torch.zeros(abi.LIB_PAD_WORDS, dtype=torch.int32, device=dev.tdev)])
        self.idx_kmer = self.idx_pos = self.idx_bucket = self.filter = self.filter16 = None
        self.filter_bases = 0
        self.filter16_bits = 0
        self.n_idx = 0
        self.bucket_bits = 4
        # coarse position -> reference map (one entry per 64 bases) replacing a binary search over ref_off
        self.ref_block_shift = 6
        starts = torch.arange((self.n_bases >> self.ref_block_shift) + 1, device=dev.tdev, dtype=torch.int64) << self.ref_block_shift
        off_d = torch.from_numpy(off).to(dev.tdev)
        self.ref_block = (torch.searchsorted(off_d, starts, right=True) - 1).clamp_(0, max(self.n_refs - 1, 0)).to(torch.int32)
        self._build_index()

    def _base_struct(self) -> abi.Library:
        return abi.Library(self.packed.data_ptr(), self.nmask.data_ptr(), self.ref_off.data_ptr(), self.n_refs, self.n_bases,
                           0 if self.idx_kmer is None else self.idx_kmer.data_ptr(),
                           0 if self.idx_pos is None else self.idx_pos.data_ptr(), self.n_idx, self.bucket_bits,
                           0 if self.idx_bucket is None else self.idx_bucket.data_ptr(),
                           self.ref_block.data_ptr(), self.ref_block_shift, self.filter_bases,
                           0 if self.filter is None else self.filter.data_ptr(), self.filter16_bits, self.max_ref_len,
                           0 if self.filter16 is None else self.filter16.data_ptr())

    def _build_index(self):
        d = self.dev
        if self.n_bases == 0:
            self.struct = self._base_struct()
            return
        kmer = d.empty(self.n_bases, torch.int32)
        valid = d.empty(self.n_bases, torch.uint8)
        st = self._base_struct()
        d.check(d.lib.mirge_lib_kmers(d.ctx, C.byref(st), _ptr(kmer), _ptr(valid), d.stream()))
        d.launches += 1
        # prefix presence bitmap, about 16 bits per indexed position (4^f bits, f = 10..16): 128 KB for a miRNA
        # library, 32 MB for 10^7 bases, 512 MB (direct 16-mer addressing) for an mRNA library
        fb = int(min(16, max(10, math.ceil(math.log(max(16 * self.n_bases, 4), 4)))))
        self.filter = d.empty(1 << (2 * fb - 5), torch.int32)
        d.check(d.lib.mirge_lib_filter(d.ctx, _ptr(kmer), _ptr(valid), self.n_bases, fb, _ptr(self.filter), d.stream()))
        d.launches += 1
        self.filter_bases = fb
        # complete 16-mers through a hash, 64 bits per position (at most 64 MB: it has to stay in L2); a library whose
        # prefix bitmap already addresses whole 16-mers (mRNA) needs none
        n16 = int((valid >= 16).sum().item())
        if fb < 16 and n16 > 0:
            bits = int(min(29, max(16, math.ceil(math.log2(64 * n16)))))
            self.filter16 = d.empty(1 << (bits - 5), torch.int32)
            d.check(d.lib.mirge_lib_filter16(d.ctx, _ptr(kmer), _ptr(valid), self.n_bases, bits, _ptr(self.filter16), d.stream()))
            d.launches += 1
            self.filter16_bits = bits
        pos = torch.nonzero(valid >= MIN_INDEX_K).squeeze(1)
        k64 = kmer[pos].to(torch.int64) & 0xFFFFFFFF
        del kmer, valid
        # positions are ascending already, so a stable sort on the k-mer orders by (k-mer, position)
        ks, perm = torch.sort(k64, stable=True)
        pos = pos[perm]
        del k64, perm
        self.n_idx = int(ks.numel())
        to_i32 = lambda x: torch.where(x >= (1 << 31), x - (1 << 32), x).to(torch.int32)
        self.idx_kmer = to_i32(ks)
        self.idx_pos = to_i32(pos)
        del pos
        if self.n_idx == 0:
            self.idx_kmer = torch.zeros(1, dtype=torch.int32, device=d.tdev)
            self.idx_pos = torch.zeros(1, dtype=torch.int32, device=d.tdev)
        # about one index entry per bucket: most lookups of sequences that are not in the library end at
        # the bucket table (empty range) without touching the k-mer array
        bb = int(min(26, max(4, math.ceil(math.log2(max(self.n_idx, 2))) + 1)))
        self.bucket_bits = bb
        bounds = torch.arange((1 << bb) + 1, device=d.tdev, dtype=torch.int64) << (32 - bb)
        self.idx_bucket = torch.searchsorted(ks.contiguous(), bounds).to(torch.int32)
        del ks
        self.struct = self._base_struct()

    @classmethod
    def from_fasta(cls, dev: Device, path: str, key: str = "") -> "DeviceLibrary":
        names, seqs = read_fasta(path)
        return cls(dev, names, seqs, key=key or os.path.basename(path))


def _sequences_of_index(index_base: str, ebwt):
    """(names, sequences) of a library that ships as a bowtie index only.  A real ``bowtie-inspect`` on PATH is asked
    first (what the reference itself does, summary.py:776-788).  The built-in decoder (ebwt.py) is written from the
    published index layout and has never met an index built by a real bowtie-build -- a wrong base order there would
    give silently wrong annotation in every round -- so it is only used on request (MIRGE_B200_TRUST_EBWT=1), and says
    so; tests/test_tier3_real_tools.py pins it wherever bowtie-build exists."""
    import shutil
    import subprocess
    import warnings

    tool = shutil.which("bowtie-inspect")
    if tool and "mirge_b200" not in os.path.realpath(tool):  # (not the shim this package installs for summarize())
        p = subprocess.run([tool, index_base], capture_output=True, check=False)
        if p.returncode == 0 and p.stdout.startswith(b">"):
            names, seqs, cur = [], [], []
            for line in p.stdout.splitlines():
                if line.startswith(b">"):
                    if names:
                        seqs.append(b"".join(cur))
                    hdr = line[1:].split()
                    names.append(hdr[0].decode("latin-1") if hdr else "")
                    cur = []
                else:
                    cur.append(line.strip())
            seqs.append(b"".join(cur))
            return names, seqs
    if os.environ.get("MIRGE_B200_TRUST_EBWT", "0") != "1":
        raise MirgeError(
            "library %s ships as a bowtie index only and no bowtie-inspect is on PATH.  Provide the sequences as FASTA next "
            "to it (`bowtie-inspect %s > %s.fa`, on any machine that has bowtie), or set MIRGE_B200_TRUST_EBWT=1 to use the "
            "built-in .ebwt decoder, which has not been validated against an index built by a real bowtie-build."
            % (os.path.basename(index_base), index_base, index_base))
    warnings.warn("mirge_b200: decoding %s.*.ebwt with the built-in, not yet bowtie-validated decoder (MIRGE_B200_TRUST_EBWT=1); "
                  "annotation depends on it" % index_base, RuntimeWarning, stacklevel=3)
    return ebwt.decode_index(index_base)


class LibrarySet:
    """The libraries of one organism keyed by round library name (ROUND_LIBS)."""

    def __init__(self, libs: Dict[str, DeviceLibrary]):
        self.libs = libs

    def __getitem__(self, k: str) -> DeviceLibrary:
        return self.libs[k]

    def __contains__(self, k: str) -> bool:
        return k in self.libs

    @classmethod
    def from_fasta_dict(cls, dev: Device, fastas: Dict[str, Tuple[Sequence[str], Sequence[bytes]]]) -> "LibrarySet":
        return cls({k: DeviceLibrary(dev, n, s, key=k) for k, (n, s) in fastas.items()})

    @classmethod
    def from_mirge_lib(cls, dev: Device, libraries_path: str, organism: str, ref_db: str, spike_in: bool = False) -> "LibrarySet":
        """Locate the libraries the way bwtAlign addresses its indexes (manifoldAlign.py:97-98,115-117,133):
        <libraries_path>/<organism>/index.Libs/<organism><suffix>[<ref_db>].  Sequences come from the FASTA
        of the same basename (index.Libs or fasta.Libs, .fa/.fasta[.gz]) or, when only the bowtie index
        ships, from decoding <basename>.{1,3,4}.ebwt (ebwt.py)."""
        from . import ebwt

        out: Dict[str, DeviceLibrary] = {}
        base = os.path.join(libraries_path, organism)
        for rnd, key in enumerate(ROUND_LIBS):
            if key in out or (key == "spike-in" and not spike_in):
                continue
            name = organism + INDEX_SUFFIX[rnd] + (ref_db if rnd in (0, 1, 8) else "")
            found = None
            for sub in ("index.Libs", "fasta.Libs"):
                for ext in (".fa", ".fasta", ".fa.gz", ".fasta.gz"):
                    p = os.path.join(base, sub, name + ext)
                    if os.path.exists(p):
                        found = p
                        break
                if found:
                    break
            if found:
                out[key] = DeviceLibrary.from_fasta(dev, found, key=key)
                continue
            eb = os.path.join(base, "index.Libs", name)
            if os.path.exists(eb + ".1.ebwt"):
                names, seqs = _sequences_of_index(eb, ebwt)
                out[key] = DeviceLibrary(dev, names, seqs, key=key)
                continue
            raise MirgeError("library %s not found under %s (no FASTA, no .ebwt index)" % (name, base))
        return cls(out)
