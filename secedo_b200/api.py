"""Host-side mirror of the reference's interface for the hot path, on top of the C ABI.

Same names, argument order/meaning and error behaviour as the reference:

    Filter(theta, cell_proportion=4)                       util/is_significant.hpp:40-52
    Filter.is_significant(base_count)                      util/is_significant.hpp:60
    Filter.filter(pos_data, id_to_pos, marker, num_threads) -> (filtered, avg_coverage)   :68-72
    compute_similarity_matrix(pos_data, num_cells, max_fragment_length, group_id_to_pos,
        mutation_rate, homozygous_rate, seq_error_rate, num_threads, marker, normalization)
                                                           similarity_matrix.hpp:51-60

``pos_data`` is a :class:`secedo_b200.pileup.Pileup` (host CSR, the flat form of
``vector<vector<PosData>>``) or a :class:`DevicePileup` already staged in HBM. The C++ flavour of
this shim, which defines the reference's own symbols, lives in ``secedo_b200/host``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence, Tuple, Union

import numpy as np

from . import _lib
from ._lib import NORMALIZATIONS, PATHS, SgpuError, SpectralStats, Stats
from .pileup import NO_POS, Pileup


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Context:
    """One GPU. All work of a context is issued on one CUDA stream."""

    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        rc = self._lib.sgpu_init(int(device), C.byref(self._h))
        if rc != 0:
            msg = self._lib.sgpu_last_error(self._h).decode() if self._h else "sgpu_init failed"
            if self._h:
                self._lib.sgpu_shutdown(self._h)
                self._h = C.c_void_p()
            raise SgpuError(rc, msg)
        self.device = int(device)

    def check(self, rc: int) -> None:
        if rc != 0:
            raise SgpuError(rc, self._lib.sgpu_last_error(self._h).decode())

    def set_stream(self, cuda_stream: Optional[int]) -> None:
        self.check(self._lib.sgpu_set_stream(self._h, C.c_void_p(cuda_stream) if cuda_stream else None))

    def synchronize(self) -> None:
        self.check(self._lib.sgpu_synchronize(self._h))

    def output_wait(self) -> None:
        """Wait for the download started by :meth:`Counts.finalize_async`."""
        self.check(self._lib.sgpu_output_wait(self._h))

    def launch_count(self) -> int:
        """CUDA kernels launched by this context so far."""
        return int(self._lib.sgpu_launch_count(self._h))

    def set_option(self, name: str, value: int) -> None:
        """Scheduling knobs (``async_gemm`` 0 / 1, ``prefer_shared`` 0 / 1): see ``sgpu_set_option`` in
        include/secedo_b200.h. Results never depend on them."""
        self.check(self._lib.sgpu_set_option(self._h, name.encode(), int(value)))

    def tensor_times(self):
        """(ms, launches) of the first-order tensor kernels that no ``accumulate`` statistics have reported yet; waits for
        the kernels still in flight (they run on a stream of their own, beside the next batch's filter and staging)."""
        ms, n = C.c_float(0), C.c_uint64(0)
        self.check(self._lib.sgpu_tensor_times(self._h, C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def synth_pileup(self, n_cells: int, coverage: float, n_chr: int, loci_per_chr: int, *, n_clones: int = 2,
                     frac_somatic: float = 0.5, frac_germline: float = 0.1, theta: float = 0.001,
                     spacing: int = 400, p_multi: float = 0.0, p_mate: float = 0.0, p_mate_mismatch: float = 0.2,
                     seed: int = 1) -> "DevicePileup":
        """Deterministic synthetic pileup generated in HBM (csrc/synth.cu); bench-scale input."""
        sp = _lib.SynthParams(n_cells=n_cells, n_chr=n_chr, loci_per_chr=loci_per_chr, n_clones=n_clones,
                              spacing=spacing, coverage=coverage, frac_somatic=frac_somatic,
                              frac_germline=frac_germline, theta=theta, p_multi=p_multi, p_mate=p_mate,
                              p_mate_mismatch=p_mate_mismatch, seed=seed)
        h = C.c_void_p()
        self.check(self._lib.sgpu_synth_pileup(self._h, C.byref(sp), C.byref(h)))
        return DevicePileup(self, h)

    def ipc_open(self, handle: bytes) -> int:
        """Map another process's count planes (:meth:`Counts.ipc_handle`) into this process; device pointer."""
        ptr = C.c_void_p()
        self.check(self._lib.sgpu_ipc_open(self._h, C.create_string_buffer(handle, 64), C.byref(ptr)))
        return ptr.value

    def ipc_close(self, ptr: int) -> None:
        self.check(self._lib.sgpu_ipc_close(self._h, C.c_void_p(ptr)))

    def host_register(self, host_ptr: int, nbytes: int) -> int:
        """Page-lock + map host memory (e.g. a shared-memory segment); returns the device alias."""
        dev = C.c_void_p()
        self.check(self._lib.sgpu_host_register(self._h, C.c_void_p(host_ptr), int(nbytes), C.byref(dev)))
        return dev.value

    def host_unregister(self, host_ptr: int) -> None:
        self.check(self._lib.sgpu_host_unregister(self._h, C.c_void_p(host_ptr)))

    def close(self) -> None:
        if self._h:
            self._lib.sgpu_shutdown(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ staging
    def upload(self, p: Pileup) -> "DevicePileup":
        h = C.c_void_p()
        fn = self._lib.sgpu_pileup_upload_wide if p.wide else self._lib.sgpu_pileup_upload
        self.check(fn(self._h, p.n_chr, _ptr(p.chr_ptr), _ptr(p.row_ptr), _ptr(p.position), _ptr(p.read_id), _ptr(p.gid_base),
                      C.byref(h)))
        return DevicePileup(self, h)

    def upload_async(self, p: Pileup) -> "DevicePileup":
        """Upload on the context's copy stream without waiting: overlaps the kernels of the work issued
        next. The host arrays must stay alive (and should be pinned) until the pileup is first used."""
        h = C.c_void_p()
        fn = self._lib.sgpu_pileup_upload_wide_async if p.wide else self._lib.sgpu_pileup_upload_async
        self.check(fn(self._h, p.n_chr, _ptr(p.chr_ptr), _ptr(p.row_ptr), _ptr(p.position), _ptr(p.read_id), _ptr(p.gid_base),
                      C.byref(h)))
        dp = DevicePileup(self, h)
        dp._keepalive = p
        return dp

    def upload_lazy_async(self, p: Pileup) -> "DevicePileup":
        """Like :meth:`upload_async`, but the read ids stay in (pinned, mapped) host memory: the filter pulls the
        read ids of the loci it keeps over PCIe, the rejected loci's never travel."""
        h = C.c_void_p()
        self.check(self._lib.sgpu_pileup_upload_lazy_async(self._h, p.n_chr, _ptr(p.chr_ptr), _ptr(p.row_ptr),
                                                           _ptr(p.position), _ptr(p.read_id), _ptr(p.gid_base), C.byref(h)))
        dp = DevicePileup(self, h)
        dp._keepalive = p
        return dp

    def pileup_from_bin(self, files: Sequence, id_to_group: Sequence[int], max_coverage: int = 100,
                        positions: Optional[Sequence[Sequence[int]]] = None):
        """Direct ingestion of the reference's binary pileup files (``read_pileup_bin``,
        util/pileup_reader.cpp:139-257), one per chromosome: ``files`` holds paths or bytes-like objects.
        Returns ``(DevicePileup, n_cells, n_groups, max_fragment_length)``; the last is 1000 like the
        reference without ``--compute_read_stats``."""
        bufs = []
        for f in files:
            if isinstance(f, (str, os.PathLike)):
                f = np.fromfile(f, dtype=np.uint8)
            bufs.append(np.frombuffer(f, dtype=np.uint8) if not isinstance(f, np.ndarray) else np.ascontiguousarray(f, np.uint8))
        n = len(bufs)
        ptrs = (C.c_void_p * max(n, 1))(*[b.ctypes.data if b.size else None for b in bufs])
        sizes = np.array([b.size for b in bufs], np.uint64)
        g = np.ascontiguousarray(id_to_group, np.uint16)
        pos_ptrs, pos_n, keep = None, None, []
        if positions is not None:
            keep = [np.ascontiguousarray(x, np.uint32) for x in positions]
            assert len(keep) == n
            pos_ptrs = (C.c_void_p * max(n, 1))(*[x.ctypes.data if x.size else None for x in keep])
            pos_n = np.array([x.size for x in keep], np.uint64)
        h, nc, ng = C.c_void_p(), C.c_uint32(), C.c_uint32()
        self.check(self._lib.sgpu_pileup_from_bin(self._h, n, ptrs, _ptr(sizes), _ptr(g), g.size, int(max_coverage), pos_ptrs,
                                                  _ptr(pos_n), C.byref(h), C.byref(nc), C.byref(ng)))
        return DevicePileup(self, h), nc.value, ng.value, 1000

    def wrap_device(self, chr_ptr: np.ndarray, d_row_ptr: int, d_position: int, d_read_id: int, d_gid_base: int,
                    keepalive=None) -> "DevicePileup":
        chr_ptr = np.ascontiguousarray(chr_ptr, np.uint64)
        h = C.c_void_p()
        self.check(self._lib.sgpu_pileup_wrap_device(self._h, chr_ptr.size - 1, _ptr(chr_ptr), C.c_void_p(d_row_ptr),
                                                     C.c_void_p(d_position), C.c_void_p(d_read_id),
                                                     C.c_void_p(d_gid_base), C.byref(h)))
        dp = DevicePileup(self, h)
        dp._keepalive = keepalive
        return dp


TAIL_NONE, TAIL_AUTO = 0xFFFFFFFF, 0xFFFFFFFE  # tail_position values of Counts.accumulate_range


class MultiContext:
    """Several GPUs behind one call, in ONE process (``sgpu_multi_*``): what the C++ shim's computeSimilarityMatrix uses
    when more than one GPU is visible. ``devices=None`` takes all visible GPUs."""

    def __init__(self, devices: Optional[Sequence[int]] = None):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        arr = None if devices is None else (C.c_int * len(devices))(*devices)
        rc = self._lib.sgpu_multi_init(arr, 0 if devices is None else len(devices), C.byref(self._h))
        if rc != 0:
            msg = self._lib.sgpu_multi_last_error(self._h).decode() if self._h else "sgpu_multi_init failed"
            if self._h:
                self._lib.sgpu_multi_shutdown(self._h)
                self._h = C.c_void_p()
            raise SgpuError(rc, msg)

    @property
    def size(self) -> int:
        return int(self._lib.sgpu_multi_size(self._h))

    def similarity(self, filtered: Pileup, num_cells: int, max_fragment_length: int, group_id_to_pos: Sequence[int],
                   mutation_rate: float, homozygous_rate: float, seq_error_rate: float, num_threads: int,
                   normalization: str = "ADD_MIN", path: str = "auto", return_stats: bool = False):
        if normalization not in NORMALIZATIONS:
            raise ValueError("Invalid normalization: " + str(normalization))
        assert not filtered.wide, "sgpu_multi_similarity takes the reference's 14-bit group ids"
        g = np.ascontiguousarray(group_id_to_pos, np.uint32)
        out = np.zeros((int(num_cells), int(num_cells)), np.float64)
        st = Stats()
        rc = self._lib.sgpu_multi_similarity(self._h, filtered.n_chr, _ptr(filtered.chr_ptr), _ptr(filtered.row_ptr),
                                             _ptr(filtered.position), _ptr(filtered.read_id), _ptr(filtered.gid_base),
                                             int(num_cells), int(max_fragment_length), _ptr(g), g.size, float(mutation_rate),
                                             float(homozygous_rate), float(seq_error_rate), int(num_threads),
                                             NORMALIZATIONS[normalization], PATHS[path], _ptr(out), C.byref(st))
        if rc != 0:
            raise SgpuError(rc, self._lib.sgpu_multi_last_error(self._h).decode())
        return (out, st.as_dict()) if return_stats else out

    def close(self) -> None:
        if self._h:
            self._lib.sgpu_multi_shutdown(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx: Optional[Context] = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


class DevicePileup:
    """Device-resident CSR pileup (``sgpu_pileup``)."""

    def __init__(self, ctx: Context, handle: C.c_void_p):
        self.ctx, self._h, self._keepalive = ctx, handle, None

    def dims(self) -> Tuple[int, int, int]:
        a, b, c = C.c_uint32(), C.c_uint64(), C.c_uint64()
        self.ctx.check(self.ctx._lib.sgpu_pileup_dims(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    @property
    def n_chr(self) -> int:
        return self.dims()[0]

    @property
    def n_loci(self) -> int:
        return self.dims()[1]

    @property
    def n_entries(self) -> int:
        return self.dims()[2]

    @property
    def wide(self) -> bool:
        return bool(self.ctx._lib.sgpu_pileup_is_wide(self._h))

    def download(self) -> Pileup:
        n_chr, n_loci, n_entries = self.dims()
        wide = self.wide
        chr_ptr, row_ptr = np.zeros(n_chr + 1, np.uint64), np.zeros(n_loci + 1, np.uint64)
        pos, rid = np.zeros(n_loci, np.uint32), np.zeros(n_entries, np.uint32)
        gb = np.zeros(n_entries, np.uint32 if wide else np.uint16)
        fn = self.ctx._lib.sgpu_pileup_download_wide if wide else self.ctx._lib.sgpu_pileup_download
        self.ctx.check(fn(self.ctx._h, self._h, _ptr(chr_ptr), _ptr(row_ptr), _ptr(pos), _ptr(rid), _ptr(gb)))
        return Pileup(chr_ptr, row_ptr, pos, rid, gb)

    def free(self) -> None:
        if self._h and self.ctx._h:
            self.ctx._lib.sgpu_pileup_free(self.ctx._h, self._h)
        self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


PosDataLike = Union[Pileup, DevicePileup]


def _staged(ctx: Context, p: PosDataLike) -> Tuple[DevicePileup, bool]:
    if isinstance(p, DevicePileup):
        return p, False
    return ctx.upload(p), True


class Filter:
    """Mirror of the reference's ``Filter`` (util/is_significant.hpp:13-80)."""

    def __init__(self, theta: float, cell_proportion: int = 4, ctx: Optional[Context] = None):
        self.theta, self.cell_proportion = float(theta), int(cell_proportion)
        self.ctx = ctx or default_context()

    def is_significant(self, base_count: Sequence[int]) -> Union[bool, np.ndarray]:
        """``base_count``: 4 pooled counts (any base order) or an (n, 4) array of them."""
        a = np.ascontiguousarray(base_count, np.uint16)
        single = a.ndim == 1
        a = a.reshape(-1, 4)
        out = np.zeros(a.shape[0], np.uint8)
        self.ctx.check(self.ctx._lib.sgpu_is_significant(self.ctx._h, _ptr(a), a.shape[0], self.theta,
                                                         self.cell_proportion, _ptr(out)))
        return bool(out[0]) if single else out.astype(bool)

    def filter_device(self, pos_data: PosDataLike, id_to_pos: Sequence[int]) -> Tuple[DevicePileup, float]:
        ctx = self.ctx
        id_to_pos = np.ascontiguousarray(id_to_pos, np.uint32)
        dp, owned = _staged(ctx, pos_data)
        try:
            h, cov = C.c_void_p(), C.c_double()
            ctx.check(ctx._lib.sgpu_filter(ctx._h, dp._h, _ptr(id_to_pos), id_to_pos.size, self.theta,
                                           self.cell_proportion, C.byref(h), C.byref(cov)))
        finally:
            if owned:
                dp.free()
        return DevicePileup(ctx, h), cov.value

    def filter(self, pos_data: PosDataLike, id_to_pos: Sequence[int], marker: str = "",
               num_threads: int = 1) -> Tuple[Pileup, float]:
        """Returns (filtered pileup on the host, average coverage) like the reference; ``marker`` and
        ``num_threads`` are accepted for signature parity (the reference only logs / ignores them)."""
        del marker, num_threads
        dev, cov = self.filter_device(pos_data, id_to_pos)
        try:
            return dev.download(), cov
        finally:
            dev.free()


class Counts:
    """Device-resident integer read-pair count matrices (``sgpu_counts``)."""

    def __init__(self, ctx: Context, num_cells: int):
        self.ctx, self.num_cells = ctx, int(num_cells)
        self._h = C.c_void_p()
        ctx.check(ctx._lib.sgpu_counts_create(ctx._h, self.num_cells, C.byref(self._h)))
        self.last_stats: Optional[dict] = None

    def zero(self) -> None:
        self.ctx.check(self.ctx._lib.sgpu_counts_zero(self.ctx._h, self._h))

    def accumulate(self, filtered: PosDataLike, max_fragment_length: int, group_id_to_pos: Sequence[int],
                   mutation_rate: float, homozygous_rate: float, seq_error_rate: float, num_threads: int,
                   path: str = "auto") -> dict:
        ctx = self.ctx
        g = np.ascontiguousarray(group_id_to_pos, np.uint32)
        dp, owned = _staged(ctx, filtered)
        st = Stats()
        try:
            ctx.check(ctx._lib.sgpu_counts_accumulate(ctx._h, self._h, dp._h, int(max_fragment_length), _ptr(g), g.size,
                                                      float(mutation_rate), float(homozygous_rate),
                                                      float(seq_error_rate), int(num_threads), PATHS[path],
                                                      C.byref(st)))
        finally:
            if owned:
                dp.free()
        self.last_stats = st.as_dict()
        return self.last_stats

    def accumulate_range(self, piece: PosDataLike, max_fragment_length: int, group_id_to_pos: Sequence[int],
                         mutation_rate: float, homozygous_rate: float, seq_error_rate: float,
                         own_pos_begin: Sequence[int], own_pos_end: Sequence[int], tail_position: Sequence[int],
                         path: str = "auto", num_threads: int = 1) -> dict:
        """A piece of its chromosomes (owned loci by position range + halos of max_fragment_length bp): adds the piece's
        share of the counts. ``tail_position`` comes from :func:`chromosome_cutoff`, or is ``TAIL_AUTO`` for a piece that
        holds the end of its chromosome (decided from the piece, with ``num_threads``). See include/secedo_b200.h."""
        ctx = self.ctx
        g = np.ascontiguousarray(group_id_to_pos, np.uint32)
        lo, hi = np.ascontiguousarray(own_pos_begin, np.uint32), np.ascontiguousarray(own_pos_end, np.uint32)
        tp = np.ascontiguousarray(tail_position, np.uint32)
        dp, owned = _staged(ctx, piece)
        assert lo.size == hi.size == tp.size == dp.n_chr, "one value per chromosome of the piece"
        st = Stats()
        try:
            ctx.check(ctx._lib.sgpu_counts_accumulate_range(ctx._h, self._h, dp._h, int(max_fragment_length), _ptr(g), g.size,
                                                            float(mutation_rate), float(homozygous_rate), float(seq_error_rate),
                                                            int(num_threads), _ptr(lo), _ptr(hi), _ptr(tp), PATHS[path],
                                                            C.byref(st)))
        finally:
            if owned:
                dp.free()
        self.last_stats = st.as_dict()
        return self.last_stats

    def buffers(self):
        """(i32 device pointer, n_i32, f64 device pointer or None, n_f64, hist device pointer, n_hist)."""
        i32, f64, hist = C.c_void_p(), C.c_void_p(), C.c_void_p()
        n_i32, n_f64, n_hist = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self.ctx.check(self.ctx._lib.sgpu_counts_buffers(self._h, C.byref(i32), C.byref(n_i32), C.byref(f64),
                                                         C.byref(n_f64), C.byref(hist), C.byref(n_hist)))
        return i32.value, n_i32.value, f64.value, n_f64.value, hist.value, n_hist.value

    def set_layout(self, planes_used: int, want_spill: bool) -> None:
        self.ctx.check(self.ctx._lib.sgpu_counts_set_layout(self.ctx._h, self._h, int(planes_used), int(want_spill)))

    def pack(self):
        """Upper triangles of the planes in use, packed into one device buffer: (pointer, n int32)."""
        ptr, n = C.c_void_p(), C.c_uint64()
        self.ctx.check(self.ctx._lib.sgpu_counts_pack(self.ctx._h, self._h, C.byref(ptr), C.byref(n)))
        return ptr.value, n.value

    def unpack(self) -> None:
        """Packed buffer (after the cross-rank reduction) back into the planes."""
        self.ctx.check(self.ctx._lib.sgpu_counts_unpack(self.ctx._h, self._h))

    def pack_range(self, first_plane: int, n_planes: int):
        ptr, n = C.c_void_p(), C.c_uint64()
        self.ctx.check(self.ctx._lib.sgpu_counts_pack_range(self.ctx._h, self._h, int(first_plane), int(n_planes), C.byref(ptr),
                                                            C.byref(n)))
        return ptr.value, n.value

    def unpack_range(self, first_plane: int, n_planes: int) -> None:
        self.ctx.check(self.ctx._lib.sgpu_counts_unpack_range(self.ctx._h, self._h, int(first_plane), int(n_planes)))

    # ---- multi-GPU epilogue over peer memory (include/secedo_b200.h: sgpu_slab_raw / sgpu_slab_finalize) ----
    def ipc_handle(self, spill: bool = False) -> bytes:
        """CUDA IPC handle (64 bytes) of the int32 planes (or of the fp64 spill plane), for the other ranks of the node."""
        buf = C.create_string_buffer(64)
        self.ctx.check(self.ctx._lib.sgpu_counts_ipc_handle(self.ctx._h, self._h, 1 if spill else 0, buf))
        return buf.raw

    def _peer_array(self, peer_planes: Sequence[Optional[int]]):
        """device pointers as a C array; None is a null pointer (a GPU without a spill plane)"""
        return (C.c_void_p * len(peer_planes))(*[C.c_void_p(None if p is None else int(p)) for p in peer_planes])

    def slab_raw(self, peer_planes: Sequence[int], slab: int, n_slabs: int, max_fragment_length: int, mutation_rate: float,
                 homozygous_rate: float, seq_error_rate: float, peer_spill: Optional[Sequence[Optional[int]]] = None) -> int:
        """Sum the planes of all GPUs (device pointers valid on this GPU, own planes included) over this GPU's share of
        the tiles and transform them; returns the device pointer of {-min, max} (2 doubles) of the share. ``peer_spill``:
        one entry per peer, None for a GPU without a spill plane."""
        assert peer_spill is None or len(peer_spill) == len(peer_planes), "one spill entry per peer"
        ext = C.c_void_p()
        self.ctx.check(self.ctx._lib.sgpu_slab_raw(self.ctx._h, self._h, self._peer_array(peer_planes),
                                                   self._peer_array(peer_spill) if peer_spill else None, len(peer_planes),
                                                   int(slab), int(n_slabs), int(max_fragment_length), float(mutation_rate),
                                                   float(homozygous_rate), float(seq_error_rate), C.byref(ext)))
        return ext.value

    def slab_finalize(self, normalization: str, out_ptr: Optional[int] = None) -> int:
        """Normalise this GPU's share and write it (and its mirror image) into the n x n matrix at ``out_ptr`` (device
        memory or mapped host memory), or into a device matrix owned by this object; returns the pointer written to."""
        if normalization not in NORMALIZATIONS:
            raise ValueError(f"Invalid normalization: {normalization}")
        dev = C.c_void_p()
        self.ctx.check(self.ctx._lib.sgpu_slab_finalize(self.ctx._h, self._h, NORMALIZATIONS[normalization],
                                                        C.c_void_p(out_ptr) if out_ptr else None, C.byref(dev)))
        return dev.value

    def slab_range(self) -> Tuple[int, int]:
        a, b = C.c_uint64(), C.c_uint64()
        self.ctx.check(self.ctx._lib.sgpu_slab_range(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def checksum(self, peer_planes: Optional[Sequence[int]] = None, slab: int = 0, n_slabs: int = 1) -> int:
        """64-bit linear checksum of the upper triangles of the planes in use (of the element-wise sum of the peers'
        planes over share ``slab`` when ``peer_planes`` is given)."""
        out = C.c_uint64()
        arr = self._peer_array(peer_planes) if peer_planes else None
        self.ctx.check(self.ctx._lib.sgpu_counts_checksum(self.ctx._h, self._h, arr, len(peer_planes) if peer_planes else 0,
                                                          int(slab), int(n_slabs), C.byref(out)))
        return out.value

    def sparse_pack(self, first_plane: int = 2):
        """Non-zeros of the planes from ``first_plane`` on as device lists: (idx pointer, val pointer, nnz)."""
        idx, val, nnz = C.c_void_p(), C.c_void_p(), C.c_uint64()
        self.ctx.check(self.ctx._lib.sgpu_counts_sparse_pack(self.ctx._h, self._h, int(first_plane), C.byref(idx), C.byref(val),
                                                             C.byref(nnz)))
        return idx.value, val.value, nnz.value

    def sparse_add(self, first_plane: int, idx_ptr: int, val_ptr: int, nnz: int) -> None:
        self.ctx.check(self.ctx._lib.sgpu_counts_sparse_add(self.ctx._h, self._h, int(first_plane), C.c_void_p(idx_ptr),
                                                            C.c_void_p(val_ptr), int(nnz)))

    def download(self):
        """Symmetric host copies: (S1, D1, H[3], class_hist) for bit-exact checks."""
        n = self.num_cells
        S1, D1 = np.zeros((n, n), np.int32), np.zeros((n, n), np.int32)
        H = np.zeros((3, n, n), np.int32)
        hist = np.zeros((_lib.MAX_CLASS, _lib.MAX_CLASS), np.uint64)
        self.ctx.check(self.ctx._lib.sgpu_counts_download(self.ctx._h, self._h, _ptr(S1), _ptr(D1), _ptr(H), _ptr(hist)))
        return S1, D1, H, hist

    def finalize(self, max_fragment_length: int, mutation_rate: float, homozygous_rate: float,
                 seq_error_rate: float, normalization: str, out: Optional[np.ndarray] = None,
                 to_host: bool = True) -> Optional[np.ndarray]:
        """``to_host=False`` runs the epilogue but leaves the matrix in HBM (device-only timing)."""
        if normalization not in NORMALIZATIONS:
            raise ValueError("Invalid normalization: " + str(normalization))  # similarity_matrix.cpp:264
        n = self.num_cells
        if to_host:
            if out is None:
                out = np.zeros((n, n), np.float64)
            assert out.dtype == np.float64 and out.flags.c_contiguous and out.size == n * n
        else:
            out = None
        st = Stats()
        self.ctx.check(self.ctx._lib.sgpu_similarity_finalize(self.ctx._h, self._h, int(max_fragment_length),
                                                              float(mutation_rate), float(homozygous_rate),
                                                              float(seq_error_rate), NORMALIZATIONS[normalization],
                                                              _ptr(out), C.byref(st)))
        if self.last_stats is not None:
            self.last_stats["ms_epilogue"] = st.ms_epilogue
        return out

    def finalize_async(self, max_fragment_length: int, mutation_rate: float, homozygous_rate: float,
                       seq_error_rate: float, normalization: str, out: np.ndarray) -> None:
        """Epilogue now, download of the matrix into ``out`` (pinned host memory) on a stream of its own;
        :meth:`Context.output_wait` returns when ``out`` is complete."""
        if normalization not in NORMALIZATIONS:
            raise ValueError("Invalid normalization: " + str(normalization))
        n = self.num_cells
        assert out.dtype == np.float64 and out.flags.c_contiguous and out.size == n * n
        self.ctx.check(self.ctx._lib.sgpu_similarity_finalize_async(self.ctx._h, self._h, int(max_fragment_length),
                                                                    float(mutation_rate), float(homozygous_rate),
                                                                    float(seq_error_rate), NORMALIZATIONS[normalization],
                                                                    _ptr(out)))

    def finalize_spectral(self, max_fragment_length: int, mutation_rate: float, homozygous_rate: float,
                          seq_error_rate: float, normalization: str, k: int = 7, tol: float = 0.0,
                          want_matrix: bool = False):
        """Epilogue + Laplacian + the ``k`` smallest eigenpairs without the matrix leaving HBM
        (what ``spectral_clustering`` takes from ``arma::eig_sym``, spectral_clustering.cpp:127-138).
        Returns (eigenvalues[k], eigenvectors[n, k], stats, matrix or None)."""
        if normalization not in NORMALIZATIONS:
            raise ValueError("Invalid normalization: " + str(normalization))
        n = self.num_cells
        out = np.zeros((n, n), np.float64) if want_matrix else None
        ev, vec = np.zeros(k, np.float64), np.zeros((k, n), np.float64)
        st, sp = Stats(), SpectralStats()
        self.ctx.check(self.ctx._lib.sgpu_similarity_finalize_spectral(
            self.ctx._h, self._h, int(max_fragment_length), float(mutation_rate), float(homozygous_rate),
            float(seq_error_rate), NORMALIZATIONS[normalization], _ptr(out), int(k), float(tol), _ptr(ev), _ptr(vec),
            C.byref(st), C.byref(sp)))
        d = sp.as_dict()
        d["ms_epilogue"] = st.ms_epilogue
        return ev, np.ascontiguousarray(vec.T), d, out

    def free(self) -> None:
        if self._h and self.ctx._h:
            self.ctx._lib.sgpu_counts_free(self.ctx._h, self._h)
        self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def compute_similarity_matrix(pos_data: PosDataLike, num_cells: int, max_fragment_length: int,
                              group_id_to_pos: Sequence[int], mutation_rate: float, homozygous_rate: float,
                              seq_error_rate: float, num_threads: int, marker: str = "",
                              normalization: str = "ADD_MIN", *, ctx: Optional[Context] = None, path: str = "auto",
                              out: Optional[np.ndarray] = None, return_stats: bool = False):
    """``computeSimilarityMatrix`` (similarity_matrix.hpp:51-60) on one GPU. ``num_threads`` selects
    the reference's tail cutoff (the result of the reference depends on it, SURVEY.md F2)."""
    del marker
    if normalization not in NORMALIZATIONS:
        raise ValueError("Invalid normalization: " + str(normalization))  # std::logic_error in the reference
    ctx = ctx or default_context()
    g = np.ascontiguousarray(group_id_to_pos, np.uint32)
    n = int(num_cells)
    if out is None:
        out = np.zeros((n, n), np.float64)
    assert out.dtype == np.float64 and out.flags.c_contiguous and out.size == n * n
    dp, owned = _staged(ctx, pos_data)
    st = Stats()
    try:
        ctx.check(ctx._lib.sgpu_similarity(ctx._h, dp._h, n, int(max_fragment_length), _ptr(g), g.size,
                                           float(mutation_rate), float(homozygous_rate), float(seq_error_rate),
                                           int(num_threads), NORMALIZATIONS[normalization], PATHS[path], _ptr(out),
                                           C.byref(st)))
    finally:
        if owned:
            dp.free()
    return (out, st.as_dict()) if return_stats else out


def chromosome_cutoff(ends: PosDataLike, max_fragment_length: int, num_threads: int, whole: Sequence[bool],
                      ctx: Optional[Context] = None):
    """The reference's tail cutoff of whole chromosomes decided from their ENDS (``sgpu_chromosome_cutoff``): returns
    (tail_position uint32[n_chr], resolved bool[n_chr])."""
    ctx = ctx or default_context()
    dp, owned = _staged(ctx, ends)
    w = np.ascontiguousarray(whole, np.uint8)
    n_chr = dp.n_chr
    assert w.size == n_chr
    tp, rs = np.zeros(n_chr, np.uint32), np.zeros(n_chr, np.uint8)
    try:
        ctx.check(ctx._lib.sgpu_chromosome_cutoff(ctx._h, dp._h, int(max_fragment_length), int(num_threads), _ptr(w), _ptr(tp),
                                                  _ptr(rs)))
    finally:
        if owned:
            dp.free()
    return tp, rs.astype(bool)


def log_probs(mutation_rate: float, homozygous_rate: float, seq_error_rate: float, max_fragment_length: int, n: int,
              ctx: Optional[Context] = None):
    """LS / LD tables evaluated on the device (similarity_matrix.cpp:117-170)."""
    ctx = ctx or default_context()
    ls, ld = np.zeros((n, n)), np.zeros((n, n))
    ctx.check(ctx._lib.sgpu_log_probs(ctx._h, float(mutation_rate), float(homozygous_rate), float(seq_error_rate),
                                      int(max_fragment_length), int(n), _ptr(ls), _ptr(ld)))
    return ls, ld


def expectation_maximization(pos_data: PosDataLike, cell_id_to_cell_pos: Sequence[int], num_threads: int, theta: float,
                             prob_cluster_b: Sequence[float], *, ctx: Optional[Context] = None, max_iterations: int = 0,
                             return_stats: bool = False):
    """``expectation_maximization`` (expectation_maximization.hpp:27-31): refines the probability of every cell to
    belong to the second cluster. The reference updates ``prob_cluster_b`` in place; here the refined vector is
    returned. ``num_threads`` is unused, as in the reference (expectation_maximization.cpp:133)."""
    del num_threads
    ctx = ctx or default_context()
    m = np.ascontiguousarray(cell_id_to_cell_pos, np.uint32)
    prob = np.array(prob_cluster_b, dtype=np.float64, order="C")
    dp, owned = _staged(ctx, pos_data)
    it, ms = C.c_uint32(0), C.c_float(0)
    try:
        ctx.check(ctx._lib.sgpu_expectation_maximization(ctx._h, dp._h, _ptr(m) if m.size else None, m.size, float(theta),
                                                         _ptr(prob), prob.size, int(max_iterations), C.byref(it), C.byref(ms)))
    finally:
        if owned:
            dp.free()
    return (prob, {"iterations": int(it.value), "ms": float(ms.value)}) if return_stats else prob


def laplacian(a: np.ndarray, ctx: Optional[Context] = None) -> np.ndarray:
    """``laplacian`` (spectral_clustering.cpp:33-52): I - D^-1/2 A D^-1/2 of a symmetric matrix with zero diagonal."""
    ctx = ctx or default_context()
    a = np.ascontiguousarray(a, np.float64)
    assert a.ndim == 2 and a.shape[0] == a.shape[1]
    out = np.zeros_like(a)
    ctx.check(ctx._lib.sgpu_laplacian(ctx._h, _ptr(a), a.shape[0], _ptr(out)))
    return out


def spectral_embedding(similarity: np.ndarray, k: int = 7, tol: float = 0.0, ctx: Optional[Context] = None,
                       return_stats: bool = False):
    """The part of ``arma::eig_sym(eigenvalues, eigenvectors, laplacian(similarity))`` that
    ``spectral_clustering`` uses (spectral_clustering.cpp:127-138, :166-171, :218, :236): the ``k`` smallest
    eigenvalues (ascending) and their eigenvectors as the columns of an (n, k) array."""
    ctx = ctx or default_context()
    a = np.ascontiguousarray(similarity, np.float64)
    assert a.ndim == 2 and a.shape[0] == a.shape[1]
    n = a.shape[0]
    ev, vec = np.zeros(k, np.float64), np.zeros((k, n), np.float64)
    sp = SpectralStats()
    ctx.check(ctx._lib.sgpu_spectral_embedding(ctx._h, _ptr(a), n, int(k), float(tol), _ptr(ev), _ptr(vec), C.byref(sp)))
    vec = np.ascontiguousarray(vec.T)
    return (ev, vec, sp.as_dict()) if return_stats else (ev, vec)


def spectral_matvec(m: np.ndarray, x: np.ndarray, w: Optional[np.ndarray] = None, alpha: float = 1.0, beta: float = 0.0,
                    gamma: float = 0.0, ctx: Optional[Context] = None) -> np.ndarray:
    """Test hook of the block product kernel of the eigen-solver: alpha M X + beta X + gamma W."""
    ctx = ctx or default_context()
    m = np.ascontiguousarray(m, np.float64)
    x = np.ascontiguousarray(x, np.float64)
    w = None if w is None else np.ascontiguousarray(w, np.float64)
    out = np.zeros_like(x)
    ctx.check(ctx._lib.sgpu_spectral_matvec(ctx._h, _ptr(m), m.shape[0], x.shape[1], _ptr(x), _ptr(w), float(alpha),
                                            float(beta), float(gamma), _ptr(out)))
    return out


__all__ = ["Context", "DevicePileup", "Filter", "Counts", "compute_similarity_matrix", "log_probs", "default_context", "expectation_maximization", "laplacian", "spectral_embedding",
           "NO_POS", "SgpuError"]
