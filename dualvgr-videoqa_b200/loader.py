"""Input pipeline for the train / eval engines (SURVEY.md §8f.3) — what the reference's DataLoader.py:61-84 does per sample
(open both HDF5 files, index one video, build fp32 tensors; 2.79 MB per sample over a pageable H2D copy, train.py:134),
restated for a step that takes ~5 ms:

  * FeatureStore: the appearance / motion features of all videos memory-mapped ONCE (no per-sample file open), optionally
    stored as bf16 (half the bytes on disk, in page cache and on the host link; the kernels take bf16 features directly,
    dvgr_prep_features_ex). Layout = the reference's HDF5 datasets (preprocess/preprocess_features.py:143-203):
    resnet_features [V, N, 16, 2048], resnext_features [V, N, 2048], ids [V]; read from .npy files (np.memmap) — or from
    the original .h5 files when h5py is importable.
  * PinnedBatchLoader: a background thread gathers the next batches into a ring of PINNED host buffers; the consumer issues
    the host-to-device copies on a copy stream (double-buffered device slots) and hands device tensors to
    TrainEngine.load_batch / EvalEngine.step. The training stream never waits on a page fault or a pageable copy.
  * DeviceFeatureStore + DeviceBatchLoader: the whole store uploaded once into device memory; a batch is then its video
    rows plus the question / answer arrays, and the input prologue kernels read the clips at those rows
    (DualVGR.forward_from_store, TrainEngine / EvalEngine *_from_store)."""
import queue
import threading

import numpy as np
import torch


class FeatureStore:
    def __init__(self, appearance, motion, ids=None):
        """appearance [V, N, F, Dv], motion [V, N, Dv]: numpy arrays / memmaps (float32, or uint16 holding bf16 bits)."""
        self.app, self.mot = appearance, motion
        self.ids = np.arange(appearance.shape[0]) if ids is None else np.asarray(ids)
        self.row = {int(v): i for i, v in enumerate(self.ids)}
        self.bf16 = appearance.dtype == np.uint16

    @classmethod
    def open(cls, appearance_path, motion_path):
        if appearance_path.endswith(".h5"):
            import h5py                                   # optional: the reference's own files
            fa, fm = h5py.File(appearance_path, "r"), h5py.File(motion_path, "r")
            return cls(fa["resnet_features"], fm["resnext_features"], fa["ids"][()])
        return cls(np.load(appearance_path, mmap_mode="r"), np.load(motion_path, mmap_mode="r"))

    @staticmethod
    def to_bf16_bits(x):
        """float32 array -> uint16 array of bf16 bit patterns (round to nearest even), the storage format of a bf16 store."""
        u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
        return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)

    def torch_dtype(self):
        return torch.bfloat16 if self.bf16 else torch.float32


class PinnedBatchLoader:
    """Iterates device batches (app, mot, question, question_len, answers[, extra...]) over `samples`.

    samples: dict of host arrays indexed by sample: 'video_idx' (row in the store, or 'video_id' resolved through store.ids),
    'question' [S, L] int64, 'question_len' [S] int64, 'answer' [S] int64, optional 'category' [S] int64."""

    def __init__(self, store, samples, batch_size, device, shuffle=False, seed=0, drop_last=True, slots=3):
        self.store, self.samples, self.B, self.dev = store, samples, batch_size, torch.device(device)
        self.shuffle, self.rng, self.drop_last, self.slots = shuffle, np.random.default_rng(seed), drop_last, max(2, slots)
        vid = samples.get("video_idx")
        if vid is None:
            vid = np.array([store.row[int(v)] for v in samples["video_id"]])
        self.vid = np.asarray(vid)
        self.S = len(self.vid)
        N, F, Dv = store.app.shape[1:]
        L = samples["question"].shape[1]
        fdt = store.torch_dtype()
        self.has_cat = "category" in samples

        def slot(pin):
            kw = dict(pin_memory=True) if pin else dict(device=self.dev)
            d = {"app": torch.empty((batch_size, N, F, Dv), dtype=fdt, **kw),
                 "mot": torch.empty((batch_size, N, Dv), dtype=fdt, **kw),
                 "q": torch.empty((batch_size, L), dtype=torch.int64, **kw),
                 "qlen": torch.empty((batch_size,), dtype=torch.int64, **kw),
                 "ans": torch.empty((batch_size,), dtype=torch.int64, **kw)}
            if self.has_cat:
                d["cat"] = torch.empty((batch_size,), dtype=torch.int64, **kw)
            return d

        self.host = [slot(True) for _ in range(self.slots)]
        self.device_slots = [slot(False) for _ in range(2)]
        self.copy_stream = torch.cuda.Stream(device=self.dev)
        self.bytes_per_batch = sum(t.numel() * t.element_size() for t in self.host[0].values())

    def __len__(self):
        return self.S // self.B if self.drop_last else (self.S + self.B - 1) // self.B

    def _fill(self, slot, idx):
        """Gathers samples `idx` into pinned slot `slot` (runs on the worker thread; numpy releases the GIL in the copies)."""
        n = len(idx)
        order = np.argsort(self.vid[idx], kind="stable")            # ascending rows: sequential reads from the memmap
        rows = self.vid[idx][order]
        h = self.host[slot]
        app = h["app"].view(torch.uint16).numpy() if self.store.bf16 else h["app"].numpy()
        mot = h["mot"].view(torch.uint16).numpy() if self.store.bf16 else h["mot"].numpy()
        for k, r in zip(order, rows):
            app[k] = self.store.app[r]
            mot[k] = self.store.mot[r]
        h["q"][:n] = torch.from_numpy(np.ascontiguousarray(self.samples["question"][idx]))
        h["qlen"][:n] = torch.from_numpy(np.ascontiguousarray(self.samples["question_len"][idx]))
        h["ans"][:n] = torch.from_numpy(np.ascontiguousarray(self.samples["answer"][idx]))
        if self.has_cat:
            h["cat"][:n] = torch.from_numpy(np.ascontiguousarray(self.samples["category"][idx]))
        return n

    def __iter__(self):
        order = self.rng.permutation(self.S) if self.shuffle else np.arange(self.S)
        batches = [order[i:i + self.B] for i in range(0, self.S, self.B)]
        if self.drop_last and batches and len(batches[-1]) < self.B:
            batches.pop()
        free, ready = queue.Queue(), queue.Queue()
        for s in range(self.slots):
            free.put(s)

        def worker():
            try:
                for idx in batches:
                    s = free.get()
                    ready.put((s, self._fill(s, idx)))
                ready.put(None)
            except BaseException as e:                                # surface worker failures in the consumer
                ready.put(e)

        threading.Thread(target=worker, daemon=True).start()
        cur = torch.cuda.current_stream(self.dev)
        consumed = [torch.cuda.Event(), torch.cuda.Event()]
        for e in consumed:
            e.record(cur)
        pending = None                     # (device slot, n, copy-done event, pinned slot)
        k = 0

        def start_copy(item):
            nonlocal k
            s, n = item
            d = k % 2
            k += 1
            with torch.cuda.stream(self.copy_stream):
                self.copy_stream.wait_event(consumed[d])            # the step that read this device slot has finished
                for name, t in self.host[s].items():
                    self.device_slots[d][name][:n].copy_(t[:n], non_blocking=True)
                done = torch.cuda.Event()
                done.record(self.copy_stream)
            return d, n, done, s

        while True:
            item = ready.get()
            if isinstance(item, BaseException):
                raise item
            nxt = start_copy(item) if item is not None else None
            if pending is not None:
                d, n, done, s = pending
                cur.wait_event(done)
                done.synchronize()                                   # the pinned slot may be refilled once its copy is done
                free.put(s)
                dev = self.device_slots[d]
                out = [dev["app"][:n], dev["mot"][:n], dev["q"][:n], dev["qlen"][:n], dev["ans"][:n]]
                if self.has_cat:
                    out.append(dev["cat"][:n])
                yield tuple(out)
                consumed[d].record(torch.cuda.current_stream(self.dev))
            pending = nxt
            if item is None:
                break


class DeviceFeatureStore:
    """The whole feature store resident in device memory: app [V, N, F, Dv], mot [V, N, Dv] (fp32, or bf16), plus the
    ids / row map of the host store and `err`, a sticky [1] int32 word that the gathering prologue kernels
    (ops.prep_features_gather) set when a batch names a row outside [0, V). With it, a step's only input transfer is the
    batch's video rows and question / answer arrays (DeviceBatchLoader); DualVGR.forward_from_store reads the clips.

    The upload runs once, in chunks of whole videos of at most `chunk_bytes` (or one video) through ONE pinned staging
    buffer. bf16=True stores fp32 features as bf16 (round to nearest even, the bits of FeatureStore.to_bf16_bits); a
    bf16 store stays bf16. Before allocating, the store's size is checked against the free device memory minus
    `reserve_bytes` (the training step's working set: ~3 GB at B=256)."""

    def __init__(self, store, device, bf16=False, reserve_bytes=4 << 30, chunk_bytes=256 << 20):
        self.device = torch.device(device)
        self.ids, self.row = store.ids, store.row
        self.V = int(store.app.shape[0])
        cast = bool(bf16) and not store.bf16
        src_dt = store.torch_dtype()
        dt = torch.bfloat16 if (store.bf16 or cast) else torch.float32
        app_shape, mot_shape = tuple(store.app.shape), tuple(store.mot.shape)
        esz = torch.empty((), dtype=dt).element_size()
        src_esz = torch.empty((), dtype=src_dt).element_size()
        per_video = (int(np.prod(app_shape[1:])) + int(np.prod(mot_shape[1:]))) * src_esz
        rows_per_chunk = max(1, int(chunk_bytes) // max(1, per_video))
        self.nbytes = (int(np.prod(app_shape)) + int(np.prod(mot_shape))) * esz
        # device-side fp32 landing buffer of a chunk that is cast to bf16 on the device
        need = self.nbytes + (rows_per_chunk * per_video if cast else 0)
        free, _ = torch.cuda.mem_get_info(self.device)
        avail = int(free) - int(reserve_bytes)
        if need > avail:
            raise MemoryError(f"DeviceFeatureStore: the store needs {need} bytes of device memory, {avail} are available "
                              f"({int(free)} free on {self.device} minus a {int(reserve_bytes)}-byte working-set reserve)")
        self.app = torch.empty(app_shape, dtype=dt, device=self.device)
        self.mot = torch.empty(mot_shape, dtype=dt, device=self.device)
        self.err = torch.zeros(1, dtype=torch.int32, device=self.device)
        stage = torch.empty(rows_per_chunk * per_video // src_esz, dtype=src_dt, pin_memory=True)
        landing = torch.empty(rows_per_chunk * per_video // src_esz, dtype=src_dt, device=self.device) if cast else None
        stream = torch.cuda.Stream(device=self.device)
        done = torch.cuda.Event()
        with torch.cuda.stream(stream):
            for host, dst in ((store.app, self.app), (store.mot, self.mot)):
                per_row = int(np.prod(dst.shape[1:]))
                for r0 in range(0, self.V, rows_per_chunk):
                    r1 = min(self.V, r0 + rows_per_chunk)
                    n = (r1 - r0) * per_row
                    done.synchronize()                     # the previous chunk's copy has left the staging buffer
                    view = stage[:n].view(torch.uint16) if store.bf16 else stage[:n]
                    np.copyto(view.numpy().reshape((r1 - r0,) + dst.shape[1:]), host[r0:r1])
                    if cast:
                        landing[:n].copy_(stage[:n], non_blocking=True)
                        dst[r0:r1].copy_(landing[:n].view((r1 - r0,) + dst.shape[1:]))
                    else:
                        dst[r0:r1].view(-1).copy_(stage[:n], non_blocking=True)
                    done.record(stream)
        done.synchronize()
        del stage, landing

    def read_error(self, clear=False):
        """1 when a batch gathered since the last clear named a row outside [0, V), else 0 (synchronises). A set word also
        turns every train step's loss into NaN (TrainEngine) until it is cleared."""
        v = int(self.err.item())
        if clear:
            self.clear_error()
        return v

    def clear_error(self):
        self.err.zero_()


class DeviceBatchLoader:
    """Iterates device batches (rows int32, question, question_len, answers[, category]) over `samples` for a
    DeviceFeatureStore: the clip features never move, so a batch is B video rows plus the question / answer arrays (~45 KB
    at B=256), copied from pinned host slots on a copy stream into double-buffered device slots as PinnedBatchLoader does.

    samples: the dict PinnedBatchLoader takes ('video_idx' or 'video_id', 'question', 'question_len', 'answer', optional
    'category'). Every row is checked against the store's V here, before anything is launched."""

    def __init__(self, dstore, samples, batch_size, device, shuffle=False, seed=0, drop_last=True):
        self.store, self.samples, self.B, self.dev = dstore, samples, batch_size, torch.device(device)
        self.shuffle, self.rng, self.drop_last = shuffle, np.random.default_rng(seed), drop_last
        vid = samples.get("video_idx")
        if vid is None:
            missing = [v for v in samples["video_id"] if int(v) not in dstore.row]
            if missing:
                raise ValueError(f"DeviceBatchLoader: video ids {missing[:8]} are not in the store")
            vid = np.array([dstore.row[int(v)] for v in samples["video_id"]])
        self.vid = np.asarray(vid, dtype=np.int64)
        bad = np.flatnonzero((self.vid < 0) | (self.vid >= dstore.V))
        if bad.size:
            raise ValueError(f"DeviceBatchLoader: samples {bad[:8].tolist()} name video rows "
                             f"{self.vid[bad[:8]].tolist()} outside the store's [0, {dstore.V})")
        self.S = len(self.vid)
        L = samples["question"].shape[1]
        self.has_cat = "category" in samples

        def slot(pin):
            kw = dict(pin_memory=True) if pin else dict(device=self.dev)
            d = {"rows": torch.empty((batch_size,), dtype=torch.int32, **kw),
                 "q": torch.empty((batch_size, L), dtype=torch.int64, **kw),
                 "qlen": torch.empty((batch_size,), dtype=torch.int64, **kw),
                 "ans": torch.empty((batch_size,), dtype=torch.int64, **kw)}
            if self.has_cat:
                d["cat"] = torch.empty((batch_size,), dtype=torch.int64, **kw)
            return d

        self.host = [slot(True) for _ in range(2)]
        self.device_slots = [slot(False) for _ in range(2)]
        self.copy_stream = torch.cuda.Stream(device=self.dev)
        self.bytes_per_batch = sum(t.numel() * t.element_size() for t in self.host[0].values())

    def __len__(self):
        return self.S // self.B if self.drop_last else (self.S + self.B - 1) // self.B

    def __iter__(self):
        order = self.rng.permutation(self.S) if self.shuffle else np.arange(self.S)
        batches = [order[i:i + self.B] for i in range(0, self.S, self.B)]
        if self.drop_last and batches and len(batches[-1]) < self.B:
            batches.pop()
        cur = torch.cuda.current_stream(self.dev)
        consumed = [torch.cuda.Event(), torch.cuda.Event()]
        copied = [torch.cuda.Event(), torch.cuda.Event()]
        for e in consumed + copied:
            e.record(cur)

        def start_copy(k, idx):
            d, n = k % 2, len(idx)
            h = self.host[d]
            copied[d].synchronize()                                  # this pinned slot's previous copy has completed
            h["rows"][:n] = torch.from_numpy(self.vid[idx].astype(np.int32))
            h["q"][:n] = torch.from_numpy(np.ascontiguousarray(self.samples["question"][idx]))
            h["qlen"][:n] = torch.from_numpy(np.ascontiguousarray(self.samples["question_len"][idx]))
            h["ans"][:n] = torch.from_numpy(np.ascontiguousarray(self.samples["answer"][idx]))
            if self.has_cat:
                h["cat"][:n] = torch.from_numpy(np.ascontiguousarray(self.samples["category"][idx]))
            with torch.cuda.stream(self.copy_stream):
                self.copy_stream.wait_event(consumed[d])            # the step that read this device slot has finished
                for name, t in h.items():
                    self.device_slots[d][name][:n].copy_(t[:n], non_blocking=True)
                copied[d].record(self.copy_stream)
            return d, n

        pending = start_copy(0, batches[0]) if batches else None
        for k in range(len(batches)):
            d, n = pending
            pending = start_copy(k + 1, batches[k + 1]) if k + 1 < len(batches) else None
            cur.wait_event(copied[d])
            dev = self.device_slots[d]
            out = [dev["rows"][:n], dev["q"][:n], dev["qlen"][:n], dev["ans"][:n]]
            if self.has_cat:
                out.append(dev["cat"][:n])
            yield tuple(out)
            consumed[d].record(torch.cuda.current_stream(self.dev))
