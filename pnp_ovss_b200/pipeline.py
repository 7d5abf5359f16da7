"""Batched GPU composition of the hot path, as save_img_union_attention (DRV:290-521 / DRVC:337-640) composes it
per image on the CPU: Salience DropOut rounds -> token merge -> threshold/upsample -> blur -> dense CRF -> argmax,
relabel, confusion matrix.  Everything stays on the device between stages; images of one launch share
(C, background rule, H, W) and are bucketed by that key when a batch is ragged."""
import numpy as np
import torch

from . import host, ops
from ._lib import PnpError

CRF_DEFAULTS = dict(n_iter=10, pos_w=7.0, pos_xy_std=3.0, bi_w=10.0, bi_xy_std=50.0, bi_rgb_std=5.0)  # DRV:1036-1041
BLUR_SCALE = 0.05  # DRV:1009
SAVE_LEN = 10      # DRV:643
# Blurred maps (--postprocess blur / blur+crf) take the fused low-rank kernel group (pnp_lowrank_blur_unary).  False selects the
# direct kernels (full-resolution upsample, tap-by-tap blur of every channel, separate unary): ~10x slower, same results to
# 5e-6 on the maps; kept because its summation order is the one the bit-exact golden confusion matrices were recorded with.
USE_LOWRANK_BLUR = True
# Ragged batches (real datasets: every image has its own class list and ground-truth size).  Images are bucketed by
# (padded channel count Cp, background rule, H, W): inside a bucket the class counts may differ -- the fused (d) group takes them
# per image (pnp_lowrank_blur_unary_padded) and the channels an image lacks are dead in the CRF (Q = 0 exactly), so every image
# gets bit for bit what a batch of its own would give.  Buckets are independent launch chains of small kernels: they are spread
# round-robin over BUCKET_STREAMS CUDA streams, and all bilateral lattice builds are enqueued before the first one is waited for.
PAD_CLASSES_IN_BUCKETS = True
BUCKET_STREAMS = 4
# A bucket of one small image is ~150 kernel launches whose device time is shorter than the host time to issue them: the buckets
# of a ragged batch are therefore ALSO issued from BUCKET_STREAMS host threads (one per stream; the C-ABI calls release the GIL).
BUCKET_THREADS = True


# ---------------------------------------------------------------------------------------------- (c) loop
def salience_dropout_loop(gradcam_fn, imgs, norm_imgs, drop_iter, P, save_len=SAVE_LEN, after_round0=None):
    """DRV:564-722.  gradcam_fn(imgs [B,3,S,S] cuda) -> [B,T-1,P,P] stands for
    compute_gradcam_ensemble(...)[layer][head].  imgs / norm_imgs are modified in place (pixel blocks zeroed).
    after_round0(g0) is called as soon as the round-0 map is final (its post-processing can start while the remaining
    rounds run).  Returns (gradcam_0, gradcam_agg or None, chosen int32 [B, save_len*drop_iter] or None)."""
    if drop_iter == 1:  # DRV:565-575
        return gradcam_fn(imgs).detach().clone(), None, None
    B, _, S, _ = imgs.shape
    patch = S // P
    chosen = torch.full((B, save_len * drop_iter), -1, dtype=torch.int32, device=imgs.device)
    g0 = agg = None
    for r in range(drop_iter):
        g = gradcam_fn(imgs).detach().contiguous()
        Tm = g.shape[1]
        if r == 0:
            g0 = torch.empty_like(g)
            agg = torch.empty_like(g)
        ops.salience_dropout_round(g, agg, chosen, save_len * r, imgs, norm_imgs, P, patch, 3, Tm - 1, save_len, r,
                                   ensemble_r=g0 if r == 0 else None)
        if r == 0 and after_round0 is not None:
            after_round0(g0)
    return g0, agg, chosen


# ---------------------------------------------------------------------------------------------- (b) batched merge
_SEG_ROWS = {}     # (token id row up to SEP, n_classes, decode) -> [(start, len, div)]: the walk depends on the caption only
_SEG_TABLES = {}   # (rows of a whole batch, device) -> (start, len, div device tensors, max_end): repeated batches upload nothing


def _segment_row(ids_row, n_classes, decode):
    ids = tuple(int(t) for t in ids_row)
    if host.SEP_ID in ids[1:]:
        ids = ids[:ids.index(host.SEP_ID, 1) + 1]
    key = (ids, n_classes, decode)
    if key not in _SEG_ROWS:
        if len(_SEG_ROWS) > 4096:
            _SEG_ROWS.clear()
        _SEG_ROWS[key] = tuple(host.build_token_segments(host.token_strings(list(ids), decode), n_classes))
    return _SEG_ROWS[key]


def segment_tensors(token_ids, decode, class_lists, dev):
    """Host walk of the WordPiece strings (host.build_token_segments) -> the three [B,Cmax] device tables of
    pnp_token_merge plus max_end = the last GradCAM row any segment touches (so the merge need not ask the device).
    Depends on the captions only: both reference passes of a batch share it and repeated captions are cached."""
    B = len(class_lists)
    rows = tuple(_segment_row(token_ids[b], len(class_lists[b]), decode) for b in range(B))
    key = (rows, str(dev))
    if key in _SEG_TABLES:
        return _SEG_TABLES[key]
    Cmax = max(len(c) for c in class_lists)
    start = np.zeros((B, Cmax), np.int32)
    length = np.zeros((B, Cmax), np.int32)
    div = np.ones((B, Cmax), np.float32)
    for b in range(B):
        for c, (s, l, d) in enumerate(rows[b]):
            start[b, c], length[b, c], div[b, c] = s, l, d
    max_end = int((start + length).max()) if start.size else 0
    if len(_SEG_TABLES) > 64:
        _SEG_TABLES.clear()
    _SEG_TABLES[key] = (torch.from_numpy(start).to(dev), torch.from_numpy(length).to(dev), torch.from_numpy(div).to(dev), max_end)
    return _SEG_TABLES[key]


def merge_tokens_batch(gradcam, token_ids, decode, class_lists, segs=None, padded=False):
    """gradcam [B,T-1,P,P]; token_ids [B,>=T] host ints; returns a list of per-image [C_b,P,P] CUDA tensors
    (one pnp_token_merge launch over the batch, padded to the largest C), or with padded=True the [B,Cmax,P,P] tensor itself."""
    if segs is None:
        segs = segment_tensors(token_ids, decode, class_lists, gradcam.device)
    maps = ops.token_merge(gradcam.contiguous(), segs[0], segs[1], segs[2], row_offset=3, max_end=segs[3] if len(segs) > 3 else None)
    if padded:
        return maps
    return [maps[b, :len(class_lists[b])] for b in range(gradcam.shape[0])]


# ---------------------------------------------------------------------------------------------- (d)(e)(f)
class SpatialLatticeCache:
    """The Gaussian-kernel lattice depends on (H, W, sxy) only; build once per shape (SURVEY 7 hard part 1).  Real datasets
    have many ground-truth sizes, so the cache is a small LRU (a 336x336 spatial lattice is about 11 MB)."""

    def __init__(self, max_entries=32):
        import threading
        from collections import OrderedDict
        self._cache = OrderedDict()
        self._max = max_entries
        self._lock = threading.Lock()     # bucket threads look shapes up concurrently

    def get(self, H, W, sxy, device):
        sx, sy = (sxy, sxy) if not isinstance(sxy, (tuple, list)) else sxy
        key = (int(H), int(W), float(sx), float(sy), str(device))
        with self._lock:
            if key in self._cache:
                self._cache.move_to_end(key)
            else:
                self._cache[key] = ops.build_lattice(H, W, (sx, sy), device=device)
                while len(self._cache) > self._max:
                    self._cache.popitem(last=False)
            return self._cache[key]


_SPATIAL = SpatialLatticeCache()


def _mark(stats, name):
    """Stage timing for bench.py: record a CUDA event on the current stream when stats carries an 'events' list."""
    if stats is not None and "events" in stats:
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        stats["events"].append((name, ev))


def postprocess_batch(class_maps, guides, gts, luts, hist, *, threshold, rescale, with_background, mode, n_class,
                      crf=None, bad_count=None, return_labels=False, stats=None, bilateral=None, n_classes=None):
    """class_maps [B,C,P,P] -> labels -> hist (accumulated in place).  guides uint8 [B,H,W,3]; gts float32 [B,H,W];
    luts int32 [B,C'] (composed relabel tables).  mode: the --postprocess string ('', 'blur', 'crf', 'blur+crf').
    gts None (images without ground truth; hist is then unused): returns (ids int32 [B,H,W] relabelled through luts, conf float32
    [B,H,W] = the CRF marginal of each chosen label, or None when the mode has no CRF) instead of counting anything.
    bilateral: a lattice already built over `guides` (the two reference passes of one batch share it).
    n_classes: int32 [B] CUDA tensor when the images have different class counts (class_maps padded to the largest; blurred modes
    only); luts then has Cp columns and the CRF runs over all Cp channels (the dead ones stay at Q = 0)."""
    B, C = class_maps.shape[:2]
    P_grid = class_maps.shape[-1]
    H, W = (gts if gts is not None else guides).shape[1:3]
    N = H * W
    use_blur = bool(mode) and "blur" in mode
    use_crf = bool(mode) and "crf" in mode
    p = dict(CRF_DEFAULTS)
    p.update(crf or {})
    Cc = C + (1 if with_background else 0)
    labels = U = Q = None
    if n_classes is not None and not (use_blur and P_grid <= 32 and USE_LOWRANK_BLUR):
        raise PnpError("per-image class counts need the fused low-rank (d) group (a blurred mode, P <= 32)")
    if use_blur and P_grid <= 32 and USE_LOWRANK_BLUR:
        # blurred maps: the whole (d) group as one fused low-rank launch group that emits the CRF unary (or the labels) directly
        out = ops.lowrank_blur_unary(class_maps.contiguous(), H, W, threshold, rescale, with_background, BLUR_SCALE * max(H, W),
                                     unary=use_crf, labels=not use_crf, n_classes=n_classes)
        if n_classes is not None:
            Cc = ops.crf_pad_channels(Cc)    # every padded channel takes part; the ones an image lacks carry unary +inf
        U, labels = out.get("unary"), out.get("labels")
        _mark(stats, "upsample+blur+unary")
    else:
        x = ops.threshold_upsample(class_maps.contiguous(), H, W, threshold, rescale, with_background)
        _mark(stats, "upsample")
        minmax = None
        if use_blur:
            x, minmax = ops.gaussian_blur(x, BLUR_SCALE * max(H, W), normalize=not use_crf)
            _mark(stats, "blur")
        if use_crf:
            U = ops.crf_unary_from_maps(x.view(B, Cc, N), minmax if use_blur else None)
            _mark(stats, "unary")
        else:
            labels = ops.argmax_channels(x.view(B, Cc, N))
        del x
    if use_crf:
        lat_s = _SPATIAL.get(H, W, p["pos_xy_std"], U.device)
        lat_b = bilateral if bilateral is not None else ops.build_lattice(H, W, p["bi_xy_std"], rgb=guides, srgb=p["bi_rgb_std"])
        if stats is not None:
            stats["M_s"], stats["M_b"], stats["max_row_b"] = lat_s.M, lat_b.M, lat_b.struct.max_row
        _mark(stats, "lattice")
        Q, labels = ops.crf_inference([lat_s, lat_b], [p["pos_w"], p["bi_w"]], U, Cc, p["n_iter"], want_labels=True)
        _mark(stats, "crf")
    if gts is None:
        ids, conf = ops.label_map(labels, luts, Q)
        _mark(stats, "label_map")
        return ids.view(B, H, W), (conf.view(B, H, W) if conf is not None else None)
    pred = torch.empty((B, N), dtype=torch.float32, device=labels.device) if return_labels else None
    ops.confusion_accumulate(labels, gts.view(B, N), n_class, hist, lut=luts, pred_out=pred, bad_count=bad_count)
    _mark(stats, "confusion")
    return pred.view(B, H, W) if return_labels else None


def _as_device_batch(items, members, dtype, dev):
    """items: a device tensor [B,...] (used as is / index-selected) or a list of host arrays (stacked + uploaded)."""
    if isinstance(items, torch.Tensor) and items.is_cuda:
        if len(members) == items.shape[0]:
            return items
        return items[torch.as_tensor(members, device=dev)].contiguous()
    return torch.stack([torch.as_tensor(np.require(items[b], requirements=["C", "W"])).to(dtype) for b in members]).to(dev)


_SIDE_STREAMS = {}
_BUCKET_STREAMS = {}


def _bucket_streams(dev, n):
    key = (dev.type, dev.index)
    pool = _BUCKET_STREAMS.setdefault(key, [])
    while len(pool) < n:
        pool.append(torch.cuda.Stream(device=dev))
    return pool[:n]


_BUCKET_POOL = {}


def _run_on_streams(dev, pool, jobs):
    """jobs[i]() under stream pool[i % len(pool)]: from one host thread per stream when BUCKET_THREADS (launch-bound chains issue
    in parallel), else in order from the calling thread.  Returns the results in order; the first exception is re-raised."""
    if not pool:
        return [job() for job in jobs]

    def under(i, job):
        torch.cuda.set_device(dev)
        with torch.cuda.stream(pool[i % len(pool)]):
            return job()

    if not BUCKET_THREADS or len(jobs) < 2:
        return [under(i, job) for i, job in enumerate(jobs)]
    from concurrent.futures import ThreadPoolExecutor
    n = len(pool)
    if n not in _BUCKET_POOL:
        _BUCKET_POOL[n] = ThreadPoolExecutor(max_workers=n, thread_name_prefix="pnp-bucket")

    def lane(k):   # one thread walks the jobs of one stream in order
        return [(i, under(i, jobs[i])) for i in range(k, len(jobs), n)]

    out = [None] * len(jobs)
    for fut in [_BUCKET_POOL[n].submit(lane, k) for k in range(n)]:
        for i, r in fut.result():
            out[i] = r
    return out


class _null_context:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


def _side_stream(dev):
    key = (dev.type, dev.index)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=dev)
    return _SIDE_STREAMS[key]


def _make_buckets(class_lists, dataset_ids, shapes, gts, guides, *, data_type, mode, patch_num, dev):
    """Group the images of a batch by (channel key, background rule, (H, W) = shapes[b]) and upload each bucket's inputs.
    Returns ({key: members}, {key: (gts [n,H,W] or None when gts is None, guides [n,H,W,3], composed relabel LUTs int32 [n,width])},
    {key: (n_classes int32 [n] when the bucket's class counts differ, else None; largest class count)})."""
    use_blur = bool(mode) and "blur" in mode
    pad_classes = PAD_CLASSES_IN_BUCKETS and use_blur and patch_num <= 32 and USE_LOWRANK_BLUR
    buckets = {}
    for b in range(len(class_lists)):
        C = len(class_lists[b])
        with_bg = host.add_background_rule(data_type, C)
        # with padded classes a bucket holds every class count that pads to the same Cp; else the exact count is part of the key
        ckey = ops.crf_pad_channels(C + (1 if with_bg else 0)) if pad_classes else C
        buckets.setdefault((ckey, with_bg, shapes[b]), []).append(b)
    inputs, ncls = {}, {}
    for key, members in buckets.items():
        with_bg = key[1]
        counts = [len(class_lists[b]) for b in members]
        ragged_c = pad_classes and len(set(counts)) > 1
        width = key[0] if ragged_c else counts[0] + (1 if with_bg else 0)     # LUT columns: Cp when the CRF runs over all of them
        lut_rows = []
        for b in members:
            row = list(host.relabel_lut(dataset_ids[b], with_bg))
            lut_rows.append(row + [0] * (width - len(row)))                    # dead channels are never the argmax
        inputs[key] = (_as_device_batch(gts, members, torch.float32, dev) if gts is not None else None,
                       _as_device_batch(guides, members, torch.uint8, dev), torch.tensor(lut_rows, dtype=torch.int32, device=dev))
        ncls[key] = (torch.tensor(counts, dtype=torch.int32, device=dev), max(counts)) if ragged_c else (None, counts[0])
    return buckets, inputs, ncls


def _n_bucket_streams(buckets, dev):
    """How many CUDA streams the buckets of a batch are spread over (0: everything on the current stream)."""
    return min(int(BUCKET_STREAMS), len(buckets)) if (len(buckets) > 1 and dev.type == "cuda") else 0


def _start_bucket_streams(dev, n_streams):
    """The streams the buckets of a ragged batch are spread over (empty: everything on the current stream).  They start after
    everything already enqueued on the current stream."""
    if not n_streams:
        return []
    cur = torch.cuda.current_stream(dev)
    pool = _bucket_streams(dev, n_streams)
    for st in pool:
        st.wait_stream(cur)
    return pool


def _join_bucket_streams(dev, pool):
    if not pool:
        return
    cur = torch.cuda.current_stream(dev)
    for st in pool:
        cur.wait_stream(st)


def _build_bucket_lattices(buckets, inputs, crf_p, dev, n_streams):
    """{key: bilateral lattice over the bucket's guide images}, and the spatial lattice of every bucket shape cached."""
    keys = list(buckets)
    for key in keys:
        _SPATIAL.get(key[2][0], key[2][1], crf_p["pos_xy_std"], dev)
    pool = _start_bucket_streams(dev, n_streams)
    # every build is enqueued before the first one is waited for (pnp_lattice_finish reads the vertex count back)
    begun = _run_on_streams(dev, pool, [lambda key=key: ops.build_lattice_begin(key[2][0], key[2][1], crf_p["bi_xy_std"], rgb=inputs[key][1],
                                                                                srgb=crf_p["bi_rgb_std"]) for key in keys])
    done = _run_on_streams(dev, pool, [lambda lw=lw: ops.build_lattice_finish(*lw) for lw in begun])
    _join_bucket_streams(dev, pool)
    return dict(zip(keys, done))


def _run_buckets(merged, buckets, ncls, dev, n_streams, one_bucket):
    """one_bucket(key, class_maps) for every bucket, spread over the bucket streams; class_maps are the bucket's rows of the padded
    token-merge output `merged`, cut to the bucket's largest class count.  Returns the results in bucket order."""
    B = merged.shape[0]
    pool = _start_bucket_streams(dev, n_streams)

    def run(key, members):
        c_max = ncls[key][1]
        if len(members) == B and c_max == merged.shape[1]:
            cm = merged
        else:
            cm = merged[torch.as_tensor(members, device=dev), :c_max].contiguous()
        return one_bucket(key, cm)

    out = _run_on_streams(dev, pool, [lambda key=key, members=members: run(key, members) for key, members in buckets.items()])
    _join_bucket_streams(dev, pool)
    return out


def batch_confusion(gradcam_fn, imgs, token_ids, decode, class_lists, dataset_ids, gts, guides, *, drop_iter, patch_num,
                    threshold, data_type, mode, n_class, coco=False, crf=None, norm_imgs=None, stats=None, overlap=False,
                    labels_out=None, bad_count=None, defer=False):
    """One batch of save_img_union_attention: returns (hist_round0 or None, hist_all_drop or None, chosen) with the
    matrices as int64 CUDA tensors [n,n] -- what the reference saves to hist_withfiltered_caption/ and
    all_drop_hist_with_filtered_caption/ (DRV:495-520).  `coco` selects the COCO driver's deltas (DRVC:420, 527, 602).

    imgs [B,3,S,S] cuda (modified in place by the DropOut rounds); gts: float32 [H,W] arrays (list) or one CUDA tensor
    [B,H,W]; guides: uint8 [H,W,3] arrays (list) or one CUDA tensor [B,H,W,3]; dataset_ids[b][i] = id written for
    local class i.

    overlap: the bilateral lattice build and the whole round-0 pass (which needs only the round-0 map) run on a second
    CUDA stream while DropOut rounds 1..R-1 (model passes) occupy the main stream; results are identical either way.
    Off by default: with the model's GEMMs on the tensor cores a B200 runs this workload at its power cap, and co-scheduling
    the memory-bound post-processing under the GEMMs costs more than it hides (bench.py --overlap-ab: 371 ms serial, 380 ms
    overlapped, 384 ms pipelined per step); with SIMT fp32 GEMMs (round 1) the overlap was worth 1.3 %.

    defer (needs overlap and bad_count): ALSO the accumulated-map pass is enqueued on the second stream and the function
    returns as soon as the last model pass has been enqueued, so that the caller's NEXT batch starts its first model pass
    while this batch's post-processing still runs underneath it (cross-batch software pipelining).  The returned matrices
    are then complete only after `pipeline.side_stream(dev)` has been waited for (`join_side_stream`), and the caller must
    not overwrite gts / guides before that.

    labels_out: a dict that receives {"round0" / "all_drop": float32 [B,H,W] relabelled maps} (uniform batches only).
    bad_count: an int32 [1] CUDA tensor that accumulates the number of relabelled ids outside [0, n_class); when given,
    the caller checks it once per run and this function never reads the device back (no host sync per batch)."""
    dev = imgs.device
    B = imgs.shape[0]
    round0_scored = not coco or drop_iter < 3
    timed_stages = stats is not None and "events" in stats
    defer = bool(defer) and bool(overlap) and bad_count is not None and not timed_stages
    use_side = bool(overlap) and not timed_stages and ((drop_iter > 1 and round0_scored) or defer)
    main = torch.cuda.current_stream(dev) if use_side else None
    side = _side_stream(dev) if use_side else None
    use_crf = bool(mode) and "crf" in mode
    crf_p = dict(CRF_DEFAULTS)
    crf_p.update(crf or {})
    _mark(stats, "start")

    # everything that depends on the inputs only: buckets, device copies, relabel LUTs, token segment tables
    buckets, inputs, ncls = _make_buckets(class_lists, dataset_ids, [tuple(gts[b].shape) for b in range(B)], gts, guides,
                                          data_type=data_type, mode=mode, patch_num=patch_num, dev=dev)
    n_streams = _n_bucket_streams(buckets, dev) if not timed_stages else 0
    segs = segment_tensors(token_ids, decode, class_lists, dev)
    hists = {}
    if round0_scored:
        hists["round0"] = torch.zeros((n_class, n_class), dtype=torch.int64, device=dev)
    if drop_iter > 1:
        hists["all_drop"] = torch.zeros((n_class, n_class), dtype=torch.int64, device=dev)
    bad = bad_count if bad_count is not None else torch.zeros(1, dtype=torch.int32, device=dev)
    ev_inputs = main.record_event() if use_side else None
    lattices = {}
    ev_lattices = None

    def build_lattices():  # one bilateral lattice per bucket, shared by both passes (the guide images are the same)
        if use_crf:
            lattices.update(_build_bucket_lattices(buckets, inputs, crf_p, dev, n_streams))
            _mark(stats, "lattice")

    def run_pass(name, gmaps, rescale):
        merged = merge_tokens_batch(gmaps, token_ids, decode, class_lists, segs, padded=True)
        _mark(stats, "merge")

        def one_bucket(key, cm):
            gt, gd, lut = inputs[key]
            return postprocess_batch(cm, gd, gt, lut, hists[name], threshold=threshold, rescale=rescale, with_background=key[1],
                                     mode=mode, n_class=n_class, crf=crf, bad_count=bad, stats=stats, bilateral=lattices.get(key),
                                     return_labels=labels_out is not None, n_classes=ncls[key][0])

        if labels_out is not None and len(buckets) != 1:
            raise PnpError("labels_out needs a uniform batch (one bucket)")
        preds = _run_buckets(merged, buckets, ncls, dev, n_streams, one_bucket)
        if labels_out is not None:
            labels_out[name] = preds[0]

    def side_prologue():
        """First use of the side stream for this batch: inputs visible, lattices built (under the running model pass)."""
        nonlocal ev_lattices
        side.wait_event(ev_inputs)
        for t in (bad,) + tuple(hists.values()) + tuple(x for v in inputs.values() for x in v) + tuple(segs[:3]):
            t.record_stream(side)
        build_lattices()                           # the host waits for the build only (pnp_lattice_finish reads M back)
        ev_lattices = side.record_event()

    def after_round0(g0):
        if not use_side:
            return
        ev_r0 = main.record_event()
        with torch.cuda.stream(side):
            side_prologue()
            if round0_scored:
                side.wait_event(ev_r0)
                g0.record_stream(side)
                run_pass("round0", g0, True)       # 1-round path applies Scale_0_1 (DRV:362)

    g0, agg, chosen = salience_dropout_loop(gradcam_fn, imgs, norm_imgs, drop_iter, patch_num, after_round0=after_round0)
    _mark(stats, "model+gradcam+dropout")
    if use_side and drop_iter == 1:                # the loop made no callback: the only pass there is goes to the side stream now
        after_round0(g0)
    if use_side and defer:
        if agg is not None:
            ev_agg = main.record_event()
            with torch.cuda.stream(side):
                side.wait_event(ev_agg)
                agg.record_stream(side)
                run_pass("all_drop", agg, coco)
        return hists.get("round0"), hists.get("all_drop"), chosen
    if use_side:
        main.wait_event(ev_lattices)
        for lat in lattices.values():
            lat.storage.record_stream(main)
    else:
        build_lattices()
        if round0_scored:
            run_pass("round0", g0, True)
    if agg is not None:
        run_pass("all_drop", agg, coco)            # N-round path: only the COCO driver rescales (DRV:438 vs DRVC:527)
    if use_side:
        main.wait_stream(side)
    if bad_count is None and int(bad.item()):
        raise PnpError("a relabelled id fell outside [0, n_class)")
    return hists.get("round0"), hists.get("all_drop"), chosen


def batch_labels(gradcam_fn, imgs, token_ids, decode, class_lists, guides, *, drop_iter, patch_num, threshold, data_type, mode,
                 crf=None, norm_imgs=None):
    """The batch without ground truth: one label map per image, for images of any size and class list (the in-the-wild use).
    Returns, in batch order, (ids int32 [H_b,W_b], conf float32 [H_b,W_b] or None) CUDA tensors at the size of each guide image:
    ids 0 = background, i = class_lists[b][i-1]; conf = the CRF marginal of the chosen label (None when `mode` has no CRF).

    The post-processed map is the one the reference scores: the accumulated map of the DropOut rounds when drop_iter > 1 (no
    Scale_0_1 outside COCO, DRV:438 / DRVC:527), else the round-0 map (with Scale_0_1, DRV:362).  Buckets, streams, lattice
    builds and post-processing are batch_confusion's, so each image's ids equal the relabelled map a batch of its own gives there.
    imgs [B,3,S,S] cuda (modified in place by the DropOut rounds); guides: uint8 [H_b,W_b,3] arrays (list) or one CUDA tensor
    [B,H,W,3]."""
    dev = imgs.device
    B = imgs.shape[0]
    crf_p = dict(CRF_DEFAULTS)
    crf_p.update(crf or {})
    ids = [list(range(1, len(c) + 1)) for c in class_lists]
    buckets, inputs, ncls = _make_buckets(class_lists, ids, [tuple(guides[b].shape[:2]) for b in range(B)], None, guides,
                                          data_type=data_type, mode=mode, patch_num=patch_num, dev=dev)
    n_streams = _n_bucket_streams(buckets, dev)
    segs = segment_tensors(token_ids, decode, class_lists, dev)
    g0, agg, _ = salience_dropout_loop(gradcam_fn, imgs, norm_imgs, drop_iter, patch_num)
    lattices = _build_bucket_lattices(buckets, inputs, crf_p, dev, n_streams) if (bool(mode) and "crf" in mode) else {}
    gmaps, rescale = (agg, data_type.startswith("coco")) if agg is not None else (g0, True)
    merged = merge_tokens_batch(gmaps, token_ids, decode, class_lists, segs, padded=True)

    def one_bucket(key, cm):
        _, gd, lut = inputs[key]
        return postprocess_batch(cm, gd, None, lut, None, threshold=threshold, rescale=rescale, with_background=key[1], mode=mode,
                                 n_class=None, crf=crf, bilateral=lattices.get(key), n_classes=ncls[key][0])

    out = [None] * B
    for members, (ids_k, conf_k) in zip(buckets.values(), _run_buckets(merged, buckets, ncls, dev, n_streams, one_bucket)):
        for j, b in enumerate(members):
            out[b] = (ids_k[j], conf_k[j] if conf_k is not None else None)
    return out


def side_stream(dev):
    """The second CUDA stream batch_confusion overlaps post-processing on (one per device)."""
    return _side_stream(torch.device(dev) if not isinstance(dev, torch.device) else dev)


def join_side_stream(dev):
    """Make the current stream wait for everything deferred batches have enqueued on the side stream."""
    dev = torch.device(dev) if not isinstance(dev, torch.device) else dev
    torch.cuda.current_stream(dev).wait_stream(_side_stream(dev))


# ---------------------------------------------------------------------------------------------- multi-GPU + files
def allreduce_hist(hist):
    """Sum the int64 confusion matrix over ranks (NCCL over NVLink); no-op without a process group.  This replaces
    the reference's reduce-through-the-filesystem (DRV:513-520 + Calculate_mIoU.py:204-219)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(hist, op=dist.ReduceOp.SUM)
    return hist


def save_hist_npy(hist, save_path, subdir, first_img_id, max_block_num, att_head):
    """Write the matrix in the layout Calculate_mIoU.py expects (DRV:513-520: float64 [n,n] .npy)."""
    import os
    d = os.path.join(save_path, subdir)
    os.makedirs(d, exist_ok=True)
    path = os.path.join(d, "img_%s_max_blocknum_%s_atthead_%s.npy" % (first_img_id, max_block_num, att_head))
    np.save(path, hist.detach().cpu().numpy().astype(np.float64))
    return path
