"""Host-side mirror of the reference's plugin interface for the hot path, over the C ABI (include/artp.h).

Names, argument meaning and error behaviour follow the reference:
  StateValidityChecker   art_planner/include/art_planner/validity_checker/validity_checker.h:21-39
                         (setMap / updateHeightField / hasMap / isValid); installed by Planner
                         (art_planner/src/planner.cpp:125-127,162)
  MotionValidator        ompl::base::MotionValidator::checkMotion as used at
                         art_planner/src/planners/prm_motion_cost.cpp:652 (OMPL DiscreteMotionValidator)
  PathLengthObjective    art_planner/src/objectives/path_length_objective.cpp:26-70
A state is 7 doubles (x y z qx qy qz qw), the SE3StateSpace::StateType fields the reference reads
(art_planner/include/art_planner/utils.h:25-38). Batches are [n, 7] float64 arrays; numpy arrays go through
the host-buffer entry points (H2D/D2H inside), CUDA torch tensors through the *_device entry points on
torch's current stream.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi


def _is_torch_cuda(x) -> bool:
    return hasattr(x, "is_cuda") and bool(x.is_cuda)


class _Handle:
    """Owns one artp_handle (one CUDA device)."""

    def __init__(self, robot_params, device: int = 0, cost_weights=(0.0, 1.0, 5.0), risk_threshold=0.5):
        self.lib = capi.load()
        self.params = robot_params
        self.device = device
        p = capi.make_params(robot_params, device, cost_weights, risk_threshold)
        h = C.c_void_p()
        rc = self.lib.artp_create(C.byref(p), C.byref(h))
        if rc != 0:
            raise capi.ArtpError(rc, self.lib.artp_last_error(None).decode())
        self.h = h

    def check(self, rc: int) -> None:
        if rc != 0:
            raise capi.ArtpError(rc, self.lib.artp_last_error(self.h).decode())

    def close(self) -> None:
        if getattr(self, "h", None):
            self.lib.artp_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def stats(self) -> dict:
        s = capi.ArtpStats()
        self.check(self.lib.artp_get_stats(self.h, C.byref(s)))
        return {k: int(getattr(s, k)) for k, _ in capi.ArtpStats._fields_}


def _stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class StateValidityChecker:
    """art_planner::StateValidityChecker on the GPU (validity_checker.cpp:9-45)."""

    def __init__(self, params, device: int = 0, handle: _Handle | None = None):
        self._h = handle or _Handle(params, device)
        self._map = None

    # -- reference interface ------------------------------------------------------------------
    def setMap(self, synth_map) -> None:             # validity_checker.cpp:20-23
        self._map = synth_map

    def updateHeightField(self, window=None) -> None:   # validity_checker.cpp:27-31 -> setHeightField
        """window = (row0, nrows): upload only that row slab of the map (spatial shard, artp_set_map_window); geometry stays
        that of the full map, so verdicts are identical to a checker holding everything."""
        if self._map is None:
            raise capi.ArtpError(capi.ARTP_E_NOMAP, "setMap() was not called")
        m = self._map
        if window is not None:
            row0, nrows = int(window[0]), int(window[1])
            e = np.asfortranarray(m.elevation[row0:row0 + nrows, :], dtype=np.float32)
            k = np.asfortranarray(m.elevation_masked[row0:row0 + nrows, :], dtype=np.float32)
            self._h.check(self._h.lib.artp_set_map_window(self._h.h, e.ctypes.data, k.ctypes.data, m.elevation.shape[0],
                                                          m.elevation.shape[1], float(m.res), float(m.cx), float(m.cy), row0, nrows))
            return
        e = np.asfortranarray(m.elevation, dtype=np.float32)
        k = np.asfortranarray(m.elevation_masked, dtype=np.float32)
        if e.shape != k.shape:
            raise capi.ArtpError(capi.ARTP_E_INVALID, "layer shapes differ")
        self._h.check(self._h.lib.artp_set_map(self._h.h, e.ctypes.data, k.ctypes.data, e.shape[0], e.shape[1],
                                               float(m.res), float(m.cx), float(m.cy)))

    def hasMap(self) -> bool:                        # validity_checker.cpp:33-35
        return bool(self._h.lib.artp_has_map(self._h.h))

    def isValid(self, state) -> bool:                # validity_checker.cpp:39-45 (batch of 1: latency path)
        s = np.ascontiguousarray(state, dtype=np.float64).reshape(1, 7)
        return bool(self.isValidBatch(s)[0])

    # -- batched entry points -----------------------------------------------------------------
    def isValidBatch(self, states, out=None):
        """states [n, 7] float64 (numpy or CUDA torch tensor) -> uint8 mask of the same kind."""
        lib, h = self._h.lib, self._h
        if _is_torch_cuda(states):
            import torch
            assert states.dtype in (torch.float64, torch.float32) and states.is_contiguous() and states.shape[-1] == 7
            n = states.shape[0]
            if out is None:
                out = torch.empty(n, dtype=torch.uint8, device=states.device)
            fn = lib.artp_check_poses_device if states.dtype == torch.float64 else lib.artp_check_poses_f32_device
            h.check(fn(h.h, C.c_void_p(states.data_ptr()), n, C.c_void_p(out.data_ptr()), _stream_ptr()))
            return out
        f32 = getattr(states, "dtype", None) == np.float32
        s = np.ascontiguousarray(states, dtype=np.float32 if f32 else np.float64)
        assert s.ndim == 2 and s.shape[1] == 7
        n = s.shape[0]
        if out is None:
            out = np.empty(n, dtype=np.uint8)
        fn = lib.artp_check_poses_f32 if f32 else lib.artp_check_poses
        h.check(fn(h.h, s.ctypes.data, n, out.ctypes.data))
        return out

    def sampleValidBatch(self, sampler, n_wanted: int, batch: int = 65536, max_draws: int = 1 << 24):
        """The rejection-sampling loop `do sampleUniform(s) while (!isValid(s))` (prm_motion_cost.cpp:171-194,
        lazy_prm_star_min_update.cpp:549-556) in batches: sampler(m) -> [m, 7] candidates; valid ones are kept in draw
        order until n_wanted states are collected or max_draws candidates were drawn. Returns (states, drawn)."""
        kept, have, drawn = [], 0, 0
        while have < n_wanted and drawn < max_draws:
            m = min(batch, max_draws - drawn)
            cand = np.ascontiguousarray(sampler(m))
            drawn += m
            ok = cand[self.isValidBatch(cand) != 0][: n_wanted - have]
            kept.append(ok)
            have += len(ok)
        return (np.concatenate(kept) if kept else np.zeros((0, 7))), drawn

    def isValidHostPtr(self, states_ptr: int, n: int, valid_ptr: int, f32: bool = False) -> None:
        """Raw host pointers (e.g. pinned torch tensors): the exact call an OMPL adapter makes. f32: the states were
        already cast to float (what Pose3FromSE3 does first) -- identical results, half the H2D bytes."""
        fn = self._h.lib.artp_check_poses_f32 if f32 else self._h.lib.artp_check_poses
        self._h.check(fn(self._h.h, C.c_void_p(states_ptr), n, C.c_void_p(valid_ptr)))

    def compactValid(self, valid, base: int = 0):
        """Ordered indices (int64, base + i) of the non-zero entries of a CUDA uint8 mask; returns (indices, count)
        as CUDA tensors -- the payload of the multi-GPU index all-gather."""
        import torch
        n = valid.shape[0]
        idx = torch.empty(n, dtype=torch.int64, device=valid.device)
        cnt = torch.zeros(1, dtype=torch.int32, device=valid.device)
        self._h.check(self._h.lib.artp_compact_valid_device(self._h.h, C.c_void_p(valid.data_ptr()), n, int(base),
                                                            C.c_void_p(idx.data_ptr()), C.c_void_p(cnt.data_ptr()),
                                                            _stream_ptr()))
        return idx, cnt

    def processBasic(self, elevation, traversability, observed, res: float, bp):
        """processors::Basic::setMaskedElevationAndTraversability (basic.cpp:42-106) on the device, after the inpainting:
        returns (elevation_masked, traversability_thresholded), float32 Fortran-order. bp: an object with the fields of
        artp_basic_params (oracle.basic_oracle.BasicParams has them)."""
        e = np.asfortranarray(elevation, dtype=np.float32)
        t = np.asfortranarray(traversability, dtype=np.float32)
        o = None if observed is None else np.asfortranarray(observed, dtype=np.float32)
        p = capi.ArtpBasicParams(float(bp.traversability_thres), int(bp.unknown_space_untraversable), float(bp.foothold_margin),
                                 float(bp.foothold_margin_max_hole_size), float(bp.foothold_margin_max_drop),
                                 float(bp.foothold_margin_max_drop_search_radius), float(bp.foothold_margin_min_step),
                                 float(bp.foothold_size))
        masked = np.empty(e.shape, np.float32, order="F"); thr = np.empty(e.shape, np.float32, order="F")
        self._h.check(self._h.lib.artp_process_basic(self._h.h, e.ctypes.data, t.ctypes.data, None if o is None else o.ctypes.data,
                                                     e.shape[0], e.shape[1], float(res), C.byref(p), masked.ctypes.data, thr.ctypes.data))
        return masked, thr

    def estimateNormals(self, estimation_radius: float, want_host: bool = True):
        """art_planner::estimateNormals (utils.cpp:213-324) for the current elevation layer, on the device; the layers
        stay resident as the sampler's inputs. Returns (normal_x, normal_y, normal_z, plane_fit_std_dev) float32
        Fortran-order arrays, or None when want_host is False."""
        rows, cols = self._map.elevation.shape
        outs = [np.empty((rows, cols), np.float32, order="F") for _ in range(4)] if want_host else [None] * 4
        self._h.check(self._h.lib.artp_estimate_normals(self._h.h, float(estimation_radius),
                                                        *[None if a is None else a.ctypes.data for a in outs]))
        return tuple(outs) if want_host else None

    def computeSampleCdf(self, sample_probability, want_host: bool = True):
        """computeCumulativeProbabilityDistribution (probability_distribution.cpp:20-46) on the device; the CDF layers stay
        resident for SE3FromSE2Sampler. Returns (cum_prob [rows, cols] F-order, cum_prob_rowwise [rows]) or None."""
        p = np.asfortranarray(sample_probability, dtype=np.float32)
        cum = np.empty(p.shape, np.float32, order="F") if want_host else None
        row = np.empty(p.shape[0], np.float32) if want_host else None
        self._h.check(self._h.lib.artp_compute_sample_cdf(self._h.h, p.ctypes.data, None if cum is None else cum.ctypes.data,
                                                          None if row is None else row.ctypes.data))
        return (cum, row) if want_host else None

    def computeChange(self, map_new, map_old, height_change_for_update: float, want_layer: bool = True, out=None):
        """processors::computeChange (change.cpp:9-51) on the device. map_new / map_old: objects with `elevation` and
        `traversability_thresholded` ([rows, cols], grid_map column-major), `res`, `cx`, `cy`. numpy layers go through the
        host entry point and return the float `updated` layer of the new map (Fortran-order, exact 0 / 1; None when
        want_layer is False). CUDA float32 torch layers -- [rows, cols] views with column-major strides, e.g. `t.t()` of a
        contiguous [cols, rows] tensor -- go through the device entry point on torch's current stream and return the
        layer as such a view (or fill `out`). The bit-packed layer stays on the handle for roadmapUpdates()."""
        lib, h = self._h.lib, self._h
        thr = float(height_change_for_update)
        if _is_torch_cuda(map_new.elevation):
            import torch
            grids = []
            for m in (map_new, map_old):
                for a in (m.elevation, m.traversability_thresholded):
                    assert _is_torch_cuda(a) and a.dtype == torch.float32 and a.dim() == 2 and a.t().is_contiguous()
                assert m.elevation.shape == m.traversability_thresholded.shape
                rows, cols = m.elevation.shape
                grids.append(capi.ArtpGrid(m.elevation.data_ptr(), m.traversability_thresholded.data_ptr(), rows, cols,
                                           float(m.res), float(m.cx), float(m.cy)))
            if out is None and want_layer:
                rows, cols = map_new.elevation.shape
                out = torch.empty((cols, rows), dtype=torch.float32, device=map_new.elevation.device).t()
            if out is not None:
                assert out.shape == map_new.elevation.shape and out.t().is_contiguous()
            h.check(lib.artp_compute_change_device(h.h, C.byref(grids[0]), C.byref(grids[1]), thr,
                                                   None if out is None else C.c_void_p(out.data_ptr()), _stream_ptr()))
            return out
        keep, grids = [], []
        for m in (map_new, map_old):
            e = np.asfortranarray(m.elevation, dtype=np.float32)
            t = np.asfortranarray(m.traversability_thresholded, dtype=np.float32)
            if e.shape != t.shape:
                raise capi.ArtpError(capi.ARTP_E_INVALID, "layer shapes differ")
            keep += [e, t]
            grids.append(capi.ArtpGrid(e.ctypes.data, t.ctypes.data, e.shape[0], e.shape[1], float(m.res), float(m.cx),
                                       float(m.cy)))
        upd = np.empty(keep[0].shape, np.float32, order="F") if want_layer else None
        h.check(lib.artp_compute_change(h.h, C.byref(grids[0]), C.byref(grids[1]), thr,
                                        None if upd is None else upd.ctypes.data))
        return upd

    def roadmapUpdates(self, vertex_states, edges, out_vertex=None, out_edge=None):
        """LazyPRMStarMinUpdateMaintainer::update's per-vertex / per-edge questions (lazy_prm_star_min_update.cpp:18-91)
        against the last computeChange() layer: vertex_states [nv, 7] float64, edges [ne, 2] (source, target) vertex
        indices -> (vertex_flags [nv], edge_flags [ne]) uint8: 0 keep, 1 updated (-> VALIDITY_UNKNOWN), 2 outside the new
        map (vertex removed; edge removed with it). numpy arrays use the host entry point (edges as uint32); CUDA torch
        tensors (float64 states, int32 edges: same bits as uint32 below 2^31) the device entry point on torch's current
        stream -- there a bad edge index is reported by pollError()."""
        lib, h = self._h.lib, self._h
        if _is_torch_cuda(vertex_states):
            import torch
            assert vertex_states.dtype == torch.float64 and vertex_states.is_contiguous() and vertex_states.shape[-1] == 7
            assert edges.dtype == torch.int32 and edges.is_contiguous() and edges.shape[-1] == 2
            nv, ne = vertex_states.shape[0], edges.shape[0]
            if out_vertex is None:
                out_vertex = torch.empty(nv, dtype=torch.uint8, device=vertex_states.device)
            if out_edge is None:
                out_edge = torch.empty(ne, dtype=torch.uint8, device=vertex_states.device)
            h.check(lib.artp_roadmap_updates_device(h.h, C.c_void_p(vertex_states.data_ptr()), nv, C.c_void_p(edges.data_ptr()),
                                                    ne, C.c_void_p(out_vertex.data_ptr()), C.c_void_p(out_edge.data_ptr()),
                                                    _stream_ptr()))
            return out_vertex, out_edge
        s = np.ascontiguousarray(vertex_states, dtype=np.float64).reshape(-1, 7)
        e = np.asarray(edges).reshape(-1, 2)
        if e.size and (e.min() < 0 or e.max() > 0xFFFFFFFF):
            raise capi.ArtpError(capi.ARTP_E_INVALID, "edge index outside the uint32 range")
        e = np.ascontiguousarray(e, dtype=np.uint32)
        nv, ne = s.shape[0], e.shape[0]
        vf = np.empty(nv, np.uint8) if out_vertex is None else out_vertex
        ef = np.empty(ne, np.uint8) if out_edge is None else out_edge
        h.check(lib.artp_roadmap_updates(h.h, s.ctypes.data, nv, e.ctypes.data, ne, vf.ctypes.data, ef.ctypes.data))
        return vf, ef

    def isValidBatchBits(self, states, out_valid, out_bits):
        """One shard step of the multi-GPU path: verdict bytes + bit-packed mask (CUDA float64 states), one call."""
        n = states.shape[0]
        self._h.check(self._h.lib.artp_check_poses_bits_device(self._h.h, C.c_void_p(states.data_ptr()), n,
                                                               C.c_void_p(out_valid.data_ptr()), C.c_void_p(out_bits.data_ptr()),
                                                               _stream_ptr()))

    def compactValidU32(self, valid, base: int = 0, out_idx=None, out_cnt=None):
        """Ordered 32-bit indices (base + i) of the non-zero entries of a CUDA uint8 mask -> (indices int32 view, count)."""
        import torch
        n = valid.shape[0]
        if out_idx is None:
            out_idx = torch.empty(n, dtype=torch.int32, device=valid.device)
        if out_cnt is None:
            out_cnt = torch.zeros(1, dtype=torch.int32, device=valid.device)
        self._h.check(self._h.lib.artp_compact_valid_u32_device(self._h.h, C.c_void_p(valid.data_ptr()), n, int(base),
                                                                C.c_void_p(out_idx.data_ptr()), C.c_void_p(out_cnt.data_ptr()),
                                                                _stream_ptr()))
        return out_idx, out_cnt

    def packValidBits(self, valid, out=None):
        """CUDA uint8 mask [n] -> bit-packed int32 words [(n+31)//32] (item i = bit i&31 of word i>>5)."""
        import torch
        n = valid.shape[0]
        if out is None:
            out = torch.empty((n + 31) // 32, dtype=torch.int32, device=valid.device)
        self._h.check(self._h.lib.artp_pack_valid_bits_device(self._h.h, C.c_void_p(valid.data_ptr()), n,
                                                              C.c_void_p(out.data_ptr()), _stream_ptr()))
        return out

    def compactBits(self, bits, n: int, base: int = 0, out_idx=None, out_cnt=None):
        """Ordered indices of the set bits among the first n of a bit-packed CUDA mask -> (indices int64 [n], count)."""
        import torch
        if out_idx is None:
            out_idx = torch.empty(n, dtype=torch.int64, device=bits.device)
        if out_cnt is None:
            out_cnt = torch.empty(1, dtype=torch.int32, device=bits.device)
        self._h.check(self._h.lib.artp_compact_bits_device(self._h.h, C.c_void_p(bits.data_ptr()), n, int(base),
                                                           C.c_void_p(out_idx.data_ptr()), C.c_void_p(out_cnt.data_ptr()),
                                                           _stream_ptr()))
        return out_idx, out_cnt

    def setMode(self, mode: int) -> None:
        self._h.check(self._h.lib.artp_set_mode(self._h.h, int(mode)))

    def pollError(self) -> None:
        """Raise ArtpError(ARTP_E_LIMIT) if an asynchronous (device-buffer) call hit the plane-grouping overflow since the
        last poll (the affected poses were reported invalid). Synchronise the stream first."""
        self._h.check(self._h.lib.artp_poll_error(self._h.h))

    def debugSetGroupCapacity(self, max_triangles: int) -> None:
        self._h.check(self._h.lib.artp_debug_set_group_capacity(self._h.h, int(max_triangles)))

    def stats(self) -> dict:
        return self._h.stats()

    def setTiming(self, enable: bool) -> None:
        self._h.check(self._h.lib.artp_set_timing(self._h.h, int(bool(enable))))

    def lastKernelTimesMs(self):
        """(classify ms, box warp stage ms, plane-grouping stage ms) of the most recent check call (CUDA events
        recorded by the library on the call's stream)."""
        ms = (C.c_float * 3)()
        self._h.check(self._h.lib.artp_get_last_timing(self._h.h, ms))
        return float(ms[0]), float(ms[1]), float(ms[2])

    def lastStageTimesMs(self):
        """(classify, big-tile queue, reach queue (warp per box), reach queue (8-lane groups), plane grouping) ms of the most recent
        check call."""
        ms = (C.c_float * 5)()
        self._h.check(self._h.lib.artp_get_last_stage_timing(self._h.h, ms))
        return tuple(float(x) for x in ms)

    @property
    def handle(self) -> _Handle:
        return self._h


class SE3FromSE2Sampler:
    """art_planner::SE3FromSE2Sampler::sampleUniform (src/sampler.cpp:82-131) on the device, plus the fused
    sample -> isValid -> compact form of the rejection loops around it (prm_motion_cost.cpp:171-194).

    `layers` carries normal_x/y/z, plane_fit_std_dev, cum_prob, cum_prob_rowwise (grid_map matrices);
    `sp` the sampler parameters (max_roll_pert, max_pitch_pert, sample_from_distribution, low, high).
    Must be re-created / setLayers() again after every setMap on the checker."""

    def __init__(self, checker: StateValidityChecker, layers, sp, seed: int = 0):
        self._c = checker
        self.seed = int(seed)
        self._next = 0
        self.setLayers(layers, sp)

    def setLayers(self, layers, sp) -> None:
        h, lib = self._c.handle, self._c.handle.lib
        f = lambda a: None if a is None else np.asfortranarray(a, dtype=np.float32)
        keep = [f(getattr(layers, "normal_x", None)), f(getattr(layers, "normal_y", None)),
                f(getattr(layers, "normal_z", None)), f(getattr(layers, "plane_fit_std_dev", None)),
                f(getattr(layers, "cum_prob", None)),
                None if getattr(layers, "cum_prob_rowwise", None) is None
                else np.ascontiguousarray(layers.cum_prob_rowwise, dtype=np.float32)]
        p = capi.ArtpSamplerParams(float(sp.max_roll_pert), float(sp.max_pitch_pert), int(sp.sample_from_distribution),
                                   (C.c_double * 2)(*sp.low), (C.c_double * 2)(*sp.high))
        h.check(lib.artp_set_sampler(h.h, C.byref(p), *[None if a is None else a.ctypes.data for a in keep]))

    def uniforms(self, first: int, n: int) -> np.ndarray:
        """The [n, 6] uniform01 variates of samples first..first+n-1 of this sampler's Philox stream."""
        h, lib = self._c.handle, self._c.handle.lib
        u = np.empty((n, 6), np.float64)
        h.check(lib.artp_sampler_uniforms(h.h, self.seed, int(first), n, u.ctypes.data))
        return u

    def sampleUniformBatch(self, n: int, u=None, first=None, want_cells: bool = False):
        """n candidates [n, 7]. u: optional [n, 6] variates (else the Philox stream from `first`, default: continue)."""
        h, lib = self._c.handle, self._c.handle.lib
        if first is None:
            first = self._next
            if u is None:
                self._next += n
        states = np.empty((n, 7), np.float64)
        rc = np.empty((n, 2), np.int32) if want_cells else None
        uu = None if u is None else np.ascontiguousarray(u, dtype=np.float64)
        assert uu is None or uu.shape == (n, 6)
        h.check(lib.artp_sample_states(h.h, None if uu is None else uu.ctypes.data, self.seed, int(first), n,
                                       states.ctypes.data, None if rc is None else rc.ctypes.data))
        return (states, rc) if want_cells else states

    def sampleUniform(self) -> np.ndarray:
        """One state, never NaN: in uniform mode a draw outside the map is redrawn from the next counter of the stream,
        like samplePositionInMap's loop (sampler.cpp:46-50)."""
        while True:
            s = self.sampleUniformBatch(1)[0]
            if not np.isnan(s[0]):
                return s

    def sampleUniformInside(self, n: int) -> np.ndarray:
        """n states, none NaN, in draw order (rejected outside-map candidates of the uniform mode are redrawn)."""
        out = []
        have = 0
        while have < n:
            s = self.sampleUniformBatch(n - have)
            s = s[~np.isnan(s[:, 0])]
            out.append(s)
            have += len(s)
        return np.concatenate(out) if out else np.zeros((0, 7))

    def sampleValidBatch(self, n_draw: int, first=None, capacity=None, out=None):
        """Draw n_draw candidates on the device, check them, return (valid states in draw order, n_valid).
        out: optional reusable [cap, 7] float64 host buffer (numpy array or pinned CPU torch tensor); a fresh
        58 MB numpy array per 2^20 draws costs more in page faults than the whole GPU pass."""
        h, lib = self._c.handle, self._c.handle.lib
        if first is None:
            first = self._next
            self._next += n_draw
        if out is None:
            cap = n_draw if capacity is None else int(capacity)
            out = np.empty((cap, 7), np.float64)
        else:
            cap = out.shape[0] if capacity is None else min(int(capacity), out.shape[0])
        ptr = out.ctypes.data if isinstance(out, np.ndarray) else out.data_ptr()
        nv = C.c_size_t(0)
        h.check(lib.artp_sample_valid(h.h, self.seed, int(first), n_draw, C.c_void_p(ptr), cap, C.byref(nv)))
        return out[: min(nv.value, cap)], nv.value

    def sampleValidDevice(self, n_draw: int, first: int, out, count):
        """Device buffers: out = CUDA float64 [cap, 7], count = CUDA int32 [1]; asynchronous on the current stream."""
        h, lib = self._c.handle, self._c.handle.lib
        h.check(lib.artp_sample_valid_device(h.h, self.seed, int(first), n_draw, C.c_void_p(out.data_ptr()), out.shape[0],
                                             C.c_void_p(count.data_ptr()), _stream_ptr()))


class MotionValidator:
    """Discrete motion validation over StateValidityChecker (OMPL DiscreteMotionValidator semantics with a fixed
    segment count): valid(s2) and valid(interpolate(s1, s2, j/(n_steps+1))) for j = 1..n_steps."""

    def __init__(self, checker: StateValidityChecker, n_steps: int = 20):
        self._c = checker
        self.n_steps = int(n_steps)

    def checkMotion(self, s1, s2) -> bool:
        a = np.ascontiguousarray(s1, dtype=np.float64).reshape(1, 7)
        b = np.ascontiguousarray(s2, dtype=np.float64).reshape(1, 7)
        return bool(self.checkMotionBatch(a, b)[0])

    def checkMotionBatch(self, s1, s2, out=None):
        h, lib = self._c.handle, self._c.handle.lib
        if _is_torch_cuda(s1):
            import torch
            assert s1.dtype == torch.float64 and s2.dtype == torch.float64 and s1.is_contiguous() and s2.is_contiguous()
            n = s1.shape[0]
            if out is None:
                out = torch.empty(n, dtype=torch.uint8, device=s1.device)
            h.check(lib.artp_check_motions_device(h.h, C.c_void_p(s1.data_ptr()), C.c_void_p(s2.data_ptr()), n,
                                                  self.n_steps, C.c_void_p(out.data_ptr()), _stream_ptr()))
            return out
        a = np.ascontiguousarray(s1, dtype=np.float64)
        b = np.ascontiguousarray(s2, dtype=np.float64)
        n = a.shape[0]
        if out is None:
            out = np.empty(n, dtype=np.uint8)
        h.check(lib.artp_check_motions(h.h, a.ctypes.data, b.ctypes.data, n, self.n_steps, out.ctypes.data))
        return out

    @staticmethod
    def se3Space(synth_map, reach_z: float, fraction: float = 0.01):
        """The SE3 space parameters Planner::setMap installs (planner.cpp:146-156): x, y bounds = map centre +- the FULL
        map length, z bounds = finite elevation range -+ reach.z / 2; OMPL's default longest-valid-segment fraction."""
        lx, ly = synth_map.length
        e = synth_map.elevation[np.isfinite(synth_map.elevation)]
        return capi.ArtpSe3Space((C.c_double * 3)(synth_map.cx - lx, synth_map.cy - ly, float(e.min()) - reach_z / 2),
                                 (C.c_double * 3)(synth_map.cx + lx, synth_map.cy + ly, float(e.max()) + reach_z / 2), float(fraction))

    def validSegmentCount(self, space, s1, s2):
        """SE3StateSpace::validSegmentCount per edge (OMPL 1.4.2 rule, host arithmetic)."""
        a = np.ascontiguousarray(s1, dtype=np.float64); b = np.ascontiguousarray(s2, dtype=np.float64)
        nd = np.empty(a.shape[0], np.int32)
        self._c.handle.check(self._c.handle.lib.artp_valid_segment_count(C.byref(space), a.ctypes.data, b.ctypes.data, a.shape[0],
                                                                         nd.ctypes.data))
        return nd

    def checkMotionSegments(self, s1, s2, nd=None, space=None):
        """DiscreteMotionValidator::checkMotion(s1, s2, lastValid) for a batch with per-edge segment counts (nd, or the OMPL
        rule from `space`): returns (valid uint8 [n], lastValid.second float64 [n])."""
        h, lib = self._c.handle, self._c.handle.lib
        a = np.ascontiguousarray(s1, dtype=np.float64); b = np.ascontiguousarray(s2, dtype=np.float64)
        n = a.shape[0]
        seg = None if nd is None else np.ascontiguousarray(nd, dtype=np.int32)
        valid = np.empty(n, np.uint8); t = np.empty(n, np.float64)
        h.check(lib.artp_check_motions_segments(h.h, a.ctypes.data, b.ctypes.data, n, None if seg is None else seg.ctypes.data,
                                                None if space is None else C.byref(space), valid.ctypes.data, t.ctypes.data))
        return valid, t

    def checkEdgeInteriors(self, s1, s2, n_interp=None, max_lateral: float = 0.5):
        """PRMMotionCost::addValidMilestone's connection loop (prm_motion_cost.cpp:341-372) over a batch of candidate
        edges: per edge the number of leading valid interior states (== n_interp[e] iff the connection is valid).
        Returns (valid_prefix, n_interp). Host arrays, or CUDA float64 tensors (then n_interp must be given as an
        int tensor / array and the prefix sums are built with torch)."""
        h, lib = self._c.handle, self._c.handle.lib
        if _is_torch_cuda(s1):
            import torch
            assert s1.dtype == torch.float64 and s2.dtype == torch.float64 and s1.is_contiguous() and s2.is_contiguous()
            n = s1.shape[0]
            if n_interp is None:
                d = torch.sqrt((s2[:, 0] - s1[:, 0]) ** 2 + (s2[:, 1] - s1[:, 1]) ** 2)
                n_interp = (d / max_lateral).to(torch.int64)
            ni = torch.as_tensor(n_interp, device=s1.device).to(torch.int64)
            off = torch.zeros(n + 1, dtype=torch.int64, device=s1.device)
            off[1:] = torch.cumsum(ni, 0)
            total = int(off[-1].item())
            off32 = off.to(torch.int32).contiguous()      # same bits as uint32 below 2^31
            assert total < 2 ** 31
            flags = torch.empty(max(total, 1), dtype=torch.uint8, device=s1.device)
            out = torch.empty(n, dtype=torch.int32, device=s1.device)
            h.check(lib.artp_check_edge_interiors_device(
                h.h, C.c_void_p(s1.data_ptr()), C.c_void_p(s2.data_ptr()), n, C.c_void_p(off32.data_ptr()), total,
                C.c_void_p(flags.data_ptr()), C.c_void_p(out.data_ptr()), _stream_ptr()))
            return out, ni.to(torch.int32)
        a = np.ascontiguousarray(s1, dtype=np.float64)
        b = np.ascontiguousarray(s2, dtype=np.float64)
        n = a.shape[0]
        out = np.empty(n, dtype=np.int32)
        if n_interp is None:
            d = np.sqrt((b[:, 0] - a[:, 0]) ** 2 + (b[:, 1] - a[:, 1]) ** 2)
            ni = (d / max_lateral).astype(np.uint32).astype(np.int32)
        else:
            ni = np.ascontiguousarray(n_interp, dtype=np.int32)
        h.check(lib.artp_check_edge_interiors(h.h, a.ctypes.data, b.ctypes.data, n,
                                              None if n_interp is None else ni.ctypes.data, float(max_lateral),
                                              out.ctypes.data))
        return out, ni


class PathLengthObjective:
    """art_planner::PathLengthObjective::motionCost (path_length_objective.cpp:26-70), batched."""

    def __init__(self, checker: StateValidityChecker):
        self._c = checker

    def motionCost(self, s1, s2) -> float:
        a = np.ascontiguousarray(s1, dtype=np.float64).reshape(1, 7)
        b = np.ascontiguousarray(s2, dtype=np.float64).reshape(1, 7)
        return float(self.motionCostBatch(a, b)[0])

    def motionCostBatch(self, s1, s2, out=None):
        h, lib = self._c.handle, self._c.handle.lib
        if _is_torch_cuda(s1):
            import torch
            n = s1.shape[0]
            if out is None:
                out = torch.empty(n, dtype=torch.float64, device=s1.device)
            h.check(lib.artp_path_length_cost_device(h.h, C.c_void_p(s1.data_ptr()), C.c_void_p(s2.data_ptr()), n,
                                                     C.c_void_p(out.data_ptr()), _stream_ptr()))
            return out
        a = np.ascontiguousarray(s1, dtype=np.float64)
        b = np.ascontiguousarray(s2, dtype=np.float64)
        n = a.shape[0]
        if out is None:
            out = np.empty(n, dtype=np.float64)
        h.check(lib.artp_path_length_cost(h.h, a.ctypes.data, b.ctypes.data, n, out.ctypes.data))
        return out


class MotionCostObjective:
    """art_planner::MotionCostObjective's batch cost functor (objectives/motion_cost_objective.h:22-66,
    motion_cost_objective.cpp:28-33) backed by the on-device network instead of the ROS cost server
    (art_planner_ros/src/planner_ros.cpp:283-308)."""

    def __init__(self, checker: StateValidityChecker):
        self._c = checker

    def setWeights(self, state_dict) -> None:
        """Parameters keyed like the reference module's state_dict (numpy arrays or torch tensors)."""
        from . import costnet
        sd = {k: (v.detach().cpu().numpy() if hasattr(v, "detach") else np.asarray(v)) for k, v in state_dict.items()}
        blob = costnet.pack_blob(sd)
        h = self._c.handle
        assert blob.size == h.lib.artp_cost_weights_size()
        h.check(h.lib.artp_set_cost_weights(h.h, blob.ctypes.data, blob.size))

    def updateFeatures(self) -> None:
        """CostPredictor.updateFeatures over the checker's current map (predictor.py:28-36)."""
        h = self._c.handle
        h.check(h.lib.artp_update_features(h.h))

    def costQuery(self, edge_matrix, out=None):
        """edge_matrix [n, 6] float32 = [tx, ty, tyaw, sx, sy, syaw] -> [n, 3] float32 (energy, time, risk)."""
        h, lib = self._c.handle, self._c.handle.lib
        if _is_torch_cuda(edge_matrix):
            import torch
            assert edge_matrix.dtype == torch.float32 and edge_matrix.is_contiguous()
            n = edge_matrix.shape[0]
            if out is None:
                out = torch.empty((n, 3), dtype=torch.float32, device=edge_matrix.device)
            h.check(lib.artp_motion_cost_device(h.h, C.c_void_p(edge_matrix.data_ptr()), n, C.c_void_p(out.data_ptr()),
                                                _stream_ptr()))
            return out
        e = np.ascontiguousarray(edge_matrix, dtype=np.float32)
        n = e.shape[0]
        if out is None:
            out = np.empty((n, 3), dtype=np.float32)
        h.check(lib.artp_motion_cost(h.h, e.ctypes.data, n, out.ctypes.data))
        return out

    def edgeMatrixFromStates(self, s_start, s_target):
        """[n, 6] float32 rows [tx, ty, tyaw, sx, sy, syaw] as PRMMotionCostMaintainer::updateEdges fills them."""
        a = np.ascontiguousarray(s_start, dtype=np.float64); b = np.ascontiguousarray(s_target, dtype=np.float64)
        out = np.empty((a.shape[0], 6), np.float32)
        self._c.handle.check(self._c.handle.lib.artp_edge_matrix_from_states(a.ctypes.data, b.ctypes.data, a.shape[0], out.ctypes.data))
        return out

    def updateEdgesBatch(self, s_start, s_target):
        """PRMMotionCostMaintainer::updateEdges / computeCostForVertexEdges for n graph edges in one call: edge matrix ->
        cost query -> isFeasible / getCost. Returns (cost float64 [n] with +inf for infeasible edges, feasible uint8 [n],
        cost3 float32 [n, 3])."""
        h = self._c.handle
        a = np.ascontiguousarray(s_start, dtype=np.float64); b = np.ascontiguousarray(s_target, dtype=np.float64)
        n = a.shape[0]
        cost = np.empty(n, np.float64); feas = np.empty(n, np.uint8); c3 = np.empty((n, 3), np.float32)
        h.check(h.lib.artp_motion_cost_states(h.h, a.ctypes.data, b.ctypes.data, n, cost.ctypes.data, feas.ctypes.data, c3.ctypes.data))
        return cost, feas, c3

    def getCost(self, cost3):
        """(cost, feasible) per edge: w_e*E + w_t*T + w_r*R and R <= risk_threshold (motion_cost_objective.h:54-66)."""
        h = self._c.handle
        c = np.ascontiguousarray(cost3, dtype=np.float32)
        n = c.shape[0]
        cost = np.empty(n, dtype=np.float64)
        feas = np.empty(n, dtype=np.uint8)
        h.check(h.lib.artp_combine_cost(h.h, c.ctypes.data, n, cost.ctypes.data, feas.ctypes.data))
        return cost, feas

    def features(self):
        """[Hf, Wf, 48] float32 feature map (test hook)."""
        h = self._c.handle
        hf, wf = C.c_int(), C.c_int()
        h.check(h.lib.artp_get_features(h.h, None, 0, C.byref(hf), C.byref(wf)))
        out = np.empty((hf.value, wf.value, 48), dtype=np.float32)
        h.check(h.lib.artp_get_features(h.h, out.ctypes.data, out.size, C.byref(hf), C.byref(wf)))
        return out

    def setMode(self, mode: int) -> None:
        h = self._c.handle
        h.check(h.lib.artp_set_cnn_mode(h.h, int(mode)))

    def lastTrunkTimesMs(self):
        ms = (C.c_float * 3)()
        self._c.handle.check(self._c.handle.lib.artp_get_cnn_timing(self._c.handle.h, ms))
        return float(ms[0]), float(ms[1]), float(ms[2])
