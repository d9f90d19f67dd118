"""Dry run of GPU test BODIES on a box without a GPU: the `gpu_ctx` fixture is replaced by a stand-in with the same
methods answered by the CPU oracle (TEST INFRASTRUCTURE; nothing here is product code).  This checks the tests'
own logic - indexing, shapes, fixtures, tolerances against the exact values - before they meet the device; it says
nothing about the kernels.

    python tools/dryrun_gpu_tests.py            # the tests listed at the bottom
    python tools/dryrun_gpu_tests.py largest    # only the tile-matrix cases whose name contains 'largest'
"""
import os
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import oracle  # noqa: E402

oracle.build()


class _H:
    def __init__(self, **kw):
        self.__dict__.update(kw)

    def close(self):
        pass


class _Env(_H):
    def offsets(self):
        """Offsets from the oracle's environment sizes."""
        sizes = []
        for s, prim in zip(self.struct, self.prim):
            key = (int(s), int(prim))
            if key not in self.sizes:
                S = slice(self.st.off[s], self.st.off[s + 1])
                xyz = self.st.xyz[S]
                self.sizes[key] = len(oracle.environment(self.p, xyz, np.zeros(len(xyz), np.uint16), self.st.tag[S],
                                                         int(prim), self.thr)[0])
            sizes.append(self.sizes[key])
        return np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)


class OracleCtx:
    tile_launches = 0

    def set_params(self, n_categories, weight_functions=(("uniform", (3.0, 10.0)),), category_weights=None,
                   statistical_distance=("Hellinger", (2.0,)), tag_rule=None):
        self.p = oracle.Params(n_categories, [(n, list(q)) for n, q in weight_functions], category_weights,
                               (statistical_distance[0], list(statistical_distance[1])), tag_rule)
        # what decides whether score_jobs_stats may take the tile kernel (locohd_capi.cu, locohd_score_jobs_stats)
        self.tile_config = (len(weight_functions) == 1 and statistical_distance[0] == "Hellinger" and
                            list(statistical_distance[1]) == [2.0] and
                            (category_weights is None or all(w == 1.0 for w in category_weights)))
        self.n_categories = n_categories

    def from_primitives(self, xa, ca, ta, xb, cb, tb, anchors, thr, wf_idx=None):
        return oracle.from_primitives(self.p, xa, ca, ta, xb, cb, tb, anchors, thr, wf_idx=wf_idx)

    def from_primitives_grad(self, xa, ca, ta, xb, cb, tb, anchors, thr, wf_idx=None, pair_weights=None, out=None,
                             grad_a=None, grad_b=None):
        import grad_reference
        from loco_hd_b200 import _capi
        try:
            s, ga, gb = grad_reference.from_primitives_grad(oracle, self.p, xa, ca, ta, xb, cb, tb, anchors, thr,
                                                            wf_idx=wf_idx, pair_weights=pair_weights)
        except oracle.OracleError as e:
            raise _capi.LocoHDError(e.status, str(e))
        for dst, src in ((grad_a, ga), (grad_b, gb)):
            if dst is not None:
                dst[...] = src
        return s, ga if grad_a is None else grad_a, gb if grad_b is None else grad_b

    def wf_integral_points(self, name, params, x):
        return np.array([oracle.wf_integral_point(name, list(params), float(v)) for v in x])

    def wf_density_points(self, name, params, x):
        import grad_reference
        return np.array([grad_reference.wf_density(name, params, float(v)) for v in x])

    def structs_create(self, offs, xyz, cat, tag):
        return _H(off=np.asarray(offs, dtype=np.int64), xyz=np.asarray(xyz, dtype=np.float64), cat=np.asarray(cat), tag=np.asarray(tag))

    def structure(self, xyz, cat, tag):
        return self.structs_create([0, len(cat)], xyz, cat, tag)

    def envset_build(self, st, prim, thr, anchor_struct=None, keep_indices=False):
        prim = np.asarray(prim)
        s = np.zeros(len(prim), dtype=np.int64) if anchor_struct is None else np.asarray(anchor_struct, dtype=np.int64)
        return _Env(st=st, prim=prim, struct=s, thr=thr, p=self.p, sizes={})

    def _pair(self, ea, ia, eb, ib):
        sa, sb = int(ea.struct[ia]), int(eb.struct[ib])
        A, B = slice(ea.st.off[sa], ea.st.off[sa + 1]), slice(eb.st.off[sb], eb.st.off[sb + 1])
        return A, B

    def score_pairs(self, ea, eb, pairs):
        out = []
        for ia, ib in np.asarray(pairs).reshape(-1, 2):
            A, B = self._pair(ea, ia, eb, ib)
            out.append(oracle.from_primitives(self.p, ea.st.xyz[A], ea.st.cat[A], ea.st.tag[A], eb.st.xyz[B], eb.st.cat[B],
                                              eb.st.tag[B], [(int(ea.prim[ia]), int(eb.prim[ib]))], ea.thr)[0])
        return np.array(out)

    def _takes_tiles(self, ea, eb, jobs):
        """The library's choice of the tile kernel, from the same host queries it uses."""
        from loco_hd_b200 import _capi
        if int(os.environ.get("LOCOHD_NO_TILES") or 0) or not self.tile_config or len(jobs) < 4:
            return False
        if len(set(int(n) for n in jobs["n"])) != 1 or int(jobs["n"][0]) == 0:
            return False
        if not _capi.plan_job_tiles(jobs)["pays"]:
            return False
        max_a, max_b = (int(np.diff(e.offsets().astype(np.int64)).max()) for e in (ea, eb))
        return _capi.tile_geometry(self.n_categories, max_a, max_b)["teams"] >= 6

    def score_jobs_stats(self, ea, eb, jobs, scores=False, job_means=False, anchor_means=False, anchor_stds=False):
        from loco_hd_b200 import _capi
        jobs = np.asarray(jobs)
        if self._takes_tiles(ea, eb, jobs):
            self.tile_launches += 1
        all_scores = []
        for a0, b0, n in [(int(j["a_first"]), int(j["b_first"]), int(j["n"])) for j in jobs]:
            A, B = self._pair(ea, a0, eb, b0)   # a job = one run of anchors of one structure pair
            assert len(set(ea.struct[a0:a0 + n])) == 1 and len(set(eb.struct[b0:b0 + n])) == 1
            an = np.stack([ea.prim[a0:a0 + n], eb.prim[b0:b0 + n]], axis=1).astype(np.uint32)
            uniq, inv = np.unique(an, axis=0, return_inverse=True)   # repeated anchors: scored once
            try:
                s = oracle.from_primitives(self.p, ea.st.xyz[A], ea.st.cat[A], ea.st.tag[A], eb.st.xyz[B],
                                           eb.st.cat[B], eb.st.tag[B], uniq, ea.thr)
            except oracle.OracleError as e:
                raise _capi.LocoHDError(e.status, str(e))
            all_scores.append(s[inv.ravel()])
        res = {}
        if scores:
            res["scores"] = np.concatenate(all_scores)
        if job_means:
            res["job_means"] = np.array([s.mean() for s in all_scores])
        if anchor_means:
            res["anchor_means"] = np.mean(all_scores, axis=0)
        if anchor_stds:
            res["anchor_stds"] = np.std(all_scores, axis=0)
        return res


class _MonkeyPatch:
    def setenv(self, k, v):
        pass

    def delenv(self, k, raising=True):
        pass


if __name__ == "__main__":
    import test_gpu_tile_kernel as tk
    import test_highprec as hp

    ctx = OracleCtx()
    only = sys.argv[1:]
    if not only:
        tk.test_sliced_unit_order_scores_the_same_units(ctx, oracle, _MonkeyPatch())
        print("ok  test_gpu_tile_kernel.py::test_sliced_unit_order_scores_the_same_units (test logic only)")
        hp.test_cuda_kernels_against_exact_values_at_the_ensemble_shape(ctx)
        print("ok  test_highprec.py::test_cuda_kernels_against_exact_values_at_the_ensemble_shape (test logic only)")
        hp.test_cuda_path_against_exact_values(ctx)
        hp.test_cuda_batch_path_against_exact_values(ctx)
        print("ok  test_highprec.py::test_cuda_path_against_exact_values / test_cuda_batch_path_against_exact_values (test logic only)")

    import test_gpu_grad as tg
    grad_cases = [(f"test_gradients_match_the_reference[{sd}-{wf}]", tg.test_gradients_match_the_reference, (wf, sd))
                  for wf in sorted(tg.WFS) for sd in sorted(tg.SDS)]
    grad_cases += [(f"test_weight_function_densities[{n}-{p}]",
                    lambda c, o, n, p: tg.test_weight_function_densities(c, n, p), (n, p)) for n, p in tg.DENSITY_WFS]
    grad_cases += [("test_gradients_integer_kumaraswamy", tg.test_gradients_integer_kumaraswamy, ()),
                   ("test_gradients_per_pair_weight_functions", tg.test_gradients_per_pair_weight_functions, ()),
                   ("test_renyi_zero_on_disjoint_compositions", tg.test_renyi_zero_on_disjoint_compositions, ()),
                   ("test_no_pairs_leaves_zero_gradients", tg.test_no_pairs_leaves_zero_gradients, ())]
    grad_cases += [(f"test_directional_derivative_matches_finite_differences[{wf}]",
                    tg.test_directional_derivative_matches_finite_differences, (wf,)) for wf in sorted(tg.WFS)]
    for name, fn, args in grad_cases:
        if only and not any(o in name for o in only):
            continue
        fn(ctx, oracle, *args)
        print(f"ok  test_gpu_grad.py::{name} (test logic only)")

    import test_gpu_tile_matrix as tm
    tm._env_offsets = lambda env: env.offsets()   # the stand-in has no C-ABI handle to dump
    cases = [(f"test_category_counts_across_the_instantiations[C{c}]", tm.test_category_counts_across_the_instantiations, (c,))
             for c in (1, 2, 8, 9, 12, 16)]
    cases += [("test_extra_category_rows_add_exact_zeros", tm.test_extra_category_rows_add_exact_zeros, ()),
              ("test_replicated_tables_copy_entries_only", tm.test_replicated_tables_copy_entries_only, ()),
              ("test_team_counts_and_run_lengths", tm.test_team_counts_and_run_lengths, ())]
    cases += [(f"test_largest_environments[C{c}-{n}]", tm.test_largest_environments, (c, n, e))
              for c, n, e in [(8, 500, {"cp": 8, "rep_n": 0, "teams": 6}), (12, 445, {"cp": 16, "rep_n": 0, "teams": 6}),
                              (8, 506, {"cp": 8, "teams": 5})]]
    cases += [("test_weight_function_keys", tm.test_weight_function_keys, ()),
              ("test_sparse_members", tm.test_sparse_members, ())]
    cases += [(f"test_unknown_category_with_sixteen_rows[{w}]", tm.test_unknown_category_with_sixteen_rows, (w,))
              for w in ("member", "anchor")]
    cases += [("test_random_tile_cases", tm.test_random_tile_cases, ())]
    for name, fn, args in cases:
        if only and not any(o in name for o in only):
            continue
        mp = pytest.MonkeyPatch()   # the stand-in reads LOCOHD_NO_TILES; LOCOHD_TILE_TEAMS reaches the geometry query
        try:
            fn(ctx, oracle, mp, *args)
        finally:
            mp.undo()
        print(f"ok  test_gpu_tile_matrix.py::{name} (test logic only)")
