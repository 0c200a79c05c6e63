"""Single source of truth for the C-ABI of libb200pose.so.

Every entry point declared in include/b200pose.h, instantiated in csrc/*.cu and bound in _C.py is
derived from this table (tools/gen_header.py writes the header; tests/test_abi.py checks that the
built library exports exactly these symbols).

Group layouts follow the reference (pypose/lietensor/lietensor.py:196-198, 354-356, 494-496,
638-640): D = data width of a group element, K = tangent (manifold) width.
"""

GROUPS = {
    # group name: (algebra name, D, K)
    "SO3": ("so3", 4, 3),
    "SE3": ("se3", 7, 6),
    "RxSO3": ("rxso3", 5, 4),
    "Sim3": ("sim3", 8, 7),
}

DTYPES = {"f32": "float", "f64": "double"}

# (op, which name prefixes the symbol, input widths, output widths, reference citation)
# widths: "D" / "K" resolve per group; integers are literal.
LIE_OPS = [
    ("exp_fwd", "alg", [("x", "K")], [("X", "D")],
     "so3_Exp/se3_Exp/rxso3_Exp/sim3_Exp.forward, pypose/lietensor/operation.py:343-357,401-405,448-451,496-500"),
    ("exp_bwd", "alg", [("x", "K"), ("gX", "D")], [("gx", "K")],
     "*_Exp.backward: gX[:K] @ Jl(x), operation.py:365-370,413-418,459-464,508-513"),
    ("log_fwd", "grp", [("X", "D")], [("x", "K")],
     "SO3_Log/SE3_Log/RxSO3_Log/Sim3_Log.forward, operation.py:308-324,377-382,425-428,471-476"),
    ("log_bwd", "grp", [("x", "K"), ("gx", "K")], [("gX", "D")],
     "*_Log.backward: [gx @ Jl^-1(x), 0], operation.py:331-337,389-395,435-441,483-489"),
    ("inv_fwd", "grp", [("X", "D")], [("Y", "D")],
     "*_Inv.forward, operation.py:934-936,956-960,980-984,1004-1008"),
    ("inv_bwd", "grp", [("Y", "D"), ("gY", "D")], [("gX", "D")],
     "*_Inv.backward: [-gY[:K] @ Adj(Y), 0], operation.py:944-949,968-973,992-997,1016-1021"),
    ("mul_fwd", "grp", [("X", "D"), ("Y", "D")], [("Z", "D")],
     "*_Mul.forward, operation.py:833-837,859-862,884-887,909-912"),
    ("mul_bwd", "grp", [("X", "D"), ("gZ", "D")], [("gX", "D"), ("gY", "D")],
     "*_Mul.backward: gX=[gZ[:K],0], gY=[gZ[:K] @ Adj(X),0], operation.py:845-852,870-877,895-902,920-927"),
    ("act_fwd", "grp", [("X", "D"), ("p", 3)], [("out", 3)],
     "*_Act.forward, operation.py:520-525,549-551,575-577,601-603"),
    ("act_bwd", "grp", [("X", "D"), ("out", 3), ("g", 3)], [("gX", "D"), ("gp", 3)],
     "*_Act.backward, operation.py:534-542,560-568,586-594,612-620"),
    ("act4_fwd", "grp", [("X", "D"), ("p", 4)], [("out", 4)],
     "*_Act4.forward, operation.py:627-629,652-655,678-680,703-706"),
    ("act4_bwd", "grp", [("X", "D"), ("out", 4), ("g", 4)], [("gX", "D"), ("gp", 4)],
     "*_Act4.backward, operation.py:638-646,664-672,689-697,715-722"),
    ("adj_fwd", "grp", [("X", "D"), ("a", "K")], [("out", "K")],
     "*_AdjXa.forward: Adj(X) a, operation.py:729-732,755-758,781-784,807-810"),
    ("adj_bwd", "grp", [("X", "D"), ("out", "K"), ("g", "K")], [("gX", "D"), ("ga", "K")],
     "*_AdjXa.backward: gX=[-g @ ad(out),0], ga=g @ Adj(X), operation.py:742-748,768-774,794-800,820-826"),
    ("adjt_fwd", "grp", [("X", "D"), ("a", "K")], [("out", "K")],
     "*_AdjTXa.forward: Adj(X^-1) a, operation.py:1028-1030,1051-1053,1074-1076,1097-1099"),
    ("adjt_bwd", "grp", [("X", "D"), ("a", "K"), ("g", "K")], [("gX", "D"), ("ga", "K")],
     "*_AdjTXa.backward: ga=Adj(X) g, gX=[-a @ ad(ga),0], operation.py:1038-1044,1061-1067,1084-1090,1107-1113"),
    ("jinvp_fwd", "grp", [("X", "D"), ("p", "K")], [("out", "K")],
     "LieType.Jinvp: Jl^-1(Log X) p, pypose/lietensor/lietensor.py:257-264,422-429,556-563,700-707"),
]

# ops that exist for one group only
EXTRA_OPS = [
    ("b200_so3_jr", [("x", 3)], [("J", 9)],
     "so3Type.Jr, pypose/lietensor/lietensor.py:343-351"),
]


def width(w, D, K):
    return D if w == "D" else K if w == "K" else int(w)


def lie_symbols():
    """Yield (symbol, ctype, ins[(name,width)], outs[(name,width)], citation) for every Lie-op entry point."""
    for grp, (alg, D, K) in GROUPS.items():
        for op, which, ins, outs, cite in LIE_OPS:
            prefix = alg if which == "alg" else grp
            for sfx, ct in DTYPES.items():
                yield (f"b200_{prefix}_{op}_{sfx}", ct,
                       [(n, width(w, D, K)) for n, w in ins],
                       [(n, width(w, D, K)) for n, w in outs], cite)
    for base, ins, outs, cite in EXTRA_OPS:
        for sfx, ct in DTYPES.items():
            yield (f"{base}_{sfx}", ct, list(ins), list(outs), cite)


# ----------------------------------------------------------------------------------------------
# LM inner-loop entry points (csrc/lm.cu).  (symbol base, [(ctype, name, comment)], citation); every base
# exists as _f32 and _f64 (REAL is substituted); `ws` is the fp64 reduction workspace.
# ----------------------------------------------------------------------------------------------
LM_OPS = [
    ("b200_lm_poseinv_loss",
     [("const REAL*", "P", "(n,7) SE3 parameters"), ("const REAL*", "X", "(n,7) SE3 inputs"),
      ("double*", "ws", "workspace; ws[0] = sum rho(|Log(P X)|^2)"), ("int", "robust", "0 none, 1 Huber, 2 PseudoHuber, 3 Cauchy, 4 SoftLOne, 5 Arctan, 6 Scale (optim/kernel.py) with FastTriggs scaling"), ("double", "delta", "kernel parameter")],
     "RobustModel.loss of the README InvNet model, pypose/optim/optimizer.py:118-125 + README.md:120-129"),
    ("b200_lm_poseinv_trial",
     [("const REAL*", "P", "(n,7)"), ("const REAL*", "X", "(n,7)"), ("REAL*", "P_trial", "(n,7) Exp(D) P"),
      ("double*", "ws", "ws[0..3] = loss, trial loss, (JD)^T(2R+JD), failed pivots"),
      ("double", "scale", "prod(1+damping) over trials"), ("double", "dmin", "diag clamp min"),
      ("double", "dmax", "diag clamp max"), ("int", "robust", "0 none, 1 Huber, 2 PseudoHuber, 3 Cauchy, 4 SoftLOne, 5 Arctan, 6 Scale (optim/kernel.py) with FastTriggs scaling"), ("double", "delta", "kernel parameter")],
     "one LevenbergMarquardt trial: modjac + J^T J + clamp/damp + Cholesky + update + loss, "
     "pypose/optim/optimizer.py:645-673, optim/solver.py:213-216, lietensor/lietensor.py:442-444"),
    ("b200_lm_reproj_accum",
     [("const REAL*", "poses", "(ncam,7)"), ("const REAL*", "pts", "(m,3) sorted by camera"),
      ("const REAL*", "pix", "(m,2)"), ("const int*", "seg", "(ncam+1) row offsets per camera"),
      ("REAL*", "H", "(ncam,21) upper triangles of J^T J"), ("REAL*", "g", "(ncam,6) J^T r"),
      ("double*", "ws", "ws[0] = sum rho(|r|^2)"), ("int", "robust", "0 none, 1 Huber, 2 PseudoHuber, 3 Cauchy, 4 SoftLOne, 5 Arctan, 6 Scale (optim/kernel.py) with FastTriggs scaling"), ("double", "delta", "kernel parameter")],
     "J^T J / J^T R assembly of optimizer.py:655-656 for r = pi(T p) - z (README.md:170-178)"),
    ("b200_lm_solve6_retract",
     [("const REAL*", "H", "(n,21)"), ("const REAL*", "g", "(n,6)"), ("const REAL*", "P", "(n,7)"),
      ("REAL*", "P_trial", "(n,7)"), ("REAL*", "D", "(n,6) step, may be NULL"),
      ("double*", "ws", "ws[0..1] = predicted, failed pivots"), ("double", "scale", ""), ("double", "dmin", ""),
      ("double", "dmax", "")],
     "diag clamp (optimizer.py:657) + damping (:666) + Cholesky solve (solver.py:213-216) + p.add_ (:139-140)"),
    ("b200_lm_reproj_loss",
     [("const REAL*", "poses", "(ncam,7)"), ("const REAL*", "pts", "(m,3)"), ("const REAL*", "pix", "(m,2)"),
      ("const int*", "seg", "(ncam+1) row offsets per camera"), ("double*", "ws", "ws[0] = sum rho(|r|^2)"), ("int", "robust", "0 none, 1 Huber, 2 PseudoHuber, 3 Cauchy, 4 SoftLOne, 5 Arctan, 6 Scale (optim/kernel.py) with FastTriggs scaling"), ("double", "delta", "kernel parameter")],
     "model.loss after the update, optimizer.py:673"),
    ("b200_lm_pgo_linearize",
     [("const REAL*", "nodes", "(N,7) SE3 parameters"), ("const REAL*", "Z", "(E,7) relative-pose measurements"),
      ("const int*", "ei", "(E) first node of each edge"), ("const int*", "ej", "(E) second node"),
      ("REAL*", "M", "(E,21) upper triangle of J^T J per edge"), ("REAL*", "u", "(E,6) J^T r per edge"),
      ("double*", "ws", "ws[0] = sum rho(|r|^2)"), ("int", "robust", "see b200_lm_reproj_accum"), ("double", "delta", "")],
     "modjac + J^T J of optimizer.py:645-656 for r = Log(Z^-1 A^-1 B) (examples/module/pgo/pgo.py:15-25); the sparse "
     "counterpart is bae.autograd.graph.jacobian + J.mT @ J, optimizer.py:637-642"),
    ("b200_lm_pgo_linearize_w",
     [("const REAL*", "nodes", "(N,7)"), ("const REAL*", "Z", "(E,7)"), ("const int*", "ei", "(E)"), ("const int*", "ej", "(E)"),
      ("const REAL*", "W", "(E,36) or (1,36) symmetric information matrices, row-major"),
      ("long long", "w_stride", "36 per-edge, 0 one matrix for all edges"),
      ("REAL*", "M", "(E,21) upper triangle of J^T W J"), ("REAL*", "u", "(E,6) J^T W r"),
      ("REAL*", "M0", "(E,21) upper triangle of J^T J"), ("REAL*", "u0", "(E,6) J^T r"),
      ("double*", "ws", "ws[0] = sum rho(|r|^2)"), ("int", "robust", "see b200_lm_reproj_accum"), ("double", "delta", "")],
     "J^T W J / J^T W R with `weight` (optimizer.py:654-656, normalize_RWJ :80-95; examples/module/pgo/pgo.py:75 infos); the "
     "unweighted blocks feed the step quality (strategy.py:143)"),
    ("b200_lm_pgo_scatter",
     [("const REAL*", "M", "(E,21)"), ("const REAL*", "u", "(E,6)"), ("const int*", "ei", "(E)"), ("const int*", "ej", "(E)"),
      ("REAL*", "Hd", "(N,21) diagonal blocks, accumulated with atomics (zero-initialised by the caller)"),
      ("REAL*", "g", "(N,6) J^T R, accumulated")],
     "diagonal of A = J^T J (optimizer.py:642-643 diagonal_op_) and b = J^T R (optimizer.py:668)"),
    ("b200_lm_pgo_spmv",
     [("const REAL*", "M", "(E,21)"), ("const int*", "ei", "(E)"), ("const int*", "ej", "(E)"), ("const REAL*", "x", "(N,6)"),
      ("REAL*", "y", "(N,6) y += H x (atomics)")],
     "A @ p inside the (P)CG loop, optim/solver.py:319-336 (bae PCG: solver.py:343-363)"),
    ("b200_lm_pgo_loss",
     [("const REAL*", "nodes", "(N,7)"), ("const REAL*", "Z", "(E,7)"), ("const int*", "ei", "(E)"), ("const int*", "ej", "(E)"),
      ("double*", "ws", "ws[0] = sum rho(|r|^2)"), ("int", "robust", ""), ("double", "delta", "")],
     "model.loss after the update, optimizer.py:673"),
    ("b200_lm_ba_linearize",
     [("const REAL*", "poses", "(C,7)"), ("const REAL*", "points", "(P,3)"), ("const REAL*", "pix", "(m,2)"),
      ("const int*", "cidx", "(m)"), ("const int*", "pidx", "(m)"), ("REAL*", "Jc", "(m,12) rows of d r/d pose"),
      ("REAL*", "Jp", "(m,6) rows of d r/d point"), ("REAL*", "rs", "(m,2) (scaled) residual"),
      ("REAL*", "Hcc", "(C,21) accumulated (zero-initialised by the caller)"), ("REAL*", "Hpp", "(P,6) accumulated"),
      ("REAL*", "gc", "(C,6) accumulated"), ("REAL*", "gp", "(P,3) accumulated"), ("double*", "ws", "ws[0] = sum rho"),
      ("int", "robust", ""), ("double", "delta", "")],
     "modjac + J^T J for the two-parameter reprojection model, README.md:163-198; sparse counterpart "
     "bae.autograd.graph.jacobian, optimizer.py:637-642"),
    ("b200_lm_ba_wtx",
     [("const REAL*", "Jc", "(m,12)"), ("const REAL*", "Jp", "(m,6)"), ("const int*", "cidx", "(m)"), ("const int*", "pidx", "(m)"),
      ("const REAL*", "x", "(C,6)"), ("REAL*", "t", "(P,3) t += W^T x (atomics)")],
     "off-diagonal block product inside A @ p of the (P)CG loop, optim/solver.py:319-336"),
    ("b200_lm_ba_wv",
     [("const REAL*", "Jc", "(m,12)"), ("const REAL*", "Jp", "(m,6)"), ("const int*", "cidx", "(m)"), ("const int*", "pidx", "(m)"),
      ("const REAL*", "v", "(P,3)"), ("REAL*", "y", "(C,6) y += W v (atomics)")],
     "off-diagonal block product inside A @ p of the (P)CG loop, optim/solver.py:319-336"),
    ("b200_lm_ba_loss",
     [("const REAL*", "poses", "(C,7)"), ("const REAL*", "points", "(P,3)"), ("const REAL*", "pix", "(m,2)"),
      ("const int*", "cidx", "(m)"), ("const int*", "pidx", "(m)"), ("double*", "ws", "ws[0] = sum rho(|r|^2)"),
      ("int", "robust", ""), ("double", "delta", "")],
     "model.loss after the update, optimizer.py:673"),
    ("b200_lm_reproj_residual",
     [("const REAL*", "poses", "(ncam,7)"), ("const REAL*", "pts", "(m,3)"), ("const REAL*", "pix", "(m,2)"),
      ("const int*", "cidx", "(m)"), ("REAL*", "r", "(m,2)")],
     "model.forward of the reprojection model, README.md:170-178"),
    ("b200_lm_blk6_damp_inv",
     [("const REAL*", "H", "(n,21) packed upper triangles of symmetric 6x6 blocks"), ("double", "scale", "prod(1+damping)"),
      ("double", "dmin", "diag clamp min"), ("double", "dmax", "diag clamp max"),
      ("REAL*", "Hd", "(n,21) block with diag <- clamp(diag)*scale, or NULL"),
      ("REAL*", "extra", "(n,6) amount added to the diagonal, or NULL"),
      ("REAL*", "Minv", "(n,21) inverse of the damped block (block-Jacobi preconditioner), or NULL")],
     "A.diagonal().clamp_ + cumulative damping, optimizer.py:657/666; block-Jacobi preconditioner of the PCG, solver.py:276-340"),
    ("b200_lm_pt3_damp_inv",
     [("const REAL*", "H", "(P,6) packed symmetric 3x3 point blocks"), ("double", "scale", ""), ("double", "dmin", ""),
      ("double", "dmax", ""), ("REAL*", "Hinv", "(P,6) inverse of the clamped + damped block")],
     "point-block elimination of the Schur complement (the reference solves the full sparse system, optimizer.py:637-643)"),
    ("b200_lm_pt3_apply",
     [("const REAL*", "A6", "(P,6) packed symmetric 3x3"), ("const REAL*", "t", "(P,3)"), ("double", "alpha", ""),
      ("REAL*", "out", "(P,3) alpha * A t")],
     "back-substitution dp = Hpp^-1 (-gp - W^T dc)"),
    ("b200_lm_pgo_pcg",
     [("const REAL*", "M", "(E,21) per-edge J^T J"), ("const int*", "ei", "(E)"), ("const int*", "ej", "(E)"),
      ("long long", "E", "edges"), ("const REAL*", "Minv", "(n,21) preconditioner blocks"),
      ("const REAL*", "extra", "(n,6) clamp/damping added to diag H"), ("const REAL*", "g", "(n,6) J^T R; solves (H+extra) x = -g"),
      ("REAL*", "x", "(n,6) solution"), ("REAL*", "r", "(n,6) work"), ("REAL*", "z", "(n,6) work"), ("REAL*", "p", "(n,6) work"),
      ("REAL*", "q", "(n,6) work"), ("REAL*", "xbest", "(n,6) copy of the iterate with the smallest |r| so far"),
      ("double*", "cg", "(16) state: rz[2], p.Ap, |r|^2, stop^2, done (1 converged, 2 breakdown, 3 stagnated, 4 maxiter), "
                        "iterations, maxiter, best |r|^2, iterations since best, save flag, patience"),
      ("double*", "ws", "reduction workspace"), ("double", "tol", "stop when |r| <= tol |b|"),
      ("long long", "maxiter", ""), ("long long", "first_iter", "0 initialises the state; otherwise continue"),
      ("long long", "iters", "iterations to enqueue (no-ops once the done flag is set)"),
      ("const unsigned long long*", "bases", "HOST (world) exchange buffers (b200_comm_open) or NULL: single GPU"),
      ("int", "rank", ""), ("int", "world", ""), ("long long", "stage", "payload byte offset of the all-reduce staging area"),
      ("long long", "result", "payload byte offset of the all-reduce result area"),
      ("long long", "epoch", "all-reduce epochs consumed so far on the PCG channel"), ("unsigned*", "tickets", "(2) zeroed")],
     "PCG.forward loop, optim/solver.py:312-340, with M = block-Jacobi; enqueues `iters` iterations without a host sync"),
    ("b200_lm_cg_finish",
     [("REAL*", "x", "(n,6) in: last iterate; out: the returned solution"), ("const REAL*", "xbest", "(n,6)"),
      ("const double*", "cg", "(16) state of the finished solve")],
     "end of CG.forward (solver.py:338-340 `return x`): the last iterate if the solve converged, otherwise the iterate "
     "with the smallest residual (finite-precision guard, DESIGN.md)"),
    ("b200_lm_pgo_predicted",
     [("const REAL*", "M", "(E,21)"), ("const int*", "ei", "(E)"), ("const int*", "ej", "(E)"), ("long long", "E", ""),
      ("const REAL*", "D", "(n,6) step"), ("const REAL*", "g", "(n,6) J^T R"), ("double*", "ws", "ws[0] = D^T H D + 2 D^T g")],
     "TrustRegion 'predicted' reduction (J D)^T (2 R + J D), optim/strategy.py:143"),
    ("b200_lm_pgo_predicted_edge",
     [("const REAL*", "M0", "(E,21)"), ("const REAL*", "u0", "(E,6)"), ("const int*", "ei", "(E)"), ("const int*", "ej", "(E)"),
      ("const REAL*", "D", "(N,6) step"), ("double*", "ws", "ws[0] = sum_e d^T M0 d + 2 d^T u0, d = D_j - D_i")],
     "TrustRegion 'predicted' reduction from per-edge blocks, optim/strategy.py:143"),
    ("b200_lm_ba_wtx_gather",
     [("const REAL*", "Y4p", "(m,4) Y4 reordered so that each point's observations are contiguous"),
      ("const REAL*", "poses", "(C,7)"), ("const int*", "cidx_p", "(m) camera index in the same order"),
      ("const int*", "pptr", "(P+1) offsets per point"),
      ("const REAL*", "Hpinv", "(P,6)"), ("const REAL*", "x", "(C,6)"), ("const REAL*", "t0", "(P,3) or NULL"),
      ("double", "alpha", ""), ("REAL*", "u", "(P,3) alpha * Hpp^-1 (t0 + W^T x), no atomics")],
     "W^T x of the Schur PCG by gather + the point-block solve; with t0 = gp, alpha = -1 the back-substitution "
     "dp = Hpp^-1 (-gp - W^T dc)"),
    ("b200_lm_ba_pcg",
     [("const REAL*", "Y4", "(m,4)"), ("const REAL*", "poses", "(C,7)"), ("const int*", "pidx", "(m) camera-sorted"),
      ("const int*", "cseg", "(C+1) row offsets per camera"), ("long long", "split", "work items per camera"),
      ("long long", "tpi", "threads per work item: 32 or 128"),
      ("long long", "m", "observations"), ("const REAL*", "Y4p", "(m,4) point-ordered copy of Y4"),
      ("const int*", "cidx_p", "(m) point-ordered camera indices"), ("const int*", "pptr", "(P+1)"), ("const REAL*", "Hc", "(C,21) damped camera blocks"), ("const REAL*", "Hpinv", "(P,6)"),
      ("const REAL*", "Minv", "(C,21) preconditioner blocks"), ("const REAL*", "bneg", "(C,6) minus the right-hand side"),
      ("REAL*", "x", "(C,6) solution"), ("REAL*", "r", "(C,6)"), ("REAL*", "z", "(C,6)"), ("REAL*", "p", "(C,6)"), ("REAL*", "q", "(C,6)"),
      ("REAL*", "t", "(P,3) work"), ("REAL*", "part", "(C*split,6) partial sums, unused when split == 1"),
      ("REAL*", "xbest", "(C,6)"), ("double*", "cg", "(16) state, see b200_lm_pgo_pcg"), ("double*", "ws", "reduction workspace"),
      ("double", "tol", ""), ("long long", "maxiter", ""), ("long long", "P", "points"), ("long long", "first_iter", ""),
      ("long long", "iters", ""),
      ("const unsigned long long*", "bases", "HOST (world) exchange buffers (b200_comm_open) or NULL: single GPU"),
      ("int", "rank", ""), ("int", "world", ""), ("long long", "stage", "payload byte offset of the all-reduce staging area"),
      ("long long", "result", "payload byte offset of the all-reduce result area"),
      ("long long", "epoch", "all-reduce epochs consumed so far on the PCG channel"), ("unsigned*", "tickets", "(2) zeroed")],
     "PCG on the Schur complement (Hcc - W Hpp^-1 W^T) dc = rhs; optim/solver.py:312-340; no atomics (ba.cu)"),
    ("b200_lm_ba_linearize_seg",
     [("const REAL*", "poses", "(C,7)"), ("const REAL*", "points", "(P,3)"), ("const REAL*", "pix", "(m,2) camera-sorted"),
      ("const int*", "pidx", "(m) camera-sorted"), ("const int*", "cseg", "(C+1) row offsets per camera"),
      ("long long", "split", "work items per camera"), ("long long", "tpi", "threads per work item: 32 or 128"),
      ("REAL*", "Y4", "(m,4) y = T p and sqrt(rho')"), ("const int*", "ppos", "(m) position in point order, or NULL"),
      ("REAL*", "Y4p", "(m,4) point-ordered copy, or NULL"), ("REAL*", "rs", "(m,2) (scaled) residual"),
      ("REAL*", "Hcc", "(C,21) written"), ("REAL*", "gc", "(C,6) written"), ("REAL*", "part", "(C*split,27) or NULL when split == 1"),
      ("double*", "ws", "ws[0] = sum rho"), ("int", "robust", ""), ("double", "delta", "")],
     "modjac + J^T J camera blocks for the two-parameter reprojection model (README.md:163-198; optimizer.py:645-656) with "
     "one writer per camera and a fixed summation order: bit-reproducible"),
    ("b200_lm_ba_point_blocks",
     [("const REAL*", "Y4p", "(m,4) point-ordered"), ("const REAL*", "pix_p", "(m,2) point-ordered pixels"),
      ("const REAL*", "poses", "(C,7)"), ("const int*", "cidx_p", "(m)"), ("const int*", "pptr", "(P+1)"),
      ("REAL*", "Hpp", "(P,6) written"), ("REAL*", "gp", "(P,3) written")],
     "J^T J / J^T R point blocks of the same model by gather (no atomics)"),
    ("b200_lm_ba_wv_seg",
     [("const REAL*", "Y4", "(m,4)"), ("const REAL*", "poses", "(C,7)"), ("const int*", "pidx", "(m)"), ("const int*", "cseg", "(C+1)"),
      ("long long", "split", ""), ("long long", "tpi", ""), ("const REAL*", "Hpinv", "(P,6) or NULL if t holds Hpp^-1 t"),
      ("const REAL*", "t", "(P,3)"), ("REAL*", "y", "(C,6) y -= W Hpp^-1 t, one writer per camera"),
      ("REAL*", "part", "(C*split,6) or NULL when split == 1")],
     "off-diagonal product of the reduced camera system, optim/solver.py:319-336, deterministic"),
    ("b200_lm_ba_schur_diag_seg",
     [("const REAL*", "Y4", "(m,4)"), ("const REAL*", "poses", "(C,7)"), ("const int*", "pidx", "(m)"), ("const int*", "cseg", "(C+1)"),
      ("long long", "split", ""), ("long long", "tpi", ""), ("const REAL*", "Hpinv", "(P,6)"),
      ("REAL*", "Sd", "(C,21) in: damped Hcc; out: minus sum_k W_k Hpp^-1 W_k^T, one writer per camera"),
      ("REAL*", "part", "(C*split,21) or NULL when split == 1")],
     "diagonal blocks of the reduced camera system (preconditioner of the Schur PCG), deterministic"),
    ("b200_lm_ba_predicted",
     [("const REAL*", "Y4", "(m,4)"), ("const REAL*", "poses", "(C,7)"), ("const REAL*", "rs", "(m,2)"), ("const int*", "cidx", "(m)"),
      ("const int*", "pidx", "(m)"), ("const REAL*", "xc", "(C,6)"), ("const REAL*", "xp", "(P,3)"),
      ("double*", "ws", "ws[0] = sum (J d)^T (2 r + J d)")],
     "TrustRegion 'predicted' reduction, optim/strategy.py:143"),
]


LM_OPS += [
    ("b200_lm_pgo_linearize_n",
     [("const REAL*", "nodes", "(N,7)"), ("const REAL*", "Z", "(E,7)"), ("const int*", "ei", "(E)"), ("const int*", "ej", "(E)"),
      ("const int*", "epos_i", "(E) slot of the edge in its first node's list"),
      ("const int*", "epos_j", "(E) slot in its second node's list"),
      ("REAL*", "Mn", "(2E,24) node-ordered blocks: upper triangle of J^T J (21) + 3 pad, written at both slots"),
      ("REAL*", "un", "(2E,6) -J^T r at the first node's slot, +J^T r at the second's"),
      ("double*", "ws", "ws[0] = sum rho(|r|^2)"), ("int", "robust", ""), ("double", "delta", "")],
     "b200_lm_pgo_linearize writing its blocks directly in node order (no atomics downstream); optimizer.py:645-656"),
    ("b200_lm_reproj2_accum_n",
     [("const REAL*", "nodes", "(N,7)"), ("const REAL*", "pts", "(m,3)"), ("const REAL*", "pix", "(m,2)"), ("const int*", "pseg", "(E+1)"),
      ("const int*", "pa", "(E)"), ("const int*", "pb", "(E)"), ("const double*", "intr", "HOST (5)"),
      ("const int*", "epos_i", "(E) slot of the pair in pose b's list"), ("const int*", "epos_j", "(E) slot in pose a's list"),
      ("REAL*", "Mn", "(2E,24)"), ("REAL*", "un", "(2E,6)"), ("double*", "ws", ""), ("int", "robust", ""), ("double", "delta", "")],
     "b200_lm_reproj2_accum writing its blocks directly in node order"),
    ("b200_lm_pgo2_node_sums",
     [("const REAL*", "Mn", "(2E,24)"), ("const REAL*", "un", "(2E,6)"), ("const int*", "nptr", "(N+1) offsets per node"),
      ("REAL*", "Hd", "(N,21) diagonal blocks of J^T J"), ("REAL*", "g", "(N,6) J^T R")],
     "diagonal of A = J^T J (optimizer.py:642-643) and b = J^T R (optimizer.py:668) by gather: one writer per node"),
    ("b200_lm_pgo2_pcg",
     [("const REAL*", "Mn", "(2E,24) node-ordered blocks"), ("const int*", "nother", "(2E) opposite node of each slot"),
      ("const int*", "nptr", "(n+1)"), ("const REAL*", "Minv", "(n,21) block-Jacobi preconditioner"),
      ("const REAL*", "extra", "(n,6) clamp / damping added to diag H"), ("const REAL*", "g", "(n,6); solves (H+extra) x = -g"),
      ("REAL*", "x", "(n,6)"), ("REAL*", "r", "(n,6)"), ("REAL*", "z", "(n,6)"), ("REAL*", "p0", "(n,6) direction, even iterations"),
      ("REAL*", "p1", "(n,6) direction, odd iterations"), ("REAL*", "q", "(n,6)"), ("REAL*", "xbest", "(n,6)"),
      ("double*", "cg", "(16) state, see b200_lm_pgo_pcg"), ("double*", "ws", ""), ("double", "tol", ""),
      ("long long", "maxiter", ""), ("long long", "first_iter", ""), ("long long", "iters", "")],
     "PCG.forward loop, optim/solver.py:312-340, two launches per iteration: direction update + (H + D) p + p.Ap by gather, "
     "then the vector update with its reductions; no atomics, bit-reproducible"),
    ("b200_lm_pgo2_predicted",
     [("const REAL*", "Mn", "(2E,24)"), ("const int*", "nother", "(2E)"), ("const int*", "nptr", "(n+1)"), ("const REAL*", "x", "(n,6) step"),
      ("const REAL*", "g", "(n,6)"), ("double*", "ws", "ws[0] = x^T H x + 2 x^T g")],
     "TrustRegion 'predicted' reduction (J D)^T (2 R + J D), optim/strategy.py:143, by gather"),
    ("b200_lm_reproj2_accum",
     [("const REAL*", "nodes", "(N,7) SE3 poses"), ("const REAL*", "pts", "(m,3) points in the frame of pose a, rows sorted by pair"),
      ("const REAL*", "pix", "(m,2)"), ("const int*", "pseg", "(E+1) row offsets per ordered pose pair"),
      ("const int*", "pa", "(E) pose a of each pair"), ("const int*", "pb", "(E) pose b of each pair"),
      ("const double*", "intr", "HOST (5): fx, skew, cx, fy, cy of proj(y); README `project` is -1, 0, 0, -1, 0"),
      ("REAL*", "M", "(E,21) sum over the pair's rows of J^T J, J = d r / d xi_a = -d r / d xi_b"),
      ("REAL*", "u", "(E,6) sum of J^T r"), ("double*", "ws", "ws[0] = sum rho(|r|^2)"), ("int", "robust", ""), ("double", "delta", "")],
     "modjac + J^T J of optimizer.py:645-656 for r = proj(T_b^-1 T_a p) - z (README.md:170-178 project; "
     "function/geometry.py:60-112,171-225 point2pixel / reprojerr; examples/module/reprojpgo/reprojpgo.py:16-28): the pairs "
     "are the edges of the block-sparse system (b200_lm_pgo_pcg with ei = pb, ej = pa)"),
    ("b200_lm_reproj2_loss",
     [("const REAL*", "nodes", "(N,7)"), ("const REAL*", "pts", "(m,3)"), ("const REAL*", "pix", "(m,2)"), ("const int*", "pseg", "(E+1)"),
      ("const int*", "pa", "(E)"), ("const int*", "pb", "(E)"), ("const double*", "intr", "HOST (5)"),
      ("double*", "ws", "ws[0] = sum rho(|r|^2)"), ("int", "robust", ""), ("double", "delta", "")],
     "model.loss after the update, optimizer.py:673, for the two-pose reprojection model"),
    ("b200_lm_reproj2_residual",
     [("const REAL*", "nodes", "(N,7)"), ("const REAL*", "pts", "(m,3)"), ("const REAL*", "pix", "(m,2)"),
      ("const int*", "ia", "(m) pose a per row"), ("const int*", "ib", "(m) pose b per row"),
      ("const double*", "intr", "HOST (5)"), ("REAL*", "r", "(m,2)")],
     "model.forward of the two-pose reprojection model"),
    ("b200_lm_reproj_step",
     [("REAL*", "poses", "(ncam,7) parameters; overwritten with the trial poses when the trial is accepted"),
      ("const REAL*", "pts", "(m,3) camera-sorted"), ("const REAL*", "pix", "(m,2)"), ("const int*", "seg", "(ncam+1)"),
      ("REAL*", "H", "(ncam,21) J^T J blocks: written by a first trial, read by a retry"), ("REAL*", "g", "(ncam,6)"),
      ("REAL*", "P_trial", "(ncam,7) work"), ("double*", "ws0", "reduction workspace of the solve kernel"),
      ("double*", "ws1", "reduction workspace of the loss kernel"),
      ("double*", "st", "(16) device state: status (0 rejected, 1 accepted, 2 solver failed), loss, last, damping, radius, down, "
                        "reject count, current loss, trial loss, predicted, failed pivots"),
      ("double*", "host_out", "(16) PINNED host memory: the deciding thread stores the state there (zero-copy) and the call "
                              "returns when it has arrived; NULL: nothing is waited for"),
      ("long long", "seq", "a number different from the previous call's; appears in host_out[15] when the state is complete"),
      ("const double*", "ctl", "HOST (14): last, cached, damping, pg down, reject count, reject limit, strategy kind "
                               "(0 Constant, 1 Adaptive, 2 TrustRegion), high, low, up, strategy down, factor, min, max"),
      ("int", "robust", "see b200_lm_reproj_accum"), ("double", "delta", ""), ("double", "scale", "prod(1+damping) so far"),
      ("double", "dmin", ""), ("double", "dmax", ""), ("int", "retry", "0: linearise + solve; 1: solve the stored blocks again"),
      ("long long", "rows", "total number of observation rows (selects 8 or 32 lanes per camera)")],
     "one trial of LevenbergMarquardt.step incl. strategy.update and the accept test, optimizer.py:659-680, "
     "strategy.py:41-46,134-151,248-274, for the single-pose reprojection model"),
    ("b200_lm_reproj_step_peer",
     [("REAL*", "poses", "(ncam,7) replicated parameters; overwritten when the trial is accepted"),
      ("const REAL*", "pts", "(m_local,3) this rank's observations, camera-sorted"), ("const REAL*", "pix", "(m_local,2)"),
      ("const int*", "seg", "(ncam+1) offsets of this rank's rows per camera"),
      ("REAL*", "H", "(ncam,21): the owner's rows hold the reduced blocks (kept for retries)"), ("REAL*", "g", "(ncam,6)"),
      ("const unsigned long long*", "bases", "HOST (world) exchange buffers, see b200_comm_open"), ("int", "rank", ""), ("int", "world", ""),
      ("long long", "part_off", "payload byte offset (16-byte aligned) of the partial blocks: world * ceil(ncam/world) slots of 28 elements"),
      ("long long", "pt_off", "payload byte offset (16-byte aligned) of the trial poses: ncam slots of 8 elements"),
      ("long long", "epoch0", "count of linearisations so far (incl. this one unless retry)"),
      ("long long", "epoch1", "count of trials so far incl. this one"),
      ("double*", "ws0", "reduction workspace"), ("double*", "ws1", ""), ("double*", "ws2", ""),
      ("double*", "st", "(16) device state, see b200_lm_reproj_step"), ("double*", "host_out", "(16) pinned host memory or NULL"), ("long long", "seq", "see b200_lm_reproj_step"),
      ("const double*", "ctl", "HOST (14), see b200_lm_reproj_step"), ("int", "robust", ""), ("double", "delta", ""),
      ("double", "scale", ""), ("double", "dmin", ""), ("double", "dmax", ""), ("int", "retry", ""),
      ("long long", "rows", "number of LOCAL observation rows (selects 8 or 32 lanes per camera)"),
      ("int", "gather", "0: blocks reduce-scattered to camera owners, trial poses all-gathered (3 exchanges per trial); "
                        "1: every rank receives all partial blocks and solves every camera (2 exchanges; the partial-block "
                        "region then holds world * ncam slots)"),
      ("const unsigned char*", "present", "(world, ncam) 1 where that rank holds rows of that camera, or NULL = every rank "
                                          "holds rows of every camera: a rank sends no block for a camera it has no rows of, "
                                          "and the receivers skip those slots"),
      ("const int*", "cams", "(nloc) the cameras this rank holds rows of, ascending (required with `present`), or NULL = all"),
      ("long long", "nloc", "")],
     "b200_lm_reproj_step with the observations sharded over `world` GPUs: [H | g] is reduce-scattered to camera owners, "
     "trial poses are all-gathered and the scalar sums exchanged by stores into the peers' buffers (SURVEY.md §8e row 4); "
     "optimizer.py:659-680"),
    ("b200_lm_poseinv_step_peer",
     [("REAL*", "P", "(n,7) this rank's poses"), ("const REAL*", "X", "(n,7)"), ("REAL*", "P_trial", "(n,7) work"),
      ("const unsigned long long*", "bases", "HOST (world) exchange buffers"), ("int", "rank", ""), ("int", "world", ""),
      ("long long", "epoch", "count of trials so far incl. this one"), ("double*", "ws", ""), ("double*", "st", "(16)"),
      ("double*", "host_out", "(16) pinned host memory or NULL"), ("long long", "seq", "see b200_lm_reproj_step"), ("const double*", "ctl", "HOST (14)"), ("int", "robust", ""),
      ("double", "delta", ""), ("double", "scale", ""), ("double", "dmin", ""), ("double", "dmax", "")],
     "b200_lm_poseinv_step with the poses sharded over `world` GPUs: only the four scalar sums are exchanged "
     "(SURVEY.md §8e row 3); optimizer.py:659-680"),
    ("b200_lm_poseinv_step",
     [("REAL*", "P", "(n,7) parameters; overwritten when the trial is accepted"), ("const REAL*", "X", "(n,7)"),
      ("REAL*", "P_trial", "(n,7) work"), ("double*", "ws", "reduction workspace"), ("double*", "st", "(16) device state"),
      ("double*", "host_out", "(16) pinned host memory or NULL"), ("long long", "seq", "see b200_lm_reproj_step"), ("const double*", "ctl", "HOST (14), see b200_lm_reproj_step"),
      ("int", "robust", ""), ("double", "delta", ""), ("double", "scale", ""), ("double", "dmin", ""), ("double", "dmax", "")],
     "one trial of LevenbergMarquardt.step for README.md:120-129 InvNet, optimizer.py:659-680"),
]


def lm_symbols():
    """Yield (symbol, [(ctype, name, comment)], citation)."""
    for base, args, cite in LM_OPS:
        for sfx, ct in DTYPES.items():
            yield f"{base}_{sfx}", [(t.replace("REAL", ct), n, c) for t, n, c in args], cite


# ----------------------------------------------------------------------------------------------
# scans (csrc/scan.cu): explicit declarations, (symbol base, args, citation); REAL as above.
# ----------------------------------------------------------------------------------------------
SCAN_OPS = [
    (f"b200_{g}_cumprod",
     [("const REAL*", "in", f"(B,L,{d})"), ("REAL*", "out", f"(B,L,{d})"), ("long long", "B", "sequences"),
      ("long long", "L", "scan length"), ("int", "left", "1: y_i = x_i y_{i-1}; 0: y_i = y_{i-1} x_i")],
     "cumprod / cummul on group LieTensors = cumops_ with the group product, pypose/basics/ops.py:29-58, "
     "lietensor.py:171-193")
    for g, (_, d, _) in GROUPS.items()
] + [
    (f"b200_{g}_cumprod_lb",
     [("const REAL*", "in", f"(B,L,{d})"), ("REAL*", "out", f"(B,L,{d})"), ("long long", "B", "sequences"),
      ("long long", "L", "scan length"), ("int", "left", "1: y_i = x_i y_{i-1}; 0: y_i = y_{i-1} x_i"),
      ("void*", "ws", "b200_scan_workspace_bytes(B, L, sizeof(REAL)) bytes of scratch, 16-byte aligned")],
     "the same scan with the time axis split over CTAs (tile products, scan of the tile products, apply): for few long sequences; "
     "pypose/basics/ops.py:29-58, lietensor.py:171-193")
    for g, (_, d, _) in GROUPS.items()
] + [
    ("b200_imu_integrate",
     [("const REAL*", "dt", "(B,F,1)"), ("const REAL*", "gyro", "(B,F,3)"), ("const REAL*", "acc", "(B,F,3)"),
      ("const REAL*", "rot", "(B,F,4) known rotations or NULL"), ("const REAL*", "init_rot", "(B,4) / (1,4) or NULL"),
      ("long long", "init_stride", "4 for per-sequence init_rot, 0 to broadcast one"),
      ("const REAL*", "gravity3_host", "HOST pointer to the 3 gravity components"),
      ("REAL*", "a", "(B,F,3) or NULL to skip all six integrate outputs"), ("REAL*", "Dp", "(B,F,3)"),
      ("REAL*", "Dv", "(B,F,3)"), ("REAL*", "Dr", "(B,F,4)"), ("REAL*", "Dt", "(B,F,1)"), ("REAL*", "w", "(B,F,4)"),
      ("const REAL*", "init_pos", "(B,3) / (1,3) or NULL"), ("const REAL*", "init_vel", "(B,3) / (1,3) or NULL"),
      ("long long", "pv_stride", "3 per-sequence, 0 broadcast"),
      ("REAL*", "rot_out", "(B,F,4) predicted rotation or NULL to skip the three predict outputs"),
      ("REAL*", "vel_out", "(B,F,3)"), ("REAL*", "pos_out", "(B,F,3)"), ("long long", "B", "trajectories"),
      ("long long", "F", "samples per trajectory")],
     "IMUPreintegrator.integrate + .predict, pypose/module/imu_preintegrator.py:314-384, 386-426"),
    ("b200_imu_cov",
     [("const REAL*", "Rk", "(B,F,4) per-sample rotation increments (w)"), ("const REAL*", "Rij", "(B,F,4) accumulated rotations"),
      ("const REAL*", "a", "(B,F,3) gravity-compensated accelerations"), ("const REAL*", "dt", "(B,F,1)"),
      ("const REAL*", "gyro_cov", "(B,1|F,3) diagonal"), ("const REAL*", "acc_cov", "(B,1|F,3) diagonal"),
      ("long long", "cov_stride_b", "elements between trajectories in gyro/acc_cov"),
      ("long long", "cov_stride_f", "3 if per-sample, 0 if one per trajectory"),
      ("const REAL*", "init_cov", "(B,9,9) / (1,9,9)"), ("long long", "init_stride", "81 or 0"),
      ("REAL*", "cov", "(B,9,9)"), ("REAL*", "work", "B*(3*NC+1)*81 elements, NC = ceil(F/chunk)"),
      ("long long", "chunk", "time steps per chunk"), ("long long", "B", ""), ("long long", "F", "")],
     "IMUPreintegrator.propagate_cov, pypose/module/imu_preintegrator.py:428-465"),
]


def scan_symbols():
    for base, args, cite in SCAN_OPS:
        for sfx, ct in DTYPES.items():
            yield f"{base}_{sfx}", [(t.replace("REAL", ct), n, c) for t, n, c in args], cite


# ----------------------------------------------------------------------------------------------
# k-nearest neighbours and the ICP correspondence step (csrc/knn.cu): (symbol base, args, citation); REAL as above.
# Splits and workspace size come from b200_knn_plan.
# ----------------------------------------------------------------------------------------------
KNN_OPS = [
    ("b200_knn",
     [("const REAL*", "ref", "(B|1, N1, D) queries, row-major"), ("long long", "ref_bstride", "elements between batches, 0: one cloud for all"),
      ("const REAL*", "nbr", "(B|1, N2, D) neighbours"), ("long long", "nbr_bstride", "elements between batches, 0: one cloud for all"),
      ("long long", "B", "batches"), ("long long", "N1", "queries per batch"), ("long long", "N2", "neighbours per batch, < 2^31"),
      ("int", "D", "1..8"), ("int", "k", "1..min(32, N2)"), ("int", "ord", "1, 2, or 0 for inf"),
      ("int", "largest", "1: the k furthest"), ("long long", "splits", "S from b200_knn_plan"),
      ("void*", "ws", "b200_knn_plan bytes of scratch, or NULL when splits == 1"),
      ("REAL*", "values", "(B, N1, k) ord-norm distances, sorted"), ("long long*", "indices", "(B, N1, k) neighbour indices")],
     "knn, pypose/function/geometry.py:228-313 (norm of the broadcast difference + topk), streamed without the "
     "(N1, N2, D) difference tensor; ties keep the lower neighbour index"),
    ("b200_icp_moments",
     [("const REAL*", "src", "(B|1, N1, 3) source points"), ("long long", "src_bstride", "elements between batches, 0: one cloud for all"),
      ("const REAL*", "tgt", "(B|1, N2, 3) target points"), ("long long", "tgt_bstride", "elements between batches, 0: one cloud for all"),
      ("const REAL*", "pose", "(B, 7) current SE3 estimate T applied to src"), ("long long", "B", "batches"),
      ("long long", "N1", "source points"), ("long long", "N2", "target points, 1 .. 2^31 - 1"), ("int", "ord", "1, 2, or 0 for inf"),
      ("long long", "splits", "S from b200_knn_plan with k = 1"), ("void*", "ws", "b200_knn_plan bytes, or NULL when splits == 1"),
      ("double*", "moments", "(B, 17) accumulated (zeroed by the caller): count, sum T s (3), sum t (3), "
                             "sum t (T s)^T row-major (9), sum of nearest-neighbour distances")],
     "one iteration of ICP.forward, pypose/module/icp.py: knn(T source, target, k=1) + gather + the moments of "
     "svdtf (geometry.py:315-358), without materialising the transformed cloud"),
]


# host-side queries of csrc/knn.cu: (symbol, return type, [(ctype, name, comment)], description)
KNN_QUERIES = [
    ("b200_knn_plan", "long long",
     [("long long", "B", "batches"), ("long long", "N1", "queries per batch"), ("long long", "N2", "neighbours per batch"),
      ("int", "k", "results per query"), ("int", "elem_size", "4 or 8"), ("int", "sms", "multiprocessors of the device"),
      ("long long*", "splits", "out: S, the number of N2 chunks (1 = no split)")],
     "Number of N2 splits for a search of B x N1 queries over N2 neighbours, chosen from the shapes; returns the "
     "workspace bytes that split needs (0 when S == 1)"),
]


def knn_symbols():
    for base, args, cite in KNN_OPS:
        for sfx, ct in DTYPES.items():
            yield f"{base}_{sfx}", [(t.replace("REAL", ct), n, c) for t, n, c in args], cite
