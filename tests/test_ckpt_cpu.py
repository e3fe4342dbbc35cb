"""Checkpoint compatibility with the reference (src/ckpt.cc) -- CPU tests, no GPU.

quantum_basis_b200/ckpt.py reads and writes the reference's out_Qckpt/ files.  Both directions are run against the
compiled, unmodified reference (oracle/_ref/qb_ref --lanczos-ckpt: the reference's own lanczos() with enable_ckpt = true):
  * the reference stops after 20 steps -> ckpt.lanczos_load reads its files -> a numpy restatement of the loop continues
    to the reference's own stopping step and E0;
  * the oracle runs 25 steps -> ckpt.lanczos_store writes the files -> the REFERENCE resumes from them and arrives at the
    step count, E0 and coefficients of its uninterrupted run (tests/golden/heis12_full.npz).
The device loop that sits between load and store in production (qbgpu_lanczos_resume_*) is covered by the GPU tests.
"""
import os
import shutil
import tempfile

import numpy as np
import pytest

from quantum_basis_b200 import ckpt

MAXIT = 200
PREC = 2e-12


def _needs_qb_ref(oracle):
    if not oracle.have_qb_ref():
        pytest.skip("oracle/_ref/qb_ref is not built (needs the reference's sources at build time)")


@pytest.fixture(scope="module")
def case(oracle):
    A, meta, ex = oracle.load_golden("heis12_full")
    work = tempfile.mkdtemp(prefix="qb_ckpt_")
    path = os.path.join(work, "A.qbcsr")
    oracle.write_qbcsr(path, A)
    yield A, meta, ex, work, path
    shutil.rmtree(work, ignore_errors=True)


def _numpy_resume(oracle, A, k, v, hess, state, maxit):
    """The reference's loop (src/lanczos.cc:193-264, purpose sr_val0) continued from step k on host arrays."""
    n = A.dim
    cnt, accuracy, t0, t1 = int(state[0]), state[1], state[2], state[3]
    m = k
    col = lambda j: v[(j % 2) * n:(j % 2 + 1) * n]   # noqa: E731
    if cnt > 15 and accuracy < PREC:
        return m
    while m < maxit - 1:
        m += 1
        w = -hess[m - 1] * col(m - 2) + oracle.spmv(A, col(m - 1).copy())
        hess[maxit + m - 1] = np.vdot(col(m - 1), w).real
        w = w - hess[maxit + m - 1] * col(m - 1)
        hess[m] = np.linalg.norm(w)
        col(m)[:] = w / hess[m]
        if abs(hess[m]) < PREC:
            break
        ritz, s = oracle.hess_eigen(hess, maxit, m)
        if m > 3:
            accuracy = abs(hess[m] * s[m - 1, 0])
            cnt = cnt + 1 if abs((ritz[0] - t0) / ritz[0]) < PREC else 0
            if cnt > 15 and accuracy < PREC:
                break
        t0, t1 = ritz[0], ritz[1]
    return m


def test_resume_from_a_checkpoint_written_by_the_reference(oracle, case):
    _needs_qb_ref(oracle)
    A, meta, ex, work, path = case
    n = A.dim
    w = os.path.join(work, "ref_writes")
    r = oracle.run_qb_ref(["file_z", path, "--lanczos-ckpt", "sr_val0", MAXIT, 20], workdir=w)
    assert r["ckpt_steps"] == 20
    d = os.path.join(w, ckpt.DIRNAME)
    k, v, hess, state = ckpt.lanczos_load(d, MAXIT, n, np.complex128, "sr_val0")
    assert k == 20
    assert np.array_equal(hess[MAXIT:MAXIT + 20], np.asarray(r["ckpt_a"])) and np.array_equal(hess[:21], np.asarray(r["ckpt_b"]))
    assert np.abs(hess[MAXIT:MAXIT + 20] - ex["lanczos_a"][:20]).max() < 1e-12
    vk, vk1 = v[(k % 2) * n:(k % 2 + 1) * n], v[((k - 1) % 2) * n:((k - 1) % 2 + 1) * n]
    assert abs(np.linalg.norm(vk) - 1) < 1e-12 and abs(np.linalg.norm(vk1) - 1) < 1e-12 and abs(np.vdot(vk1, vk)) < 1e-10
    # the stop rule's memory (lczs_mlns.dat) against a replay from the coefficients alone
    replay = ckpt.stop_state_from_coefficients(hess, MAXIT, k)
    assert state[0] == replay[0] and abs(state[2] - replay[2]) < 1e-10 and abs(state[3] - replay[3]) < 1e-10
    assert abs(state[1] - replay[1]) <= 1e-6 * abs(replay[1]) + 1e-14
    m = _numpy_resume(oracle, A, k, v, hess, state, MAXIT)
    ritz, _ = oracle.hess_eigen(hess, MAXIT, m)
    assert m == meta["lanczos_steps"]                                  # stops where the uninterrupted reference run stops
    assert abs(ritz[0] - meta["lanczos_E0"]) <= 1e-10 * abs(meta["lanczos_E0"])


def test_the_reference_resumes_from_a_checkpoint_written_here(oracle, case):
    _needs_qb_ref(oracle)
    A, meta, ex, work, path = case
    n = A.dim
    k = 25
    m, a, b, vbuf = oracle.lanczos(A, oracle.vec_randomize(n, 1), maxit=k + 1)     # exactly k steps
    assert m == k
    hess = np.zeros(2 * MAXIT)
    hess[MAXIT:MAXIT + k] = a
    hess[:k + 1] = b
    w = os.path.join(work, "we_write")
    d = os.path.join(w, ckpt.DIRNAME)
    ckpt.lanczos_store(d, k, MAXIT, n, np.asarray(vbuf)[:2 * n], hess, "sr_val0", ckpt.stop_state_from_coefficients(hess, MAXIT, k))
    assert sorted(os.listdir(d)) == ["HessenbergA.dat", "HessenbergB.dat", f"lanczosV{k - 1}.dat", f"lanczosV{k}.dat", "lczs_mlns.dat"]
    r = oracle.run_qb_ref(["file_z", path, "--lanczos-ckpt", "sr_val0", MAXIT, MAXIT - 1], workdir=w)
    assert r["ckpt_steps"] == meta["lanczos_steps"]
    assert abs(r["ckpt_E0"] - meta["lanczos_E0"]) <= 1e-10 * abs(meta["lanczos_E0"])
    assert np.abs(np.asarray(r["ckpt_a"])[:30] - ex["lanczos_a"][:30]).max() < 1e-9
    # and a run the reference finished is recognised as finished: nothing left to do
    k2, v2, h2, st2 = ckpt.lanczos_load(d, MAXIT, n, np.complex128, "sr_val0")
    assert k2 == meta["lanczos_steps"] and st2[0] > 15 and st2[1] < PREC
    assert _numpy_resume(oracle, A, k2, v2, h2, st2, MAXIT) == k2


@pytest.mark.parametrize("every", [1, 7])
@pytest.mark.parametrize("crash", ["new_files", "commit"])
def test_an_interrupted_update_is_rolled_forward_or_rewound(oracle, case, every, crash):
    """Two-phase commit (src/ckpt.cc:37-106): a crash before the commit marker rewinds to the last committed step (one step
    back for the reference's every-step checkpoints, `every` steps back here), a crash after it rolls forward."""
    A, meta, ex, work, path = case
    n = A.dim
    d = tempfile.mkdtemp(prefix="qb_ckpt_crash_")
    try:
        k1, k2 = 12, 12 + every
        states = {}
        for k in (k1, k2):
            m, a, b, vbuf = oracle.lanczos(A, oracle.vec_randomize(n, 1), maxit=k + 1)
            hess = np.zeros(2 * MAXIT); hess[MAXIT:MAXIT + k] = a; hess[:k + 1] = b
            states[k] = (np.asarray(vbuf)[:2 * n].copy(), hess)
        st = lambda k: ckpt.stop_state_from_coefficients(states[k][1], MAXIT, k)   # noqa: E731
        ckpt.lanczos_store(d, k1, MAXIT, n, states[k1][0], states[k1][1], "sr_val0", st(k1))
        with pytest.raises(ckpt._Interrupted):
            ckpt.lanczos_store(d, k2, MAXIT, n, states[k2][0], states[k2][1], "sr_val0", st(k2), _crash_after=crash)
        k, v, hess, state = ckpt.lanczos_load(d, MAXIT, n, np.complex128, "sr_val0")
        want = k2 if crash == "commit" else k1
        assert k == want
        assert np.array_equal(hess, states[want][1])
        for j in (k, k - 1):
            assert np.array_equal(v[(j % 2) * n:(j % 2 + 1) * n], states[want][0][(j % 2) * n:(j % 2 + 1) * n])
        left = sorted(os.listdir(d))
        assert left == sorted(["HessenbergA.dat", "HessenbergB.dat", f"lanczosV{k - 1}.dat", f"lanczosV{k}.dat", "lczs_mlns.dat"])
    finally:
        shutil.rmtree(d, ignore_errors=True)


def test_damaged_files_are_refused(oracle, case):
    A, meta, ex, work, path = case
    n = A.dim
    d = tempfile.mkdtemp(prefix="qb_ckpt_bad_")
    try:
        m, a, b, vbuf = oracle.lanczos(A, oracle.vec_randomize(n, 1), maxit=9)
        hess = np.zeros(2 * MAXIT); hess[MAXIT:MAXIT + 8] = a; hess[:9] = b
        ckpt.lanczos_store(d, 8, MAXIT, n, np.asarray(vbuf)[:2 * n], hess, "sr_val0", [0, 0.0, 0.0, 0.0])
        with open(os.path.join(d, "lanczosV8.dat"), "r+b") as f:
            f.seek(100); f.write(b"\x00\x01\x02\x03")                 # CRC-32 no longer matches
        with pytest.raises(ckpt.QbgpuError):
            ckpt.lanczos_load(d, MAXIT, n, np.complex128, "sr_val0")
        ckpt.lanczos_clean(d)
        assert ckpt.lanczos_load(d, MAXIT, n, np.complex128, "sr_val0")[0] == 0
        assert ckpt.lanczos_load(os.path.join(d, "nowhere"), MAXIT, n, np.complex128, "dnmcs")[0] == 0
    finally:
        shutil.rmtree(d, ignore_errors=True)


# --------------------------------------------------------------------------------------------------- conjugate gradient
def _numpy_cg(oracle, A, E0, m, v, r, p, maxit):
    """eigenvec_CG (src/lanczos.cc:281-341) on host arrays from step m; returns (m, accu)."""
    eps = np.finfo(np.float64).eps
    accu = 0.0 if m == 0 else np.linalg.norm(r)
    while m < maxit:
        if accu < PREC:
            rnorm = np.linalg.norm(v)
            if m == 0 or abs(rnorm - 1.0) > PREC:
                v /= rnorm
                r[:] = E0 * v - oracle.spmv(A, v.copy())
                p[:] = r
                accu = np.linalg.norm(r)
                m += 1
                if accu < PREC:
                    break
            else:
                break
        else:
            pp = (eps - E0) * p + oracle.spmv(A, p.copy())
            alpha = accu * accu / np.vdot(p, pp)
            v += alpha * p
            r -= alpha * pp
            beta = np.linalg.norm(r) / accu
            p[:] = r + beta * beta * p
            accu *= beta
            m += 1
    return m, accu


def test_cg_checkpoints_in_both_directions(oracle, case):
    _needs_qb_ref(oracle)
    A, meta, ex, work, path = case
    n, E0 = A.dim, meta["lanczos_E0"]
    # the reference stops at step 10 -> we load and continue to its own stopping step and vector
    w = os.path.join(work, "cg_ref_writes")
    r = oracle.run_qb_ref(["file_z", path, "--cg-ckpt", repr(E0), 10, os.path.join(work, "cg10.bin")], workdir=w)
    assert r["cgck_steps"] == 10
    d = os.path.join(w, ckpt.DIRNAME)
    assert sorted(f for f in os.listdir(d) if f.startswith("CG_")) == ["CG_P10.dat", "CG_R10.dat", "CG_V10.dat"]
    m, v, rr, p = ckpt.cg_load(d, 1000, n, np.complex128)
    assert m == 10
    m, accu = _numpy_cg(oracle, A, E0, m, v, rr, p, 1000)
    assert m == meta["cg_steps"] and accu < PREC
    ph = np.vdot(ex["cg_vec"], v)
    assert np.linalg.norm(v - ph / abs(ph) * ex["cg_vec"]) < 1e-8
    # we run 12 steps and store -> the REFERENCE resumes and finishes as in its uninterrupted run
    v = oracle.vec_randomize(n, 1); rr = np.zeros_like(v); p = np.zeros_like(v)
    m, accu = _numpy_cg(oracle, A, E0, 0, v, rr, p, 12)
    assert m == 12
    w2 = os.path.join(work, "cg_we_write")
    d2 = os.path.join(w2, ckpt.DIRNAME)
    ckpt.cg_store(d2, m, v, rr, p)
    out = os.path.join(work, "cg_final.bin")
    r2 = oracle.run_qb_ref(["file_z", path, "--cg-ckpt", repr(E0), 1000, out], workdir=w2)
    assert r2["cgck_steps"] == meta["cg_steps"] and r2["cgck_accuracy"] < PREC
    vf = np.fromfile(out, dtype=np.complex128)
    ph = np.vdot(ex["cg_vec"], vf)
    assert np.linalg.norm(vf - ph / abs(ph) * ex["cg_vec"]) < 1e-8
    # an update interrupted before its commit marker falls back to the last complete step; clean removes everything
    ckpt.cg_store(d2, 5, v, rr, p)
    with open(os.path.join(d2, "CG_updt.Qckpt1"), "wb") as f:
        f.write((6).to_bytes(8, "little"))
    with open(os.path.join(d2, "CG_V6.dat"), "wb") as f:
        f.write(b"half written")
    assert ckpt.cg_load(d2, 1000, n, np.complex128)[0] == 5 and not os.path.exists(os.path.join(d2, "CG_V6.dat"))
    ckpt.cg_clean(d2)
    assert ckpt.cg_load(d2, 1000, n, np.complex128)[0] == 0


# ------------------------------------------------------------------------------------------- the outer E0 / V0 / E1 / V1 state file
def test_e0_state_file_has_the_references_layout_and_survives_a_crash_at_every_point(tmp_path):
    """ckpt_lczsE0_init / ckpt_lczsE0_updt (src/model.cc:2519-2746): 4 bools + MKL_INT nconv + E0, E1, gap = 36 bytes; an update
    interrupted before its new content is complete leaves the OLD state, one interrupted after it is rolled FORWARD (and the
    finished stage's own Lanczos / CG checkpoints are dropped, as the reference does)."""
    import struct
    d = str(tmp_path / ckpt.DIRNAME)
    st = ckpt.e0_state_init(d, sym=1, sec=0, momentum=[3])
    f0 = os.path.join(d, "lczs_E0_sym1_sec0_K3.Qckpt")
    assert os.path.getsize(f0) == 4 * 1 + 8 + 3 * 8 == 36                     # filesize_ideal, src/model.cc:2543
    assert st == dict(E0_done=False, V0_done=False, E1_done=False, V1_done=False, nconv=0, E0=0.0, E1=0.0, gap=0.0)
    st.update(E0_done=True, E0=-7.25)
    ckpt.e0_state_update(st, d, 1, 0, [3])
    assert struct.unpack("<????qddd", open(f0, "rb").read()) == (True, False, False, False, 0, -7.25, 0.0, 0.0)
    assert ckpt.e0_state_init(d, 1, 0, [3])["E0"] == -7.25
    assert sorted(os.listdir(d)) == ["lczs_E0_sym1_sec0_K3.Qckpt"]
    # a stage's own checkpoint that must survive an update that did not commit, and go when it did
    open(os.path.join(d, "HessenbergA.dat"), "wb").write(b"x")
    new = dict(st, V0_done=True, nconv=1)
    for crash, expect_new in ((1, False), (2, True), (3, True)):
        with pytest.raises(ckpt._Interrupted):
            ckpt.e0_state_update(new, d, 1, 0, [3], _crash_after=crash)
        got = ckpt.e0_state_init(d, 1, 0, [3])
        assert got["V0_done"] == expect_new and got["E0"] == -7.25
        assert not os.path.exists(f0 + "1") and not os.path.exists(f0 + "2") and os.path.getsize(f0) == 36
        assert os.path.exists(os.path.join(d, "HessenbergA.dat")) == (not expect_new)
        if expect_new:                                                         # back to the old state for the next round
            ckpt.e0_state_update(st, d, 1, 0, [3])
            open(os.path.join(d, "HessenbergA.dat"), "wb").write(b"x")
    # the full basis carries no momentum tag (src/model.cc:2545-2552)
    ckpt.e0_state_init(d, sym=0, sec=2)
    assert os.path.exists(os.path.join(d, "lczs_E0_sym0_sec2.Qckpt"))
    # V1_done without the vectors is refused
    with pytest.raises(Exception):
        ckpt.e0_state_update(dict(st, V0_done=True, E1_done=True, V1_done=True), d, 1, 0, [3])
